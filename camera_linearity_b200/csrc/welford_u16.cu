// K3 for 16-bit cameras: Welford mean / standard-error frames of uint16 frame stacks (16-bit data, or 12-bit data
// stored in uint16), with or without an ICRF of up to 65536 rows.  Same two forms and the same semantics as the
// 8-bit kernels of welford.cu (see there and include/camera_linearity.h); the quantised mean is a uint16 frame,
// np.around(mean * MAX_DN).astype(np.uint16) with NumPy's wrapping cast.
//
//  * stack, no ICRF (welford_stack_u16_kernel): sum(d) (uint32) and sum(d^2) (uint64) are exact integers for
//    F <= 65536 frames, so the frames are streamed once (2 B/sample/frame, 16-byte loads = 8 samples) and
//    mean / SEM / uint16 mean are derived from the exact sums; the exact half-integer ties are replayed.
//  * stack with an ICRF (welford_stack_lut_u16_kernel): float64 sums of the first-frame-shifted table values, the
//    table (65536 x C float64: 512 KB per channel) gathered through L1/L2; samples inside a derived near-tie window
//    are replayed.
//  * replay (welford_replay_u16_kernel): the reference recurrence for listed samples (ties) or for the whole image
//    (ragged n or unaligned buffers).
//  * streaming update / finalize: the reference recurrence operation for operation, x = d / MAX_DN with __ddiv_rn.
#include "welford.cuh"

namespace cl {
namespace {

constexpr int kU16Threads = 256;
constexpr int kU16MaxFrames = 65536;       // tie analysis bound of the stack form, see DESIGN.md (K3)
constexpr uint32_t kU16TableRows = 65536;  // a table this long has a row for every uint16 DN

// np.around(x).astype(np.uint16) as NumPy on x86 computes it: round half to even, convert through a signed 32-bit
// integer, keep the low 16 bits; NaN, inf and |x| >= 2^31 give the "integer indefinite" 0x80000000, so 0.
__device__ __forceinline__ uint16_t wrap_u16(double x) {
    const double r = rint(x);
    if (!(r >= -2147483648.0 && r < 2147483648.0)) return 0;
    return (uint16_t)(uint32_t)__double2int_rn(r);
}

// Row of DN d in a table of `rows` rows.  A DN without a row reads the last one and raises `oob` (the caller
// reports it); FULL = 65536 rows, where every DN has its row and the test compiles away.
template <bool FULL>
__device__ __forceinline__ uint32_t table_row(uint32_t d, uint32_t rows, bool& oob) {
    if (FULL) return d;
    if (d >= rows) { oob = true; return rows - 1; }
    return d;
}

// ---- streaming form ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(kU16Threads)
welford_update_u16_kernel(const uint16_t* __restrict__ frames, int F, int64_t n, int C,
                          const double* __restrict__ lut, uint32_t rows, double max_dn,
                          double* __restrict__ mean, double* __restrict__ m2, int64_t count0) {
    const int64_t n_vec = (n + 3) / 4;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    bool oob = false;                     // (ops checks the DNs of a short table before the call)
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vec; v += stride) {
        const int64_t base = v * 4;
        const bool full = base + 4 <= n;
        WelfordState st[4];
        int cidx[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool ok = base + j < n;
            st[j].mean = ok ? mean[base + j] : 0.0;
            st[j].m2 = ok ? m2[base + j] : 0.0;
            cidx[j] = (int)((base + j) % C);
        }
        for (int f = 0; f < F; ++f) {
            const uint16_t* fr = frames + (int64_t)f * n + base;
            uint32_t d[4];
            if (full && ((reinterpret_cast<uintptr_t>(fr) & 7) == 0)) {
                const uint2 u = *reinterpret_cast<const uint2*>(fr);
                d[0] = u.x & 0xFFFFu; d[1] = u.x >> 16; d[2] = u.y & 0xFFFFu; d[3] = u.y >> 16;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) d[j] = (base + j < n) ? fr[j] : 0u;
            }
            const double nn = (double)(count0 + f + 1);
            const double rn = __drcp_rn(nn);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double x = lut ? __ldg(lut + (size_t)table_row<false>(d[j], rows, oob) * C + cidx[j])
                                     : __ddiv_rn((double)d[j], max_dn);
                welford_step(st[j], x, nn, rn);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (base + j < n) {
                mean[base + j] = st[j].mean;
                m2[base + j] = st[j].m2;
            }
    }
}

__global__ void welford_finalize_u16_kernel(const double* __restrict__ mean, const double* __restrict__ m2,
                                            double count, int64_t n, double max_dn,
                                            double* __restrict__ sem, uint16_t* __restrict__ mean_u16) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const double sq = __dsqrt_rn(count);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (sem && m2)   // np.sqrt(m2 / (n - 1)) / np.sqrt(n), video_processing.py:214
            sem[i] = __ddiv_rn(__dsqrt_rn(__ddiv_rn(m2[i], __dsub_rn(count, 1.0))), sq);
        if (mean_u16)    // np.around(mean * MAX_DN).astype(uint16): the R9 extension for 16-bit frames
            mean_u16[i] = wrap_u16(__dmul_rn(mean[i], max_dn));
    }
}

// ---- stack form, integer path ---------------------------------------------------------------------
// Thread <-> 8 consecutive samples (one uint4 of 8 DNs per frame); `slices` lanes of a warp share the same samples
// and take frames f = slice, slice + slices, ... (combined with __shfl_xor), as welford_stack_u8_kernel.  There is no
// dot-product instruction for 16-bit lanes: per sample-frame one extract (LOP3 / SHF), one IADD for sum(d) and one
// IMAD.WIDE.U32 that squares and accumulates into the 64-bit sum(d^2).  d^2 < 2^32; sum(d) < 2^32 for F <= 65537.
constexpr int kU16Unroll = 8;   // frames in flight per thread (8 x 16 B)

// q + d * d in one IMAD.WIDE.U32 (written as C, nvcc splits the 64-bit add into IMAD + IADD3 + IADD3.X)
__device__ __forceinline__ unsigned long long mad_wide(uint32_t d, unsigned long long q) {
    asm("mad.wide.u32 %0, %1, %1, %0;" : "+l"(q) : "r"(d));
    return q;
}

__device__ __forceinline__ void accumulate_u16x8(const uint4& a, uint32_t (&s)[8], unsigned long long (&q)[8]) {
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t lo = w[k] & 0xFFFFu, hi = w[k] >> 16;
        s[2 * k] += lo;
        s[2 * k + 1] += hi;
        q[2 * k] = mad_wide(lo, q[2 * k]);
        q[2 * k + 1] = mad_wide(hi, q[2 * k + 1]);
    }
}

__global__ void __launch_bounds__(kU16Threads, 3)
welford_stack_u16_kernel(const uint16_t* __restrict__ frames, int F, int64_t n, int slices,
                         double max_dn, double* __restrict__ mean, double* __restrict__ sem,
                         uint16_t* __restrict__ mean_u16, StackHeader* __restrict__ hdr,
                         uint32_t* __restrict__ ties, uint32_t tie_capacity) {
    const int64_t n_vec = n / 8;                        // n % 8 == 0 on this path
    const int vec_per_warp = 32 / slices;
    const int lane = threadIdx.x & 31;
    const int slice = lane / vec_per_warp;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t n_groups = (n_vec + vec_per_warp - 1) / vec_per_warp;
    for (int64_t g = warp_global; g < n_groups; g += n_warps) {
        const int64_t v = g * vec_per_warp + (lane % vec_per_warp);
        const bool active = v < n_vec;
        uint32_t sum[8];
        unsigned long long sq[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { sum[j] = 0; sq[j] = 0; }
        if (active) {
            const int64_t step = (int64_t)slices * n_vec;            // uint4 from one of this lane's frames to the next
            const uint4* p = reinterpret_cast<const uint4*>(frames) + v + (int64_t)slice * n_vec;
            int f = slice;
            for (; f + (kU16Unroll - 1) * slices < F; f += kU16Unroll * slices) {
                uint4 x[kU16Unroll];
#pragma unroll
                for (int u = 0; u < kU16Unroll; ++u) { x[u] = __ldg(p); p += step; }
#pragma unroll
                for (int u = 0; u < kU16Unroll; ++u) accumulate_u16x8(x[u], sum, sq);
            }
            for (; f < F; f += slices) { accumulate_u16x8(__ldg(p), sum, sq); p += step; }
        }
        for (int o = vec_per_warp; o < 32; o <<= 1) {   // combine the frame slices (exact)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                sum[j] += __shfl_xor_sync(0xffffffffu, sum[j], o);
                sq[j] += __shfl_xor_sync(0xffffffffu, sq[j], o);
            }
        }
        if (active && slice == 0) {
            // the epilogue idiom of welford_stack_u8_kernel: reciprocals of the uniform divisors once per thread,
            // the mean as the Markstein-corrected (correctly rounded) quotient, the integer quotient from the double
            // one with an exact remainder, sqrt()'s main path: its operand is 0 (selected) or within
            // [1 / (F MAX_DN^2), 2^64 / MAX_DN^2], inside that path for the 1 <= MAX_DN <= 2^32 this kernel takes
            const double fF = (double)F;
            const double denom = fF * max_dn;
            const double sqF = sqrt(fF);
            const double r_denom = __drcp_rn(denom), r_F = __drcp_rn(fF), r_sqF = __drcp_rn(sqF),
                         r_m2f1 = __dmul_rn(__drcp_rn(fF * (max_dn * max_dn)), __drcp_rn(fF - 1.0));
            uint32_t mu[4] = {0, 0, 0, 0};
            const int64_t base = v * 8;
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
                double mo[2], so[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t s32 = sum[j + h];
                    const double sd = u32_to_double(s32);
                    const double q0 = __dmul_rn(sd, r_denom);
                    mo[h] = __fma_rn(__fma_rn(-q0, denom, sd), r_denom, q0);              // == RN(s / denom)
                    // F s2 - s^2 is exact in 64 bits: both terms are at most (F 65535)^2 < 2^64 for F <= 65536;
                    // it is rounded once, to double
                    const unsigned long long num = (unsigned long long)F * sq[j + h] - (unsigned long long)s32 * s32;
                    const double t = __dmul_rn(__ull2double_rn(num), r_m2f1);
                    bool ok;
                    const double root = sqrt_main_path(t, ok);
                    so[h] = (F > 1) ? __dmul_rn(ok ? root : 0.0, r_sqF)
                                    : __longlong_as_double(0x7ff8000000000000LL);                // F == 1: sqrt(0 / 0)
                    uint32_t qd = __double2uint_rz(__dmul_rn(sd, r_F));                       // floor(s / F), +-1
                    uint32_t r = s32 - qd * (uint32_t)F;
                    if ((int32_t)r < 0) { --qd; r += (uint32_t)F; }
                    else if (r >= (uint32_t)F) { ++qd; r -= (uint32_t)F; }
                    uint32_t m16 = qd;
                    if (2ull * r > (unsigned)F) m16 = qd + 1;
                    else if (2ull * r == (unsigned)F) {
                        m16 = qd + (qd & 1u);              // provisional (half-even); replayed exactly
                        const unsigned int slot = atomicAdd(&hdr->tie_count, 1u);
                        if (slot < tie_capacity) ties[slot] = (uint32_t)(base + j + h);
                    }
                    mu[(j + h) / 2] |= (m16 & 0xFFFFu) << (16 * ((j + h) % 2));
                }
                if (mean) *reinterpret_cast<double2*>(mean + base + j) = make_double2(mo[0], mo[1]);
                if (sem) *reinterpret_cast<double2*>(sem + base + j) = make_double2(so[0], so[1]);
                asm volatile("" ::: "memory");         // keep the pairs' chains apart, as welford_stack_u8_kernel
            }
            if (mean_u16) *reinterpret_cast<uint4*>(mean_u16 + base) = make_uint4(mu[0], mu[1], mu[2], mu[3]);
        }
    }
}

// ---- exact replay ---------------------------------------------------------------------------------
// One lane per sample runs the reference recurrence over all F frames: the listed samples (ties: only the uint16
// mean is written) or a contiguous range (the whole image when the stack kernels cannot run: float outputs too).
// The DNs of the next 16 frames are in flight while the lane steps through the current 16; x comes from the table
// in global memory, or d / MAX_DN with __ddiv_rn (off the dependent chain).
constexpr int kU16ReplayBatch = 16;

__global__ void __launch_bounds__(128)
welford_replay_u16_kernel(const uint16_t* __restrict__ frames, int F, int64_t n, int C,
                          const double* __restrict__ lut, uint32_t rows, double max_dn,
                          const StackHeader* __restrict__ hdr, const uint32_t* __restrict__ ties,
                          uint32_t tie_capacity, int64_t range_first, int64_t range_count, bool write_float,
                          double* __restrict__ mean, double* __restrict__ sem, uint16_t* __restrict__ mean_u16) {
    int64_t count = range_count;
    if (ties) count = min(hdr->tie_count, tie_capacity);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    bool oob = false;                     // (reported by the stack kernel, which sees every DN)
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += stride) {
        const int64_t i = ties ? (int64_t)ties[t] : range_first + t;
        const int c = (int)(i % C);
        const uint16_t* fp = frames + i;
        WelfordState st{0.0, 0.0};
        uint32_t d[kU16ReplayBatch], dn[kU16ReplayBatch];
#pragma unroll
        for (int u = 0; u < kU16ReplayBatch; ++u) d[u] = u < F ? __ldg(fp + (int64_t)u * n) : 0u;
        for (int f0 = 0; f0 < F; f0 += kU16ReplayBatch) {
#pragma unroll
            for (int u = 0; u < kU16ReplayBatch; ++u) {
                const int f = f0 + kU16ReplayBatch + u;
                dn[u] = f < F ? __ldg(fp + (int64_t)f * n) : 0u;
            }
#pragma unroll
            for (int u = 0; u < kU16ReplayBatch; ++u) {
                if (f0 + u < F) {
                    const double nn = (double)(f0 + u + 1);
                    const double x = lut ? __ldg(lut + (size_t)table_row<false>(d[u], rows, oob) * C + c)
                                         : __ddiv_rn((double)d[u], max_dn);
                    welford_step(st, x, nn, __drcp_rn(nn));
                }
            }
#pragma unroll
            for (int u = 0; u < kU16ReplayBatch; ++u) d[u] = dn[u];
        }
        if (mean_u16) mean_u16[i] = wrap_u16(__dmul_rn(st.mean, max_dn));
        if (write_float) {
            const double fF = (double)F;
            if (mean) mean[i] = st.mean;
            if (sem) sem[i] = __ddiv_rn(__dsqrt_rn(__ddiv_rn(st.m2, __dsub_rn(fF, 1.0))), __dsqrt_rn(fF));
        }
    }
}

// ---- stack form with an ICRF ----------------------------------------------------------------------
// y = x - x_first accumulated in float64 as welford_stack_lut_kernel does (well conditioned for static scenes).
// Thread <-> 4 samples (one 8-byte load of 4 DNs per frame, two batches of 4 frames in registers); the table rows
// are gathered from global memory (L1 / L2: 512 KB per channel does not fit shared memory).
//
// Near-ties.  With M = max |x| over a sample's frames, u = 2^-53, the reference's mean is within
// u M (F + 4 (1 + ln F)) of the exact mean (per step: the rounding of mean + q, and of delta and delta / n, each
// <= 2 u M / n) and this kernel's within u M (F + 2) (recursive summation of |y| <= M, the quotient and the shift);
// both products mean * MAX_DN add u M MAX_DN.  So |kernel - reference| < w = u M MAX_DN (4F + 16) in scaled units,
// and every sample whose scaled mean is within w of a half-integer is replayed.  M <= |x_first| + sqrt(sum y^2).
constexpr int kLut16Samples = 4;
constexpr int kLut16Frames = 4;

template <bool FULL>
__device__ __forceinline__ void lut16_accumulate4(uint2 q, const double* const (&tab)[4], uint32_t C,
                                                  const double (&x0)[4], double (&s1)[4], double (&s2)[4],
                                                  uint32_t rows, bool& oob) {
    const uint32_t w[2] = {q.x, q.y};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t d = (j & 1) ? (w[j >> 1] >> 16) : (w[j >> 1] & 0xFFFFu);
        const double x = __ldg(tab[j] + table_row<FULL>(d, rows, oob) * C);
        const double y = x - x0[j];
        s1[j] += y;
        s2[j] = fma(y, y, s2[j]);
    }
}

template <bool FULL>
__global__ void __launch_bounds__(kU16Threads, FULL ? 4 : 3)
welford_stack_lut_u16_kernel(const uint16_t* __restrict__ frames, int F, int64_t n, int C,
                             const double* __restrict__ lut, uint32_t rows, double max_dn,
                             double* __restrict__ mean, double* __restrict__ sem, uint16_t* __restrict__ mean_u16,
                             StackHeader* __restrict__ hdr, uint32_t* __restrict__ ties, uint32_t tie_capacity) {
    const int64_t n_vec = (n + kLut16Samples - 1) / kLut16Samples;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const bool aligned8 = ((reinterpret_cast<uintptr_t>(frames) & 7) == 0) && (n % 4 == 0);
    const double fF = (double)F;
    const double wscale = ldexp(max_dn * (4.0 * fF + 16.0), -53);
    bool oob = false;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vec; v += stride) {
        const int64_t base = v * kLut16Samples;
        const bool full = aligned8 && base + kLut16Samples <= n;
        double x0[kLut16Samples], s1[kLut16Samples], s2[kLut16Samples];
        const double* tab[kLut16Samples];     // this sample's channel column of the table
#pragma unroll
        for (int j = 0; j < kLut16Samples; ++j) {
            s1[j] = s2[j] = x0[j] = 0.0;
            tab[j] = lut + (base + j) % C;
            if (base + j < n) x0[j] = __ldg(tab[j] + table_row<FULL>(frames[base + j], rows, oob) * (uint32_t)C);
        }
        if (full) {
            const uint2* fp = reinterpret_cast<const uint2*>(frames + base);
            const int64_t n4 = n >> 2;
            int f0 = 0;
            uint2 q[kLut16Frames];
            if (kLut16Frames <= F) {
#pragma unroll
                for (int u = 0; u < kLut16Frames; ++u) q[u] = __ldcs(fp + u * n4);
                fp += kLut16Frames * n4;
            }
            for (; f0 + 2 * kLut16Frames <= F; f0 += kLut16Frames) {
                uint2 nq[kLut16Frames];
#pragma unroll
                for (int u = 0; u < kLut16Frames; ++u) nq[u] = __ldcs(fp + u * n4);
                fp += kLut16Frames * n4;
#pragma unroll
                for (int u = 0; u < kLut16Frames; ++u) lut16_accumulate4<FULL>(q[u], tab, C, x0, s1, s2, rows, oob);
#pragma unroll
                for (int u = 0; u < kLut16Frames; ++u) q[u] = nq[u];
            }
            if (f0 + kLut16Frames <= F) {
#pragma unroll
                for (int u = 0; u < kLut16Frames; ++u) lut16_accumulate4<FULL>(q[u], tab, C, x0, s1, s2, rows, oob);
                f0 += kLut16Frames;
            }
            for (; f0 < F; ++f0) {
                const uint2 q1 = __ldcs(fp);
                fp += n4;
                lut16_accumulate4<FULL>(q1, tab, C, x0, s1, s2, rows, oob);
            }
        } else {
            for (int f = 0; f < F; ++f) {
                const uint16_t* fr = frames + (int64_t)f * n + base;
                uint32_t w[2] = {0u, 0u};
                for (int j = 0; j < 4; ++j)
                    if (base + j < n) w[j >> 1] |= (uint32_t)fr[j] << (16 * (j & 1));
                lut16_accumulate4<FULL>(make_uint2(w[0], w[1]), tab, C, x0, s1, s2, rows, oob);
            }
        }
#pragma unroll
        for (int j = 0; j < kLut16Samples; ++j) {
            if (base + j >= n) continue;
            const double my_ = s1[j] / fF;
            const double mu = x0[j] + my_;
            double m2 = s2[j] - s1[j] * my_;
            if (m2 < 0.0) m2 = 0.0;
            if (mean) mean[base + j] = mu;
            if (sem) sem[base + j] = sqrt(m2 / (fF - 1.0)) / sqrt(fF);
            const double scaled = mu * max_dn;
            const double fr = scaled - floor(scaled);
            const double w = (fabs(x0[j]) + sqrt(s2[j])) * wscale;       // the near-tie window, see above
            if (fabs(fr - 0.5) <= w) {
                const unsigned int slot = atomicAdd(&hdr->tie_count, 1u);
                if (slot < tie_capacity) ties[slot] = (uint32_t)(base + j);
            }
            if (mean_u16) mean_u16[base + j] = wrap_u16(scaled);
        }
    }
    if (!FULL && oob) atomicOr(&hdr->dn_out_of_range, 1u);
}

bool table_ok(const double* lut, int lut_rows) { return !lut || (lut_rows >= 1 && lut_rows <= (int)kU16TableRows); }

}  // namespace
}  // namespace cl

extern "C" {

int cl_welford_update_u16(const uint16_t* frames, int n_frames, int64_t n_samples, int channels,
                          const double* lut, int lut_rows, double max_dn, double* mean, double* m2,
                          int64_t count0, void* stream) {
    using namespace cl;
    CL_REQUIRE(n_frames >= 0 && n_samples >= 0 && channels >= 1 && channels <= CL_MAX_CHANNELS);
    CL_REQUIRE(count0 >= 0 && max_dn > 0.0 && table_ok(lut, lut_rows));
    if (n_frames == 0 || n_samples == 0) return CL_OK;
    CL_REQUIRE(frames && mean && m2);
    CL_REQUIRE(n_samples % channels == 0);
    if (!aligned(frames, 2) || !aligned(mean, 8) || !aligned(m2, 8) || !aligned(lut, 8)) return CL_ERR_ALIGNMENT;
    welford_update_u16_kernel<<<grid_for((n_samples + 3) / 4, kU16Threads, 8), kU16Threads, 0,
                                (cudaStream_t)stream>>>(frames, n_frames, n_samples, channels, lut,
                                                        (uint32_t)lut_rows, max_dn, mean, m2, count0);
    return launched();
}

int cl_welford_finalize_u16(const double* mean, const double* m2, int64_t count, int64_t n_samples,
                            double max_dn, double* sem, uint16_t* mean_u16, void* stream) {
    using namespace cl;
    CL_REQUIRE(n_samples >= 0 && count >= 0);
    if (n_samples == 0) return CL_OK;
    CL_REQUIRE(mean != nullptr);
    if (!aligned(mean, 8) || !aligned(m2, 8) || !aligned(sem, 8) || !aligned(mean_u16, 2)) return CL_ERR_ALIGNMENT;
    welford_finalize_u16_kernel<<<grid_for(n_samples, kU16Threads, 8), kU16Threads, 0, (cudaStream_t)stream>>>(
        mean, m2, (double)count, n_samples, max_dn, sem, mean_u16);
    return launched();
}

int cl_welford_stack_u16(const uint16_t* frames, int n_frames, int64_t n_samples, int channels,
                         const double* lut, int lut_rows, double max_dn, double* mean, double* sem,
                         uint16_t* mean_u16, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace cl;
    CL_REQUIRE(n_frames >= 1 && n_samples >= 0 && channels >= 1 && channels <= CL_MAX_CHANNELS);
    CL_REQUIRE(max_dn > 0.0 && table_ok(lut, lut_rows));
    if (n_samples == 0) return CL_OK;
    CL_REQUIRE(frames != nullptr);
    CL_REQUIRE(n_samples % channels == 0);
    if (n_frames > kU16MaxFrames || n_samples > 0xFFFFFFFFll) return CL_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < cl_welford_stack_workspace_bytes(n_frames, n_samples))
        return CL_ERR_WORKSPACE;
    if (!aligned(workspace, 16) || !aligned(frames, 2) || !aligned(lut, 8) || !aligned(mean, 8) ||
        !aligned(sem, 8) || !aligned(mean_u16, 2))
        return CL_ERR_ALIGNMENT;
    cudaStream_t s = (cudaStream_t)stream;
    StackHeader* hdr = reinterpret_cast<StackHeader*>(workspace);
    uint32_t* ties = reinterpret_cast<uint32_t*>(hdr + 1);
    const uint32_t cap = (uint32_t)n_samples;
    const uint32_t rows = lut ? (uint32_t)lut_rows : 0u;
    cudaError_t e = cudaMemsetAsync(hdr, 0, sizeof(StackHeader), s);
    if (e != cudaSuccess) return cuda_status(e);
    int st;
    if (lut) {
        const int64_t vecs = (n_samples + kLut16Samples - 1) / kLut16Samples;
        if (rows == kU16TableRows)
            welford_stack_lut_u16_kernel<true><<<grid_for(vecs, kU16Threads, 4), kU16Threads, 0, s>>>(
                frames, n_frames, n_samples, channels, lut, rows, max_dn, mean, sem, mean_u16, hdr, ties, cap);
        else
            welford_stack_lut_u16_kernel<false><<<grid_for(vecs, kU16Threads, 3), kU16Threads, 0, s>>>(
                frames, n_frames, n_samples, channels, lut, rows, max_dn, mean, sem, mean_u16, hdr, ties, cap);
        st = launched();
        if (st != CL_OK) return st;
    } else {
        const bool vec_ok = aligned(frames, 16) && (n_samples % 8 == 0) && aligned(mean, 16) && aligned(sem, 16) &&
                            aligned(mean_u16, 16) && max_dn >= 1.0 && max_dn <= 4294967296.0;
        if (!vec_ok) {
            // ragged / unaligned input (or a MAX_DN outside the epilogue's range): exact replay of every sample
            welford_replay_u16_kernel<<<grid_for(n_samples, 128, 16), 128, 0, s>>>(
                frames, n_frames, n_samples, channels, nullptr, 0u, max_dn, hdr, nullptr, 0, 0, n_samples, true,
                mean, sem, mean_u16);
            return launched();
        }
        const int64_t n_vec = n_samples / 8;
        int slices = 1;                        // frame slices: enough threads to fill the machine when the image is small
        const int64_t want = (int64_t)sm_count() * 1024;
        while (slices < 32 && n_vec * slices < want && slices * 2 <= n_frames) slices *= 2;
        const int64_t threads = ((n_vec * slices + 31) / 32) * 32;
        welford_stack_u16_kernel<<<grid_for(threads, kU16Threads, 3), kU16Threads, 0, s>>>(
            frames, n_frames, n_samples, slices, max_dn, mean, sem, mean_u16, hdr, ties, cap);
        st = launched();
        if (st != CL_OK) return st;
    }
    if (mean_u16) {   // exact replay of the (near-)tie samples decides their uint16 mean
        welford_replay_u16_kernel<<<sm_count() * 8, 128, 0, s>>>(
            frames, n_frames, n_samples, channels, lut, rows, max_dn, hdr, ties, cap, 0, 0, false, nullptr, nullptr,
            mean_u16);
        st = launched();
        if (st != CL_OK) return st;
    }
    return CL_OK;
}

}  // extern "C"
