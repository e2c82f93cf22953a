// K3: Welford mean / standard-error frames over a video (video_processing.py:161-219).
//
// Two forms (see include/camera_linearity.h):
//  * streaming update/finalize: the reference's sequential float64 recurrence, operation for
//    operation (round-to-nearest intrinsics, no FMA contraction), so mean/M2 are bit-identical
//    to NumPy.  delta/n uses a Markstein-corrected reciprocal multiply, which is the correctly
//    rounded quotient for integer n (checked against exact rationals in tests/).
//  * stack: all F frames resident.  For 8-bit frames without an ICRF, sum(d) and sum(d^2) are
//    exact integers, so the kernel streams the frames once with integer dot-product
//    accumulation (1 B/sample/frame of HBM traffic, the roofline), optional frame-sliced lanes
//    combined with warp shuffles, and derives mean/SEM from the exact sums.  uint8 mean =
//    rint(mean*255) is decided in integers; only samples whose exact mean*255 is a half-integer
//    (a rounding tie, where NumPy's answer depends on its rounding noise) are replayed with the
//    exact sequential recurrence by a second small kernel.
#include "welford.cuh"

namespace cl {
namespace {

constexpr int kThreads = 256;

// x = frame / MAX_DN (video_processing.py:203) or ICRF[frame, c] (:201)
__global__ void __launch_bounds__(kThreads)
welford_update_kernel(const uint8_t* __restrict__ frames, int F, int64_t n, int C,
                      const double* __restrict__ lut, double max_dn, double* __restrict__ mean,
                      double* __restrict__ m2, int64_t count0) {
    extern __shared__ double xt[];   // [256] or [256][C]
    const int rows = lut ? 256 * C : 256;
    for (int i = threadIdx.x; i < rows; i += blockDim.x)
        xt[i] = lut ? lut[i] : __ddiv_rn((double)i, max_dn);
    __syncthreads();
    const int64_t n_vec = (n + 3) / 4;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
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
            const uint8_t* fr = frames + (int64_t)f * n + base;
            uint32_t d[4];
            if (full && ((reinterpret_cast<uintptr_t>(fr) & 3) == 0)) {
                const uint32_t u = *reinterpret_cast<const uint32_t*>(fr);
                d[0] = u & 0xFF; d[1] = (u >> 8) & 0xFF; d[2] = (u >> 16) & 0xFF; d[3] = u >> 24;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) d[j] = (base + j < n) ? fr[j] : 0u;
            }
            const double nn = (double)(count0 + f + 1);
            const double rn = __drcp_rn(nn);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double x = lut ? xt[d[j] * C + cidx[j]] : xt[d[j]];
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

__global__ void welford_finalize_kernel(const double* __restrict__ mean, const double* __restrict__ m2,
                                        double count, int64_t n, double max_dn,
                                        double* __restrict__ sem, uint8_t* __restrict__ mean_u8) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const double sq = __dsqrt_rn(count);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (sem && m2)   // np.sqrt(m2 / (n - 1)) / np.sqrt(n), video_processing.py:214
            sem[i] = __ddiv_rn(__dsqrt_rn(__ddiv_rn(m2[i], __dsub_rn(count, 1.0))), sq);
        if (mean_u8)     // np.around(mean * MAX_DN).astype(uint8), :210-211
            mean_u8[i] = (uint8_t)wrap_bin(__dmul_rn(mean[i], max_dn), 0xFFu);
    }
}

// ---- stack form, integer path ---------------------------------------------------------------------
// Thread <-> 16 consecutive samples (one uint4 per frame).  `slices` lanes of a warp share the same
// samples and take frames f = slice, slice + slices, ...; lanes with equal slice read consecutive
// 16-byte vectors (coalesced).  Partial integer sums are combined with __shfl_xor.
__device__ __forceinline__ void accumulate_word(uint32_t x, uint32_t* s, uint32_t* q) {
    s[0] = __dp4a(x, 0x00000001u, s[0]);
    s[1] = __dp4a(x, 0x00000100u, s[1]);
    s[2] = __dp4a(x, 0x00010000u, s[2]);
    s[3] = __dp4a(x, 0x01000000u, s[3]);
    q[0] = __dp4a(x & 0x000000FFu, x, q[0]);
    q[1] = __dp4a(x & 0x0000FF00u, x, q[1]);
    q[2] = __dp4a(x & 0x00FF0000u, x, q[2]);
    q[3] = __dp4a(x & 0xFF000000u, x, q[3]);
}

constexpr int kFrameBlock = 16384;   // sum(d^2) over a block fits uint32
constexpr int kUnroll = 8;           // frames in flight per thread (8 x 16 B)

__device__ __forceinline__ void accumulate_vec(const uint4& a, uint32_t* s, uint32_t* q) {
    accumulate_word(a.x, s + 0, q + 0);
    accumulate_word(a.y, s + 4, q + 4);
    accumulate_word(a.z, s + 8, q + 8);
    accumulate_word(a.w, s + 12, q + 12);
}

// BIG = more than kFrameBlock frames: sum(d^2) needs 64-bit totals (32 more registers).
template <bool BIG>
__global__ void __launch_bounds__(kThreads, BIG ? 2 : 3)
welford_stack_u8_kernel(const uint8_t* __restrict__ frames, int F, int64_t n, int slices,
                        double max_dn, double* __restrict__ mean, double* __restrict__ sem,
                        uint8_t* __restrict__ mean_u8, StackHeader* __restrict__ hdr,
                        uint32_t* __restrict__ ties, uint32_t tie_capacity) {
    const int64_t n_vec = n / 16;                       // full vectors; the ragged tail is separate
    const int vec_per_warp = 32 / slices;
    const int lane = threadIdx.x & 31;
    const int slice = lane / vec_per_warp;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t n_groups = (n_vec + vec_per_warp - 1) / vec_per_warp;
    for (int64_t g = warp_global; g < n_groups; g += n_warps) {
        const int64_t v = g * vec_per_warp + (lane % vec_per_warp);
        const bool active = v < n_vec;
        uint32_t sum[16], q[16];
        unsigned long long sq[BIG ? 16 : 1];
#pragma unroll
        for (int j = 0; j < 16; ++j) { sum[j] = 0; q[j] = 0; }
        if (BIG) {
#pragma unroll
            for (int j = 0; j < 16; ++j) sq[BIG ? j : 0] = 0;
        }
        if (active) {
            const uint4* src = reinterpret_cast<const uint4*>(frames) + v;
            const int64_t fstride = n / 16;             // uint4 per frame (n % 16 == 0 on this path)
            for (int f0 = 0; f0 < F; f0 += kFrameBlock) {
                const int f1 = min(F, f0 + kFrameBlock);
                int f = f0 + slice;
                // (keeping two batches in registers, as the ICRF kernel does, is slower here: same-box 0.723 ms as is,
                // 0.74 / 0.745 / 0.82 ms with two batches of 4 / 3 / 6 frames -- the 16 sums + 16 squares leave no room)
                for (; f + (kUnroll - 1) * slices < f1; f += kUnroll * slices) {
                    uint4 x[kUnroll];
#pragma unroll
                    for (int u = 0; u < kUnroll; ++u) x[u] = __ldg(src + (int64_t)(f + u * slices) * fstride);
#pragma unroll
                    for (int u = 0; u < kUnroll; ++u) accumulate_vec(x[u], sum, q);
                }
                for (; f < f1; f += slices) accumulate_vec(__ldg(src + (int64_t)f * fstride), sum, q);
                if (BIG) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) { sq[BIG ? j : 0] += q[j]; q[j] = 0; }
                }
            }
        }
        // combine the frame slices (exact: integer addition is associative)
        for (int o = vec_per_warp; o < 32; o <<= 1) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                sum[j] += __shfl_xor_sync(0xffffffffu, sum[j], o);
                if (BIG) sq[BIG ? j : 0] += __shfl_xor_sync(0xffffffffu, sq[BIG ? j : 0], o);
                else q[j] += __shfl_xor_sync(0xffffffffu, q[j], o);
            }
        }
        if (active && slice == 0) {
            const double fF = (double)F;
            const double denom = fF * max_dn;
            const double sqF = sqrt(fF);
            // Every divisor of the epilogue is the same for all samples.  The library's divisions, its square root and
            // the 64-bit integer s / F, s % F cost ~250 instructions per sample (an eighth of the kernel) and fence the
            // schedule; here (F <= kFrameBlock): reciprocals once per thread, the mean as the Markstein-corrected
            // quotient (correctly rounded, like the division it replaces), the integer quotient from the double one
            // with an exact remainder, sqrt()'s main path (its operand is 0 -- selected -- or >= 1 / (F 255^2)).
            const double r_denom = __drcp_rn(denom), r_F = __drcp_rn(fF), r_sqF = __drcp_rn(sqF),
                         r_m2f1 = __dmul_rn(__drcp_rn(fF * (max_dn * max_dn)), __drcp_rn(fF - 1.0));
            uint32_t mu[4] = {0, 0, 0, 0};
            const int64_t base = v * 16;
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
                double mo[2], so[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    uint32_t qd, r;
                    if (!BIG) {
                        const uint32_t s32 = sum[j + h];
                        const double sd = u32_to_double(s32);
                        const double q0 = __dmul_rn(sd, r_denom);
                        mo[h] = __fma_rn(__fma_rn(-q0, denom, sd), r_denom, q0);             // == RN(s / denom)
                        const unsigned long long num = (unsigned long long)F * q[j + h] - (unsigned long long)s32 * s32;   // exact, >= 0, < 2^53
                        const double numd = __fma_rn(u32_to_double((uint32_t)(num >> 32)), 4294967296.0,
                                                     u32_to_double((uint32_t)num));            // exact
                        const double t = __dmul_rn(numd, r_m2f1);
                        bool ok;
                        const double root = sqrt_main_path(t, ok);
                        so[h] = (F > 1) ? __dmul_rn(ok ? root : 0.0, r_sqF)
                                        : __longlong_as_double(0x7ff8000000000000LL);               // F == 1: sqrt(0 / 0)
                        qd = __double2uint_rz(__dmul_rn(sd, r_F));                           // floor(s / F), off by one at most
                        r = s32 - qd * (uint32_t)F;
                        if ((int32_t)r < 0) { --qd; r += (uint32_t)F; }
                        else if (r >= (uint32_t)F) { ++qd; r -= (uint32_t)F; }
                    } else {
                        const unsigned long long s = sum[j + h];
                        const unsigned long long s2 = sq[BIG ? j + h : 0];
                        mo[h] = (double)s / denom;
                        const unsigned long long num = (unsigned long long)F * s2 - s * s;   // exact, >= 0
                        const double m2 = (double)num / (fF * (max_dn * max_dn));
                        so[h] = sqrt(m2 / (fF - 1.0)) / sqF;
                        qd = (uint32_t)(s / (unsigned)F);
                        r = (uint32_t)(s % (unsigned)F);
                    }
                    uint32_t m8 = qd;
                    if (2ull * r > (unsigned)F) m8 = qd + 1;
                    else if (2ull * r == (unsigned)F) {
                        m8 = qd + (qd & 1u);               // provisional (half-even); replayed exactly
                        const unsigned int slot = atomicAdd(&hdr->tie_count, 1u);
                        if (slot < tie_capacity) ties[slot] = (uint32_t)(base + j + h);
                    }
                    mu[(j + h) / 4] |= (m8 & 0xFFu) << (8 * ((j + h) % 4));
                }
                if (mean) *reinterpret_cast<double2*>(mean + base + j) = make_double2(mo[0], mo[1]);
                if (sem) *reinterpret_cast<double2*>(sem + base + j) = make_double2(so[0], so[1]);
                asm volatile("" ::: "memory");         // keep the pairs' chains apart: interleaved they spill at 80 registers
            }
            if (mean_u8) *reinterpret_cast<uint4*>(mean_u8 + base) = make_uint4(mu[0], mu[1], mu[2], mu[3]);
        }
    }
}

// Exact replay of the rounding-tie samples.  The recurrence is a chain of 5 dependent FP64 operations per frame,
// so a tie costs F x ~50 cycles whoever runs it; what the kernel chooses is how many chains run side by side.
//  * FEW ties (< kLaneModeTies), or an ICRF table with more than 4 channels: one WARP per tie -- the 32 lanes fetch the sample's byte of
//    256 frames at once (scattered 1-byte loads, all in flight together) and do the per-frame work that is off
//    the chain (x = d / MAX_DN or the LUT value, RN(1/n)), lane 0 then runs the recurrence from shared memory:
//    latency per tie = one DRAM round trip per window + F dependent steps.
//  * MANY ties (short or low-noise videos with an even frame count: up to every sample): one LANE per tie, 32
//    chains per warp in lockstep.  x comes from a shared-memory table of the 256 DN values, RN(1/n) from a shared
//    window computed once per CTA, and each lane keeps the bytes of the next 16 frames in flight while it steps
//    through the current 16, so the loads hide behind the chain.  (cfg4's synthetic video has ~15 ties in 6.2 M
//    samples -- the sum of 600 noise terms of sigma 3 rarely reaches +-300 -- and takes the first form.)
constexpr int kReplayWindow = 256;
constexpr int kReplayWarps = 4;
constexpr int kReplayBatch = 16;
constexpr uint32_t kLaneModeTies = 256;      // below this the warp-per-tie form has nothing to lose

__global__ void __launch_bounds__(kReplayWarps * 32)
welford_tie_replay_kernel(const uint8_t* __restrict__ frames, int F, int64_t n, int C,
                          const double* __restrict__ lut, double max_dn, const StackHeader* __restrict__ hdr,
                          const uint32_t* __restrict__ ties, uint32_t tie_capacity,
                          uint8_t* __restrict__ mean_u8) {
    __shared__ double xs[kReplayWarps][kReplayWindow];
    __shared__ double rs[kReplayWarps][kReplayWindow];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t count = min(hdr->tie_count, tie_capacity);
    if (count >= kLaneModeTies && (!lut || C <= kReplayWarps)) {      // (the table must fit xs: 256 * C <= 1024)
        // ---- one lane per tie ----
        double* xt = &xs[0][0];                       // [256][C] LUT values, or [256] d / MAX_DN
        double* rw = &rs[0][0];                       // RN(1 / n) of the current window of frames
        const int rows = lut ? 256 * C : 256;
        for (int i = threadIdx.x; i < rows; i += blockDim.x) xt[i] = lut ? lut[i] : __ddiv_rn((double)i, max_dn);
        for (uint32_t t0 = blockIdx.x * blockDim.x; t0 < count; t0 += gridDim.x * blockDim.x) {   // (uniform per CTA)
            const uint32_t t = t0 + threadIdx.x;
            const bool live = t < count;
            const int64_t i = live ? (int64_t)ties[t] : 0;
            const uint32_t xoff = lut ? (uint32_t)(i % C) : 0u, xmul = lut ? (uint32_t)C : 1u;
            const uint8_t* fp = frames + i;
            double mean = 0.0;
            uint32_t d[kReplayBatch], dn[kReplayBatch];
#pragma unroll
            for (int u = 0; u < kReplayBatch; ++u) d[u] = (live && u < F) ? __ldg(fp + (int64_t)u * n) : 0u;
            for (int f0 = 0; f0 < F; f0 += kReplayWindow) {
                const int len = min(kReplayWindow, F - f0);
                __syncthreads();
                for (int f = threadIdx.x; f < len; f += blockDim.x) rw[f] = __drcp_rn((double)(f0 + f + 1));
                __syncthreads();
                for (int g = 0; g < len; g += kReplayBatch) {
                    const int fnext = f0 + g + kReplayBatch;                 // first frame of the next batch
#pragma unroll
                    for (int u = 0; u < kReplayBatch; ++u)
                        dn[u] = (live && fnext + u < F) ? __ldg(fp + (int64_t)(fnext + u) * n) : 0u;
#pragma unroll
                    for (int u = 0; u < kReplayBatch; ++u)
                        if (g + u < len)
                            welford_mean_step(mean, xt[d[u] * xmul + xoff], (double)(f0 + g + u + 1), rw[g + u]);
#pragma unroll
                    for (int u = 0; u < kReplayBatch; ++u) d[u] = dn[u];
                }
            }
            if (live) mean_u8[i] = (uint8_t)wrap_bin(__dmul_rn(mean, max_dn), 0xFFu);
        }
        return;
    }
    // ---- one warp per tie ----
    for (uint32_t t = blockIdx.x * kReplayWarps + warp; t < count; t += gridDim.x * kReplayWarps) {
        const int64_t i = (int64_t)ties[t];
        const int c = (int)(i % C);
        WelfordState st{0.0, 0.0};
        for (int f0 = 0; f0 < F; f0 += kReplayWindow) {
            const int len = min(kReplayWindow, F - f0);
            __syncwarp();
#pragma unroll
            for (int u = 0; u < kReplayWindow / 32; ++u) {
                const int f = lane + 32 * u;
                if (f < len) {
                    const uint32_t d = __ldg(frames + (int64_t)(f0 + f) * n + i);
                    xs[warp][f] = lut ? lut[d * C + c] : __ddiv_rn((double)d, max_dn);
                    rs[warp][f] = __drcp_rn((double)(f0 + f + 1));
                }
            }
            __syncwarp();
            if (lane == 0) {
#pragma unroll 4
                for (int f = 0; f < len; ++f) welford_step(st, xs[warp][f], (double)(f0 + f + 1), rs[warp][f]);
            }
        }
        if (lane == 0) mean_u8[i] = (uint8_t)wrap_bin(__dmul_rn(st.mean, max_dn), 0xFFu);
    }
}

// Exact replay for listed samples (ties) or for a contiguous tail range: one lane per sample runs
// the reference recurrence over all F frames and overwrites mean_u8 (and optionally mean / sem so
// the ragged tail is complete).
__global__ void __launch_bounds__(128)
welford_replay_kernel(const uint8_t* __restrict__ frames, int F, int64_t n, int C,
                      const double* __restrict__ lut, double max_dn, const StackHeader* __restrict__ hdr,
                      const uint32_t* __restrict__ ties, uint32_t tie_capacity, int64_t range_first,
                      int64_t range_count, bool write_float, double* __restrict__ mean,
                      double* __restrict__ sem, uint8_t* __restrict__ mean_u8) {
    int64_t count = range_count;
    if (ties) {
        const unsigned int c = hdr->tie_count;
        count = c < tie_capacity ? c : tie_capacity;
    }
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < count; t += stride) {
        const int64_t i = ties ? (int64_t)ties[t] : range_first + t;
        const int c = (int)(i % C);
        WelfordState st{0.0, 0.0};
        int f = 0;
        // 32 independent byte loads in flight per lane, then 32 sequential recurrence steps
        for (; f + 32 <= F; f += 32) {
            uint32_t d[32];
#pragma unroll
            for (int u = 0; u < 32; ++u) d[u] = __ldg(frames + (int64_t)(f + u) * n + i);
#pragma unroll
            for (int u = 0; u < 32; ++u) {
                const double nn = (double)(f + u + 1);
                const double x = lut ? lut[d[u] * C + c] : __ddiv_rn((double)d[u], max_dn);
                welford_step(st, x, nn, __drcp_rn(nn));
            }
        }
        for (; f < F; ++f) {
            const uint32_t d = frames[(int64_t)f * n + i];
            const double nn = (double)(f + 1);
            const double x = lut ? lut[d * C + c] : __ddiv_rn((double)d, max_dn);
            welford_step(st, x, nn, __drcp_rn(nn));
        }
        if (mean_u8) mean_u8[i] = (uint8_t)wrap_bin(__dmul_rn(st.mean, max_dn), 0xFFu);
        if (write_float) {
            const double fF = (double)F;
            if (mean) mean[i] = st.mean;
            if (sem) sem[i] = __ddiv_rn(__dsqrt_rn(__ddiv_rn(st.m2, __dsub_rn(fF, 1.0))), __dsqrt_rn(fF));
        }
    }
}

// ---- stack form with an ICRF: float64 accumulation of the (shifted) LUT values ------------------
// y = x - x_first: sum(y), sum(y^2) stay well conditioned when the video is nearly static.
// Thread <-> 8 consecutive samples (one 8-byte load per frame), 8 frames of loads in flight, and the
// ICRF table replicated per lane in shared memory ([c][dn][copy], copy = lane % copies) so that the
// random 8-bit gathers are bank-conflict free -- the first version (4 samples, one 4-byte load in
// flight, plain table) ran at 0.96 TB/s.
// Round 2: 4 samples per thread (one 4-byte load per frame) and 512 threads per CTA, two CTAs per SM: the
// accumulators of 8 samples cost 120 registers and left 16 warps per SM, which could not hide the
// LDS -> DADD -> DADD / DFMA chain (1.77 ms for cfg4); with 64 registers 32 warps are resident (1.35 ms).
// The loop then stalled on the first use of a loaded frame word (ncu: long scoreboard 6.7 per issue, no pipe above
// 64 %): two batches of 4 frames are kept in registers, batch b+1 in flight while batch b is accumulated -> 1.225 ms.
// Same-box sweep of that batch size, ms: 2: 1.83, 3: 1.38, 4: 1.225, 5: 1.26, 6: 1.27, 8: 1.25; three batches of 4: 1.25
// -- beyond this the kernel is on its pipes (LDS.64 = 2 wavefronts per 32 sample-frames: 0.83 ms; FP64: 0.62 ms).
constexpr int kLutSamples = 4;
constexpr int kLutFrames = 4;
constexpr int kLutThreads = 512;

__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

// one frame's 4 packed DNs of this thread's samples: gather, shift, accumulate.  Per sample-frame: PRMT (byte
// extract), LEA (32-bit shared address), LDS.64, DADD, DADD, DFMA -- the first version spent 12.5 instructions
// per sample-frame (64-bit generic-pointer arithmetic, per-frame bounds checks) and was issue bound at 1.9 ms.
template <int COPIES>
__device__ __forceinline__ void lut_accumulate4(uint32_t q, const uint32_t (&toff)[4], const double (&x0)[4],
                                                double (&s1)[4], double (&s2)[4]) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t d = __byte_perm(q, 0u, 0x4440u + j);          // byte j, zero extended
        const double x = lds_f64(d * (COPIES * 8u) + toff[j]);       // one IMAD: the stride is an immediate
        const double y = x - x0[j];
        s1[j] += y;
        s2[j] = fma(y, y, s2[j]);
    }
}

template <int COPIES>
__global__ void __launch_bounds__(kLutThreads, 2)
welford_stack_lut_kernel(const uint8_t* __restrict__ frames, int F, int64_t n, int C,
                         const double* __restrict__ lut, double max_dn, double* __restrict__ mean,
                         double* __restrict__ sem, uint8_t* __restrict__ mean_u8,
                         StackHeader* __restrict__ hdr, uint32_t* __restrict__ ties,
                         uint32_t tie_capacity) {
    extern __shared__ double xt[];   // [C][256][copies]
    for (int i = threadIdx.x; i < 256 * C; i += blockDim.x) {
        const int d = i / C, c = i - d * C;
        const double x = lut[i];
        for (int r = 0; r < COPIES; ++r) xt[(c * 256 + d) * COPIES + r] = x;
    }
    __syncthreads();
    const uint32_t xt_s = (uint32_t)__cvta_generic_to_shared(xt) + (threadIdx.x & (COPIES - 1)) * 8u;
    const int64_t n_vec = (n + kLutSamples - 1) / kLutSamples;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const bool aligned4 = ((reinterpret_cast<uintptr_t>(frames) & 3) == 0) && (n % 4 == 0);
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vec; v += stride) {
        const int64_t base = v * kLutSamples;
        const bool full = aligned4 && base + kLutSamples <= n;
        double x0[kLutSamples], s1[kLutSamples], s2[kLutSamples];
        uint32_t toff[kLutSamples];           // shared-memory byte address of this sample's channel table, this lane's copy
#pragma unroll
        for (int j = 0; j < kLutSamples; ++j) {
            s1[j] = s2[j] = x0[j] = 0.0;
            toff[j] = xt_s + (uint32_t)((base + j) % C) * (256u * COPIES * 8u);
        }
        {   // x_first: the shift (frame 0 is accumulated again below, contributing y = 0 exactly)
            const uint8_t* fr = frames + base;
            for (int j = 0; j < kLutSamples; ++j)
                if (base + j < n) x0[j] = lds_f64(toff[j] + (uint32_t)fr[j] * (COPIES * 8u));
        }
        if (full) {
            const uint32_t* fp = reinterpret_cast<const uint32_t*>(frames + base);
            const int64_t n4 = n >> 2;
            int f0 = 0;
            // two batches of frames in registers: the loads of batch b+1 are in flight while batch b is accumulated
            // (the kernel was stalled on the first use of a loaded word, not on any pipe)
            uint32_t q[kLutFrames];
            if (kLutFrames <= F) {
#pragma unroll
                for (int u = 0; u < kLutFrames; ++u) q[u] = __ldcs(fp + u * n4);
                fp += kLutFrames * n4;
            }
            for (; f0 + 2 * kLutFrames <= F; f0 += kLutFrames) {
                uint32_t nq[kLutFrames];
#pragma unroll
                for (int u = 0; u < kLutFrames; ++u) nq[u] = __ldcs(fp + u * n4);
                fp += kLutFrames * n4;
#pragma unroll
                for (int u = 0; u < kLutFrames; ++u) lut_accumulate4<COPIES>(q[u], toff, x0, s1, s2);
#pragma unroll
                for (int u = 0; u < kLutFrames; ++u) q[u] = nq[u];
            }
            if (f0 + kLutFrames <= F) {
#pragma unroll
                for (int u = 0; u < kLutFrames; ++u) lut_accumulate4<COPIES>(q[u], toff, x0, s1, s2);
                f0 += kLutFrames;
            }
            for (; f0 < F; ++f0) {
                const uint32_t q = __ldcs(fp);
                fp += n4;
                lut_accumulate4<COPIES>(q, toff, x0, s1, s2);
            }
        } else {
            for (int f = 0; f < F; ++f) {
                const uint8_t* fr = frames + (int64_t)f * n + base;
                uint32_t q = 0u;
                for (int j = 0; j < 4; ++j)
                    if (base + j < n) q |= (uint32_t)fr[j] << (8 * j);
                lut_accumulate4<COPIES>(q, toff, x0, s1, s2);
            }
        }
        const double fF = (double)F;
#pragma unroll
        for (int j = 0; j < kLutSamples; ++j) {
            if (base + j >= n) continue;
            const double my_ = s1[j] / fF;
            const double mu = x0[j] + my_;
            double m2 = s2[j] - s1[j] * my_;
            if (m2 < 0.0) m2 = 0.0;
            if (mean) mean[base + j] = mu;
            if (sem) sem[base + j] = sqrt(m2 / (fF - 1.0)) / sqrt(fF);
            const double scaled = mu * max_dn;
            const double fr = scaled - floor(scaled);
            // near a rounding tie the uint8 mean depends on the reference's rounding noise
            if (fabs(fr - 0.5) < 1e-9) {
                const unsigned int slot = atomicAdd(&hdr->tie_count, 1u);
                if (slot < tie_capacity) ties[slot] = (uint32_t)(base + j);
            }
            if (mean_u8) mean_u8[base + j] = (uint8_t)wrap_bin(scaled, 0xFFu);
        }
    }
}

constexpr uint32_t kMaxFramesStack = 1000000;   // tie analysis bound, see DESIGN.md

}  // namespace
}  // namespace cl

extern "C" {

int cl_welford_update(const uint8_t* frames, int n_frames, int64_t n_samples, int channels,
                      const double* lut, double max_dn, double* mean, double* m2, int64_t count0,
                      void* stream) {
    using namespace cl;
    CL_REQUIRE(n_frames >= 0 && n_samples >= 0 && channels >= 1 && channels <= CL_MAX_CHANNELS);
    CL_REQUIRE(count0 >= 0 && max_dn > 0.0);
    if (n_frames == 0 || n_samples == 0) return CL_OK;
    CL_REQUIRE(frames && mean && m2);
    CL_REQUIRE(n_samples % channels == 0);
    const size_t smem = (lut ? 256 * channels : 256) * sizeof(double);
    welford_update_kernel<<<grid_for((n_samples + 3) / 4, kThreads, 8), kThreads, smem,
                            (cudaStream_t)stream>>>(frames, n_frames, n_samples, channels, lut,
                                                    max_dn, mean, m2, count0);
    return launched();
}

int cl_welford_finalize(const double* mean, const double* m2, int64_t count, int64_t n_samples,
                        double max_dn, double* sem, uint8_t* mean_u8, void* stream) {
    using namespace cl;
    CL_REQUIRE(n_samples >= 0 && count >= 0);
    if (n_samples == 0) return CL_OK;
    CL_REQUIRE(mean != nullptr);
    welford_finalize_kernel<<<grid_for(n_samples, kThreads, 8), kThreads, 0, (cudaStream_t)stream>>>(
        mean, m2, (double)count, n_samples, max_dn, sem, mean_u8);
    return launched();
}

size_t cl_welford_stack_workspace_bytes(int n_frames, int64_t n_samples) {
    (void)n_frames;
    // header + tie list: exact ties are ~n/F of the samples for noisy video but can be all of
    // them for adversarial input, so the list holds every sample index.
    return sizeof(cl::StackHeader) + (size_t)(n_samples > 0 ? n_samples : 0) * sizeof(uint32_t);
}

int cl_welford_stack(const uint8_t* frames, int n_frames, int64_t n_samples, int channels,
                     const double* lut, double max_dn, double* mean, double* sem, uint8_t* mean_u8,
                     void* workspace, size_t workspace_bytes, void* stream) {
    using namespace cl;
    CL_REQUIRE(n_frames >= 1 && n_samples >= 0 && channels >= 1 && channels <= CL_MAX_CHANNELS);
    CL_REQUIRE(max_dn > 0.0);
    if (n_samples == 0) return CL_OK;
    CL_REQUIRE(frames != nullptr);
    CL_REQUIRE(n_samples % channels == 0);
    if ((uint32_t)n_frames > kMaxFramesStack || n_samples > 0xFFFFFFFFll) return CL_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < cl_welford_stack_workspace_bytes(n_frames, n_samples))
        return CL_ERR_WORKSPACE;
    if (!aligned(workspace, 16)) return CL_ERR_ALIGNMENT;
    cudaStream_t s = (cudaStream_t)stream;
    StackHeader* hdr = reinterpret_cast<StackHeader*>(workspace);
    uint32_t* ties = reinterpret_cast<uint32_t*>(hdr + 1);
    const uint32_t cap = (uint32_t)n_samples;
    cudaError_t e = cudaMemsetAsync(hdr, 0, sizeof(StackHeader), s);
    if (e != cudaSuccess) return cuda_status(e);
    int st;
    if (lut) {
        int copies = 16;                       // lane-replicated table, as large as 96 KB of shared memory allow
        while (copies > 1 && (size_t)256 * channels * copies * sizeof(double) > 96 * 1024) copies /= 2;
        const size_t smem = (size_t)256 * channels * copies * sizeof(double);
        const unsigned grid = grid_for((n_samples + kLutSamples - 1) / kLutSamples, kLutThreads, 2);
        auto go = [&](auto kernel) -> int {
            cudaError_t ea = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (ea != cudaSuccess) return cuda_status(ea);
            kernel<<<grid, kLutThreads, smem, s>>>(frames, n_frames, n_samples, channels, lut, max_dn, mean, sem, mean_u8,
                                                   hdr, ties, cap);
            return launched();
        };
        st = copies == 16 ? go(welford_stack_lut_kernel<16>) : copies == 8 ? go(welford_stack_lut_kernel<8>)
                                                                           : go(welford_stack_lut_kernel<4>);
        if (st != CL_OK) return st;
    } else {
        // fast path needs 16-byte aligned frame rows
        const bool vec_ok = aligned(frames, 16) && (n_samples % 16 == 0) &&
                            (!mean || aligned(mean, 16)) && (!sem || aligned(sem, 16)) &&
                            (!mean_u8 || aligned(mean_u8, 16));
        const int64_t n_vec = vec_ok ? n_samples / 16 : 0;
        if (n_vec > 0) {
            // frame slices: enough threads to fill the machine when the image is small
            int slices = 1;
            const int64_t want = (int64_t)sm_count() * 1024;
            while (slices < 32 && n_vec * slices < want && slices * 2 <= n_frames) slices *= 2;
            const int64_t threads = ((n_vec * slices + 31) / 32) * 32;
            if (n_frames > kFrameBlock)
                welford_stack_u8_kernel<true><<<grid_for(threads, kThreads, 2), kThreads, 0, s>>>(
                    frames, n_frames, n_samples, slices, max_dn, mean, sem, mean_u8, hdr, ties, cap);
            else
                welford_stack_u8_kernel<false><<<grid_for(threads, kThreads, 3), kThreads, 0, s>>>(
                    frames, n_frames, n_samples, slices, max_dn, mean, sem, mean_u8, hdr, ties, cap);
            st = launched();
            if (st != CL_OK) return st;
        } else {
            // unaligned / ragged input: exact replay of every sample
            welford_replay_kernel<<<grid_for(n_samples, 128, 16), 128, 0, s>>>(
                frames, n_frames, n_samples, channels, nullptr, max_dn, hdr, nullptr, 0, 0, n_samples,
                true, mean, sem, mean_u8);
            return launched();
        }
    }
    // exact replay of the (near-)tie samples decides their uint8 mean
    if (mean_u8) {
        welford_tie_replay_kernel<<<sm_count() * 8, kReplayWarps * 32, 0, s>>>(
            frames, n_frames, n_samples, channels, lut, max_dn, hdr, ties, cap, mean_u8);
        st = launched();
        if (st != CL_OK) return st;
    }
    return CL_OK;
}

}  // extern "C"
