// K2: fused weighted HDR merge -- C ABI, generic register kernel and the stand-alone Measurand
// kernels (Gaussian weight, bad-pixel filter, flat-field normalisation, ROI means).
// Replaces exposure_series.py:317-397 + measurand.py:543-618 of the reference.
//
// Generic kernel ("algo 1"): any channel count, uint8 or uint16 DNs, std images or an STD table.
// Each thread owns 4 consecutive samples; pass A sums the Gaussian weights over the N exposures
// (DN bytes only), pass B re-reads the DNs (L1/L2 hits) together with the float64 std stream and
// accumulates value and variance in float64 registers.  Weight / ICRF tables are pre-multiplied
// ({w}, {w*g, dICRF}) and live in shared memory for 8-bit data, in an L2-resident workspace for
// 16-bit data.  Which kernel runs for a stack: the selection table above cl_hdr_merge.
#include "hdr_merge.cuh"

#include <algorithm>
#include <cstring>

namespace cl {
namespace {

constexpr int kThreads = 256;
constexpr int kVec = 4;

// ---- table construction -----------------------------------------------------------------------
// wt[d] = w(d / max_dn);  pb[d*C + c] = { w * lut[d][c], dlut[d][c] }
__global__ void build_tables_kernel(const double* __restrict__ lut, const double* __restrict__ dlut,
                                    double max_dn, int bits, int C, double* __restrict__ wt,
                                    double2* __restrict__ pb) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= bits) return;
    double w, dw;
    gaussian_weight(__ddiv_rn((double)d, max_dn), w, dw);
    wt[d] = w;
    for (int c = 0; c < C; ++c) pb[d * C + c] = make_double2(w * lut[d * C + c], dlut[d * C + c]);
}

template <typename DN>
__device__ __forceinline__ void load_dn4(const DN* __restrict__ img, int64_t base, int64_t n,
                                         uint32_t (&d)[kVec]) {
    if (base + kVec <= n) {
        if (sizeof(DN) == 1) {
            const uint32_t u = *reinterpret_cast<const uint32_t*>(img + base);
            d[0] = u & 0xFF; d[1] = (u >> 8) & 0xFF; d[2] = (u >> 16) & 0xFF; d[3] = u >> 24;
        } else {
            const uint2 u = *reinterpret_cast<const uint2*>(img + base);
            d[0] = u.x & 0xFFFF; d[1] = u.x >> 16; d[2] = u.y & 0xFFFF; d[3] = u.y >> 16;
        }
    } else {
#pragma unroll
        for (int j = 0; j < kVec; ++j) d[j] = (base + j < n) ? (uint32_t)img[base + j] : 0u;
    }
}

__device__ __forceinline__ void load_f64x4(const double* __restrict__ a, int64_t base, int64_t n,
                                           double (&v)[kVec]) {
    if (base + kVec <= n) {
        const double2 lo = *reinterpret_cast<const double2*>(a + base);
        const double2 hi = *reinterpret_cast<const double2*>(a + base + 2);
        v[0] = lo.x; v[1] = lo.y; v[2] = hi.x; v[3] = hi.y;
    } else {
#pragma unroll
        for (int j = 0; j < kVec; ++j) v[j] = (base + j < n) ? a[base + j] : 0.0;
    }
}

template <typename DN, bool TAB_SMEM>
__global__ void __launch_bounds__(kThreads)
merge_generic_kernel(const __grid_constant__ MergeParams p, const int64_t first_item) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int C = p.C;
    const double* wt;
    const double2* pb;
    const double* stdlut = p.std_lut;
    if (TAB_SMEM) {
        double* s_wt = reinterpret_cast<double*>(smem_raw);
        double2* s_pb = reinterpret_cast<double2*>(s_wt + p.bits);
        double* s_sl = reinterpret_cast<double*>(s_pb + p.bits * C);
        for (int d = threadIdx.x; d < p.bits; d += blockDim.x) {
            double w, dw;
            gaussian_weight(__ddiv_rn((double)d, p.max_dn), w, dw);
            s_wt[d] = w;
            for (int c = 0; c < C; ++c) {
                s_pb[d * C + c] = make_double2(w * p.lut[d * C + c], p.dlut[d * C + c]);
                if (p.std_lut) s_sl[d * C + c] = p.std_lut[d * C + c];
            }
        }
        __syncthreads();
        wt = s_wt;
        pb = s_pb;
        if (p.std_lut) stdlut = s_sl;
    } else {
        wt = p.g_wt;
        pb = p.g_pb;
    }

    const int64_t n = (int64_t)p.H * p.W * C;
    const int64_t n_items = (n + kVec - 1) / kVec;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t row = (int64_t)p.W * C;
    for (int64_t it = first_item + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < n_items;
         it += stride) {
        const int64_t base = it * kVec;
        int cidx[kVec];
#pragma unroll
        for (int j = 0; j < kVec; ++j) cidx[j] = (int)((base + j) % C);

        // ---- pass A: sum of weights (exposure_series.py:328-343) ----
        double S[kVec] = {0.0, 0.0, 0.0, 0.0};
        uint32_t hot_any = 0;  // bit k set: this item has a bad pixel in exposure k
        for (int k = 0; k < p.n; ++k) {
            uint32_t d[kVec];
            load_dn4(reinterpret_cast<const DN*>(p.dn[k]), base, n, d);
            if (p.dark[k]) {
                uint32_t dk[kVec];
                load_dn4(reinterpret_cast<const DN*>(p.dark[k]), base, n, dk);
#pragma unroll
                for (int j = 0; j < kVec; ++j) {
                    if (dk[j] >= p.hot_dn[k] && base + j < n) {
                        const int64_t i = base + j;
                        const int y = (int)(i / row);
                        const int x = (int)((i - (int64_t)y * row) / C);
                        d[j] = median_dn(reinterpret_cast<const DN*>(p.dn[k]), y, x, cidx[j], p.H,
                                         p.W, C, p.K);
                        hot_any |= 1u << k;
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < kVec; ++j) S[j] += wt[d[j]];
        }
        double rS[kVec];
#pragma unroll
        for (int j = 0; j < kVec; ++j) rS[j] = 1.0 / S[j];

        // ---- pass B: weighted radiance and variance (exposure_series.py:372-394) ----
        double av[kVec] = {0.0, 0.0, 0.0, 0.0}, as[kVec] = {0.0, 0.0, 0.0, 0.0};
        for (int k = 0; k < p.n; ++k) {
            const DN* img = reinterpret_cast<const DN*>(p.dn[k]);
            uint32_t d[kVec];
            load_dn4(img, base, n, d);
            double sg[kVec];
            if (p.std[k]) {
                load_f64x4(p.std[k], base, n, sg);
            } else {
#pragma unroll
                for (int j = 0; j < kVec; ++j) sg[j] = stdlut[(int64_t)d[j] * C + cidx[j]];
            }
            if (hot_any & (1u << k)) {
                uint32_t dk[kVec];
                load_dn4(reinterpret_cast<const DN*>(p.dark[k]), base, n, dk);
#pragma unroll
                for (int j = 0; j < kVec; ++j) {
                    if (dk[j] >= p.hot_dn[k] && base + j < n) {
                        const int64_t i = base + j;
                        const int y = (int)(i / row);
                        const int x = (int)((i - (int64_t)y * row) / C);
                        d[j] = median_dn(img, y, x, cidx[j], p.H, p.W, C, p.K);
                        sg[j] = median_std(p.std[k], img, p.std_lut, y, x, cidx[j], p.H, p.W, C, p.K);
                    }
                }
            }
            const double rt = p.inv_t[k];
#pragma unroll
            for (int j = 0; j < kVec; ++j) {
                const double2 e = pb[(int64_t)d[j] * C + cidx[j]];
                merge_accumulate(wt[d[j]], e.x, e.y, kappa_of(d[j], p.kappa_scale), sg[j], rS[j], rt,
                                 av[j], as[j]);
            }
        }

        double ov[kVec], os[kVec];
#pragma unroll
        for (int j = 0; j < kVec; ++j) ov[j] = av[j] * rS[j];
        if (p.flat_bytes) {
#pragma unroll
            for (int j = 0; j < kVec; ++j) {
                os[j] = 0.0;
                if (base + j < n)
                    flat_apply(ov[j], os[j], (as[j] * rS[j]) * rS[j],
                               flat_recip(p.flat, p.flat_bytes, base + j, p.max_dn), p.flat_std[base + j],
                               p.flat_means[cidx[j]], p.flat_means[C + cidx[j]]);
            }
        } else {
#pragma unroll
            for (int j = 0; j < kVec; ++j) os[j] = sqrt(as[j]) * rS[j];
        }
        if (base + kVec <= n) {
            *reinterpret_cast<double2*>(p.out_val + base) = make_double2(ov[0], ov[1]);
            *reinterpret_cast<double2*>(p.out_val + base + 2) = make_double2(ov[2], ov[3]);
            *reinterpret_cast<double2*>(p.out_std + base) = make_double2(os[0], os[1]);
            *reinterpret_cast<double2*>(p.out_std + base + 2) = make_double2(os[2], os[3]);
        } else {
#pragma unroll
            for (int j = 0; j < kVec; ++j)
                if (base + j < n) {
                    p.out_val[base + j] = ov[j];
                    p.out_std[base + j] = os[j];
                }
        }
    }
}

template <typename DN>
int launch_generic(const MergeParams& p, bool tab_smem, int64_t first_item, cudaStream_t stream) {
    const int64_t n = (int64_t)p.H * p.W * p.C;
    const int64_t n_items = (n + kVec - 1) / kVec - first_item;
    if (n_items <= 0) return CL_OK;
    int64_t blocks = (n_items + kThreads - 1) / kThreads;
    const int64_t cap = (int64_t)sm_count() * 6;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    if (tab_smem) {
        const size_t smem = (size_t)p.bits * 8 + (size_t)p.bits * p.C * 16 +
                            (p.std_lut ? (size_t)p.bits * p.C * 8 : 0);
        auto k = merge_generic_kernel<DN, true>;
        if (smem > 48 * 1024) {
            cudaError_t e =
                cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return cuda_status(e);
        }
        k<<<(unsigned)blocks, kThreads, smem, stream>>>(p, first_item);
    } else {
        merge_generic_kernel<DN, false><<<(unsigned)blocks, kThreads, 0, stream>>>(p, first_item);
    }
    return launched();
}

// ---- bad-pixel buckets (staged path) ----------------------------------------------------------------
// Streams the dark frames once (64 bytes per thread in flight, SIMD byte compare) and files every
// (sample, exposure) whose dark DN reaches the exposure's integer threshold in the bucket of the
// 512-pixel tile it belongs to: {pixel-in-tile, channel, exposure}.  The merge kernel's median warp
// computes the repaired DN / sigma for its next tile's bucket while the consumers are still busy
// with the current tile, so the repair costs neither a separate gather pass nor a stall.  Samples
// that do not fit a bucket (more than kBucketCap bad pairs in one tile) go to the global fix-up
// list and are recomputed in full by merge_fixup_kernel.
constexpr int kScanThreads = 256;
constexpr int kScanVecs = 4;

__device__ __forceinline__ void file_hit(const MergeParams& p, int k, uint32_t sample) {
    const uint32_t px = sample / 3u, c = sample - px * 3u;
    const uint32_t tile = px / kStagedTilePx;
    if ((int)tile >= p.n_full_tiles) return;            // ragged tail: the generic kernel repairs inline
    const uint32_t slot = atomicAdd(p.bucket_counts + (size_t)tile * 4, 1u);
    if (slot < (uint32_t)kBucketCap) {
        p.bucket_entries[((size_t)tile * kBucketCap + slot) * 4] =
            (px - tile * kStagedTilePx) | (c << 9) | ((uint32_t)k << 11);
    } else {
        const uint32_t g = atomicAdd(&p.hot_list[0], 1u);
        if (g < p.hot_cap) p.hot_list[kHotListHeader + g] = sample;
    }
}

// byte >= thr for the four bytes of x, flagged in bit 7 of each byte (SWAR; __vcmpgeu4 is emulated):
//   thr <= 128: b7 | carry((b & 0x7f) + 128 - thr)      thr > 128: b7 & carry((b & 0x7f) + 256 - thr)
__device__ __forceinline__ uint32_t bytes_ge(uint32_t x, uint32_t add, bool low) {
    const uint32_t lo = (x & 0x7f7f7f7fu) + add;
    return (low ? (x | lo) : (x & lo)) & 0x80808080u;
}

// Work unit = (dark frame j, run of kScanThreads * kScanVecs 16-byte vectors); the units of all frames
// form one flat list that the (exactly one wave of) blocks stride over, so no wave is part-empty.
// Hits are parked in a shared-memory list (a shared atomic, ~100 cycles) and filed into the global
// buckets once per block at the end: a global atomic inside the streaming loop costs ~1.5 us of
// latency per unit for every warp that sees a hit, which is most of them.
constexpr int kScanListCap = 2048;       // {sample, exposure} pairs per block; overflow files directly

__global__ void __launch_bounds__(kScanThreads)
dark_scan_kernel(const __grid_constant__ MergeParams p) {
    __shared__ uint2 hits[kScanListCap];
    __shared__ uint32_t n_hits;
    if (threadIdx.x == 0) n_hits = 0;
    __syncthreads();
    auto park = [&](int k, uint32_t sample) {
        const uint32_t slot = atomicAdd(&n_hits, 1u);
        if (slot < (uint32_t)kScanListCap) hits[slot] = make_uint2(sample, (uint32_t)k);
        else file_hit(p, k, sample);
    };
    // 32-bit index arithmetic throughout: the staged path requires fewer than 2^32 samples
    const int64_t n = (int64_t)p.H * p.W * p.C;
    const uint32_t n_vec = (uint32_t)(n / 16);  // full 16-byte vectors per dark frame
    constexpr uint32_t kUnitVecs = kScanThreads * kScanVecs;
    const uint32_t units_per_frame = (n_vec + kUnitVecs - 1) / kUnitVecs;
    const uint32_t total = units_per_frame * (uint32_t)p.n_dark;
    for (uint32_t unit = blockIdx.x; unit < total; unit += gridDim.x) {
        const uint32_t j = unit / units_per_frame;
        const uint32_t base = (unit - j * units_per_frame) * kUnitVecs + threadIdx.x;
        const int k = p.dark_k[j];
        const uint4* src = reinterpret_cast<const uint4*>(p.dark[k]);
        const uint32_t thr = p.hot_dn[k];
        const bool low = thr <= 128u;
        const uint32_t add = (low ? 128u - thr : 256u - thr) * 0x01010101u;
        uint4 q[kScanVecs];
#pragma unroll
        for (int u = 0; u < kScanVecs; ++u) {
            const uint32_t v = base + u * kScanThreads;
            q[u] = v < n_vec ? __ldg(src + v) : make_uint4(0, 0, 0, 0);     // (zeros never reach a threshold >= 1 ...
        }
#pragma unroll
        for (int u = 0; u < kScanVecs; ++u) {
            const uint32_t v = base + u * kScanThreads;
            const uint32_t h[4] = {bytes_ge(q[u].x, add, low), bytes_ge(q[u].y, add, low),
                                   bytes_ge(q[u].z, add, low), bytes_ge(q[u].w, add, low)};
            if ((h[0] | h[1] | h[2] | h[3]) == 0u || v >= n_vec) continue;  // ... and threshold 0 is caught here)
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                uint32_t m = h[w];
                while (m) {
                    const int b = (__ffs(m) - 1) >> 3;
                    park(k, v * 16 + w * 4 + b);
                    m &= m - 1;
                }
            }
        }
    }
    // ragged last (n % 16) bytes of every dark frame: a handful of bytes, filed directly by block 0
    // (kept out of the park() path: a second call site there doubled the kernel's run time)
    const uint32_t rag = (uint32_t)(n - (int64_t)n_vec * 16);
    if (blockIdx.x == 0 && rag != 0u) {
        for (uint32_t t = threadIdx.x; t < rag * (uint32_t)p.n_dark; t += kScanThreads) {
            const uint32_t jr = t / rag;
            const uint32_t i = n_vec * 16u + (t - jr * rag);
            const int k = p.dark_k[jr];
            if (reinterpret_cast<const uint8_t*>(p.dark[k])[i] >= p.hot_dn[k]) file_hit(p, k, i);
        }
    }
    __syncthreads();
    const uint32_t parked = min(n_hits, (uint32_t)kScanListCap);
    for (uint32_t e = threadIdx.x; e < parked; e += kScanThreads) file_hit(p, (int)hits[e].y, hits[e].x);
}

// The single-pass kernel's rule for one sample (hdr_merge_stream.cu): the expanded variance, unless it cancelled
// (q < kStreamCancel * A), in which case the exact two-pass formula.  Same operations in the same order as the
// kernel, so a sample gets the same bits whichever of the two computes it.
__device__ __noinline__ void recompute_sample_stream(const MergeParams& p, int64_t i) {
    const int C = p.C;
    const int c = (int)(i % C);
    const int64_t px = i / C;
    const int y = (int)(px / p.W), x = (int)(px - (int64_t)y * p.W);
    double S = 0.0, av = 0.0, A = 0.0, B = 0.0, Cc = 0.0;
    for (int k = 0; k < p.n; ++k) {
        const uint8_t* img = reinterpret_cast<const uint8_t*>(p.dn[k]);
        uint32_t d = img[i];
        const bool hot = p.dark[k] && (uint32_t) reinterpret_cast<const uint8_t*>(p.dark[k])[i] >= p.hot_dn[k];
        if (hot) d = median_dn(img, y, x, c, p.H, p.W, C, p.K);
        const double sg = hot ? median_std(p.std[k], img, p.std_lut, y, x, c, p.H, p.W, C, p.K)
                              : p.std[k] ? p.std[k][i] : p.std_lut[(int64_t)d * C + c];
        double w, dw;
        gaussian_weight(__ddiv_rn((double)d, p.max_dn), w, dw);
        const double p1 = w * p.lut[(int64_t)d * C + c];
        if (p.stream_mode == 2) {           // the STD-table kernel's arithmetic (products per DN, then 1/t)
            double xu, eu;
            lut_products(w, p1, p.dlut[(int64_t)d * C + c], kappa_of(d, p.kappa_scale), sg, xu, eu);
            merge_accumulate_expanded_lut(w, p1, xu, eu, p.inv_t[k], S, av, A, B, Cc);
        } else {
            merge_accumulate_expanded(w, p1, p.dlut[(int64_t)d * C + c], kappa_of(d, p.kappa_scale), sg, p.inv_t[k], S,
                                      av, A, B, Cc);
        }
    }
    const double rS = 1.0 / S;
    const double q = expanded_variance(A, B, Cc, rS);
    if (q < kStreamCancel * A) {
        recompute_sample<uint8_t>(p, i);
        return;
    }
    double ov = av * rS, os;
    if (p.flat_bytes)
        flat_apply(ov, os, (q * rS) * rS, flat_recip(p.flat, p.flat_bytes, i, p.max_dn), p.flat_std[i],
                   p.flat_means[c], p.flat_means[C + c]);
    else
        os = sqrt(q) * rS;
    p.out_val[i] = ov;
    p.out_std[i] = os;
}

__global__ void __launch_bounds__(128)
merge_fixup_kernel(const __grid_constant__ MergeParams p) {
    const uint32_t count = p.hot_list[0];
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (count <= p.hot_cap) {
        for (int64_t t = tid; t < count; t += stride) {
            const int64_t i = (int64_t)p.hot_list[kHotListHeader + t];
            if (p.stream_mode) recompute_sample_stream(p, i);
            else recompute_sample<uint8_t>(p, i);
        }
        return;
    }
    // the list overflowed (pathological: most of the image is "bad", or most of it cancels in the single-pass
    // kernel): rescan every full-tile sample
    const int64_t n = (int64_t)p.H * p.W * p.C;
    const int64_t n_stream = p.stream_mode ? (int64_t)p.n_full_tiles * kStagedTilePx * 3 : 0;
    for (int64_t i = tid; i < n; i += stride) {
        if (i < n_stream) {
            recompute_sample_stream(p, i);
            continue;
        }
        bool any = false;
        for (int k = 0; k < p.n && !any; ++k)
            any = p.dark[k] && reinterpret_cast<const uint8_t*>(p.dark[k])[i] >= p.hot_dn[k];
        if (any) recompute_sample<uint8_t>(p, i);
    }
}

// ---- ROI means ------------------------------------------------------------------------------------
constexpr int kRoiThreads = 256;

// CT = compile-time channel count (keeps the accumulators in registers); CT == 0: run-time C <= 8.
// All kRoiBlocks blocks are resident at once (one wave) and every thread keeps four pixels in flight.
template <int CT>
__global__ void __launch_bounds__(kRoiThreads, CT ? 3 : 1)
roi_partial_kernel(const void* __restrict__ flat, int flat_bytes, double max_dn,
                   const double* __restrict__ flat_std, int W, int C_rt, int r0, int c0, int rh, int rw,
                   double* __restrict__ partial, unsigned int* __restrict__ ticket, double count,
                   double* __restrict__ out) {
    // block b reduces ROI pixels [b*chunk, (b+1)*chunk) for every channel, fixed order
    constexpr int CM = CT ? CT : CL_MAX_CHANNELS;
    constexpr int kPix = 4;
    const int C = CT ? CT : C_rt;
    __shared__ double red[kRoiThreads / 32][2 * CM];
    const int64_t npx = (int64_t)rh * rw;
    const int64_t chunk = (npx + gridDim.x - 1) / gridDim.x;
    const int64_t lo = (int64_t)blockIdx.x * chunk;
    const int64_t hi = lo + chunk < npx ? lo + chunk : npx;
    double acc[2 * CM];
#pragma unroll
    for (int c = 0; c < 2 * CM; ++c) acc[c] = 0.0;
    for (int64_t q0 = lo + threadIdx.x; q0 < hi; q0 += (int64_t)kPix * kRoiThreads) {
        double f[kPix][CM], sd[kPix][CM];
#pragma unroll
        for (int u = 0; u < kPix; ++u) {
            const int64_t q = q0 + (int64_t)u * kRoiThreads;
            const bool on = q < hi;
            int64_t i = 0;
            if (on) {
                int64_t y, x;
                if (npx < ((int64_t)1 << 31)) {          // 32-bit divide when it fits (the common case)
                    const uint32_t yy = (uint32_t)q / (uint32_t)rw;
                    y = yy; x = (uint32_t)q - yy * (uint32_t)rw;
                } else {
                    y = q / rw; x = q - y * rw;
                }
                i = ((r0 + y) * W + (c0 + x)) * C;
            }
#pragma unroll
            for (int c = 0; c < CM; ++c) {
                const bool live = on && c < C;
                f[u][c] = live ? flat_value(flat, flat_bytes, i + c, max_dn) : 0.0;
                sd[u][c] = live ? flat_std[i + c] : 0.0;
            }
        }
#pragma unroll
        for (int u = 0; u < kPix; ++u) {                 // pixel order q0, q0 + 256, ... as a one-pixel loop would
            if (q0 + (int64_t)u * kRoiThreads >= hi) break;
#pragma unroll
            for (int c = 0; c < CM; ++c) {
                if (c >= C) break;
                acc[c] += f[u][c];
                acc[CM + c] += sd[u][c];
            }
        }
    }
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
#pragma unroll
    for (int c = 0; c < 2 * CM; ++c) {                   // acc = [mean sums x CM | std sums x CM], red = [C | C]
        const int cc = c < CM ? c : c - CM;
        if (cc >= C) continue;
        const double v = warp_sum(acc[c]);
        if (lane == 0) red[warp][c < CM ? cc : C + cc] = v;
    }
    __syncthreads();
    if (threadIdx.x < 2 * C) {
        double s = 0.0;
        for (int w = 0; w < kRoiThreads / 32; ++w) s += red[w][threadIdx.x];
        partial[(int64_t)blockIdx.x * 2 * C + threadIdx.x] = s;
    }
    // The block that draws the last ticket combines all partials -- in a FIXED order (lanes stride over the
    // blocks, then an xor tree), so the result does not depend on which block that is.  One launch instead of
    // two: the second kernel cost as much as the first (7.6 us of launch + latency for 2C numbers).
    __shared__ bool last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    if (warp < 2 * C) {                                   // kRoiThreads / 32 = 8 warps >= 2C for C <= 4
        for (int c = warp; c < 2 * C; c += kRoiThreads / 32) {
            double s = 0.0;
#pragma unroll 8
            for (int b = lane; b < (int)gridDim.x; b += 32) s += __ldcg(partial + (int64_t)b * 2 * C + c);
            s = warp_sum(s);
            if (lane == 0) out[c] = s / count;
        }
    }
}

constexpr int kRoiBlocks = 444;      // 148 SMs x 3 resident blocks; fixed so the summation order is machine-independent

// ---- stand-alone Measurand kernels ------------------------------------------------------------------
__global__ void gaussian_weight_kernel(const double* __restrict__ val, double* __restrict__ w,
                                       double* __restrict__ dw, int64_t n) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double a, b;
        gaussian_weight(val[i], a, b);
        w[i] = a;
        if (dw) dw[i] = b;
    }
}

__global__ void bad_pixel_filter_kernel(const double* __restrict__ val, const double* __restrict__ std,
                                        const double* __restrict__ dark, double thr, int K, int H,
                                        int W, int C, double* __restrict__ out_val,
                                        double* __restrict__ out_std) {
    const int64_t n = (int64_t)H * W * C;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t row = (int64_t)W * C;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double v = val[i];
        double s = std ? std[i] : 0.0;
        if (dark[i] > thr) {
            const int y = (int)(i / row);
            const int x = (int)((i - (int64_t)y * row) / C);
            const int c = (int)(i % C);
            double win[CL_MAX_MEDIAN_KERNEL * CL_MAX_MEDIAN_KERNEL];
            const int lo = K / 2;
            for (int pass = 0; pass < (std ? 2 : 1); ++pass) {
                const double* src = pass ? std : val;
                int m = 0;
                for (int dy = -lo; dy < K - lo; ++dy) {
                    const int yy = reflect_index(y + dy, H);
                    for (int dx = -lo; dx < K - lo; ++dx)
                        win[m++] = src[((int64_t)yy * W + reflect_index(x + dx, W)) * C + c];
                }
                const double med = select_rank(win, m, (K * K) / 2);
                if (pass) s = med; else v = med;
            }
        }
        out_val[i] = v;
        if (std) out_std[i] = s;
    }
}

__global__ void flat_normalize_kernel(const double* __restrict__ val, const double* __restrict__ std,
                                      const double* __restrict__ fv, const double* __restrict__ fs,
                                      const double* __restrict__ means, int64_t n, int C,
                                      double* __restrict__ out_val, double* __restrict__ out_std) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int c = (int)(i % C);
        double v = val[i], s = std[i];
        flat_apply(v, s, s * s, 1.0 / fv[i], fs[i], means[c], means[C + c]);
        out_val[i] = v;
        out_std[i] = s;
    }
}

inline unsigned grid_for(int64_t n, int threads) {
    int64_t b = (n + threads - 1) / threads;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (b > cap) b = cap;
    return (unsigned)(b < 1 ? 1 : b);
}

size_t table_bytes(int bits, int C) { return (size_t)bits * 8 + (size_t)bits * C * 16; }

// The workspace of cl_hdr_merge: cl_hdr_merge_workspace_bytes reports `total`, cl_hdr_merge carves these offsets.
//   [0, tables)         more than 256 DN rows: the generic kernel's tables or the 16-bit kernel's interleaved rows,
//                       whichever runs (sized for the larger)
//   [counts, list)      8-bit C = 3 / 1 stacks unless algo = 1: per-tile bad-pixel bucket counts {count, pad x3}
//   [list, entries)     the work list, right behind the counts so that one memset clears both: kHotListHeader
//                       words (hot_list[0] counts the entries) and hot_cap entries, padded to 16 bytes
//   [entries, end)      per-tile bucket entries {meta, pad, sigma}, 16-byte aligned for the bulk copies
// `total` reserves the whole 16 bytes the padding can take.
struct MergeWorkspace {
    size_t tables = 0, counts = 0, list = 0, entries = 0, end = 0, total = 0;
    size_t hot_cap = 0;
    int64_t n_full_tiles = 0;
};

MergeWorkspace merge_workspace(const cl_hdr_merge_args& a) {
    MergeWorkspace w;
    if (a.bits > 256)
        w.tables = std::max(table_bytes(a.bits, a.channels), wide_table_bytes(a.bits, a.channels, a.std_lut != nullptr));
    w.counts = w.list = w.entries = w.end = w.total = w.tables;
    if (a.dn_bytes == 1 && (a.channels == 3 || a.channels == 1) && a.algo != 1) {
        const int64_t n = (int64_t)a.height * a.width * a.channels;
        w.n_full_tiles = n / (kStagedTilePx * 3);
        w.hot_cap = (size_t)std::max<int64_t>(n / 16, 65536);
        const size_t entries_bytes = (size_t)w.n_full_tiles * kBucketCap * 16;
        w.list = w.counts + (size_t)w.n_full_tiles * 16;
        const size_t list_end = w.list + (kHotListHeader + w.hot_cap) * sizeof(uint32_t);
        w.entries = (list_end + 15) / 16 * 16;
        w.end = w.entries + entries_bytes;
        w.total = list_end + 16 + entries_bytes;
    }
    return w;
}

// generic kernel: any stack; its tables are built in shared memory, or (more than 256 DN rows) in the workspace
int try_merge_generic(MergeParams p, void* workspace, size_t workspace_bytes, cudaStream_t stream) {
    const bool tab_smem = p.bits <= 256;
    if (!tab_smem) {
        if (!workspace || workspace_bytes < table_bytes(p.bits, p.C)) return CL_ERR_WORKSPACE;
        if (!aligned(workspace, 16)) return CL_ERR_ALIGNMENT;
        double* wt = reinterpret_cast<double*>(workspace);
        double2* pb = reinterpret_cast<double2*>(wt + p.bits);
        build_tables_kernel<<<(p.bits + 255) / 256, 256, 0, stream>>>(p.lut, p.dlut, p.max_dn, p.bits, p.C, wt, pb);
        const int st = launched();
        if (st != CL_OK) return st;
        p.g_wt = wt;
        p.g_pb = pb;
    }
    return p.max_dn == 255.0 ? launch_generic<uint8_t>(p, tab_smem, 0, stream)
                             : launch_generic<uint16_t>(p, tab_smem, 0, stream);
}

}  // namespace

int launch_merge_generic_range(const MergeParams& p, int64_t first_item, cudaStream_t stream) {
    return launch_generic<uint8_t>(p, true, first_item, stream);
}

int launch_dark_scan(const MergeParams& p, cudaStream_t stream) {
    // bucket counts and the hot-list counter are contiguous: one linear memset
    cudaError_t e = cudaMemsetAsync(p.bucket_counts, 0,
                                    ((size_t)p.n_full_tiles * 4 + kHotListHeader) * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return cuda_status(e);
    int per_sm = 0;                      // resident blocks per SM: the grid is exactly one wave
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dark_scan_kernel, kScanThreads, 0) != cudaSuccess ||
        per_sm < 1)
        per_sm = 4;
    dark_scan_kernel<<<sm_count() * per_sm, kScanThreads, 0, stream>>>(p);
    return launched();
}

int clear_hot_list(const MergeParams& p, cudaStream_t stream) {
    return cuda_status(cudaMemsetAsync(p.hot_list, 0, kHotListHeader * sizeof(uint32_t), stream));
}

int launch_merge_fixup(const MergeParams& p, cudaStream_t stream) {
    merge_fixup_kernel<<<sm_count() * 8, 128, 0, stream>>>(p);
    return launched();
}

}  // namespace cl

extern "C" {

size_t cl_hdr_merge_workspace_bytes(const cl_hdr_merge_args* a) {
    return a ? cl::merge_workspace(*a).total : 0;
}

// Which kernel runs.  The requested algo names an ordered list of candidates; the first that handles the stack and
// has its part of the workspace runs, and each is asked once:
//   algo 0 (auto)   16-bit, single-pass, single-pass STD-table, staged, staged STD-table, generic
//   algo 1          generic
//   algo 2          staged, staged STD-table
//   algo 3          16-bit
//   algo 4          single-pass, single-pass STD-table
//
//   candidate                                handles                                        workspace
//   16-bit (hdr_merge_wide.cu)               uint16, N <= 16: the pipelined kernel when     32-byte-aligned table rows
//                                            every exposure has an uncertainty image or
//                                            none has, round 1's kernel when they mix
//   single-pass (hdr_merge_stream.cu)        tile stack, uncertainty images, N >= 2         work list
//   single-pass STD-table (.._stream_lut.cu) tile stack, STD table, N >= 2                  work list
//   staged (hdr_merge_staged.cu)             tile stack, uncertainty images                 work list with dark frames
//   staged STD-table (.._staged_lut.cu)      tile stack, STD table                          work list with dark frames
//   generic (this file)                      any stack                                      tables above 256 DN rows
// A tile stack is an 8-bit RGB or mono stack of at least one 512-pixel tile (staged_common.cuh: tile_stack), and the
// tile kernel's shared-memory layout must fit it.  When no candidate runs, nothing has been enqueued and the call
// returns CL_ERR_WORKSPACE if a candidate lacked only its workspace, CL_ERR_UNSUPPORTED otherwise.
int cl_hdr_merge(const cl_hdr_merge_args* a, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace cl;
    CL_REQUIRE(a != nullptr);
    CL_REQUIRE(a->algo >= 0 && a->algo <= 4);
    CL_REQUIRE(a->n_exposures >= 1 && a->n_exposures <= CL_MAX_EXPOSURES);
    CL_REQUIRE(a->height >= 0 && a->width >= 0 && a->channels >= 1 && a->channels <= CL_MAX_CHANNELS);
    CL_REQUIRE(a->dn_bytes == 1 || a->dn_bytes == 2);
    CL_REQUIRE((a->dn_bytes == 1 && a->bits >= 256) || (a->dn_bytes == 2 && a->bits >= 65536));
    CL_REQUIRE(a->bits <= 65536);
    CL_REQUIRE(a->dn && a->exposure_s && a->lut && a->dlut && a->out_val && a->out_std);
    CL_REQUIRE(a->median_kernel >= 1 && a->median_kernel <= CL_MAX_MEDIAN_KERNEL);
    CL_REQUIRE(a->flat_bytes == 0 || a->flat_bytes == 1 || a->flat_bytes == 2 || a->flat_bytes == 8);
    if (a->flat_bytes) CL_REQUIRE(a->flat && a->flat_std && a->flat_means);
    if ((int64_t)a->height * a->width == 0) return CL_OK;
    if ((int64_t)a->height * a->width * a->channels > (int64_t)1 << 40) return CL_ERR_UNSUPPORTED;

    MergeParams p;
    std::memset(&p, 0, sizeof(p));
    p.n = a->n_exposures; p.H = a->height; p.W = a->width; p.C = a->channels; p.bits = a->bits;
    p.K = a->median_kernel;
    p.max_dn = a->dn_bytes == 1 ? 255.0 : 65535.0;
    p.kappa_scale = -60.0 / p.max_dn;
    p.lut = a->lut; p.dlut = a->dlut; p.std_lut = a->std_lut;
    p.flat = a->flat; p.flat_std = a->flat_std; p.flat_means = a->flat_means;
    p.flat_bytes = a->flat_bytes;
    p.out_val = a->out_val; p.out_std = a->out_std;
    if (!aligned(p.out_val, 16) || !aligned(p.out_std, 16)) return CL_ERR_ALIGNMENT;
    bool all_std = true;
    for (int k = 0; k < p.n; ++k) {
        CL_REQUIRE(a->dn[k] != nullptr);
        p.dn[k] = a->dn[k];
        p.std[k] = a->std ? a->std[k] : nullptr;
        if (!p.std[k]) {
            all_std = false;
            CL_REQUIRE(a->std_lut != nullptr);
        }
        if (!aligned(p.dn[k], 16) || (p.std[k] && !aligned(p.std[k], 16))) return CL_ERR_ALIGNMENT;
        const double t = a->exposure_s[k];
        CL_REQUIRE(t == t && t != 0.0);
        p.inv_t[k] = 1.0 / t;
        p.dark[k] = a->dark ? a->dark[k] : nullptr;
        p.hot_dn[k] = 0xFFFFFFFFu;
        if (p.dark[k]) {
            if (!aligned(p.dark[k], 16)) return CL_ERR_ALIGNMENT;
            const double scale = a->dark_scale ? a->dark_scale[k] : 1.0;
            CL_REQUIRE(scale > 0.0);
            // mask = (dark_dn / MAX_DN) [* scale] > threshold  (image_set.py:223,260;
            // measurand.py:545) evaluated in IEEE double exactly as NumPy does; it is monotone
            // in dark_dn, so it reduces to an integer comparison on the device.
            const uint32_t top = (uint32_t)p.max_dn;
            for (uint32_t d = 0; d <= top; ++d) {
                volatile double v = (double)d / p.max_dn;
                if (scale != 1.0) v = v * scale;
                if (v > a->dark_threshold) { p.hot_dn[k] = d; break; }
            }
            p.any_dark = 1;
            if (p.hot_dn[k] <= top) p.dark_k[p.n_dark++] = (uint8_t)k;
        }
    }

    // the workspace, carved as merge_workspace() lays it out
    const MergeWorkspace ws = merge_workspace(*a);
    unsigned char* w = static_cast<unsigned char*>(workspace);
    if (ws.tables && w && aligned(w, 32) && workspace_bytes >= wide_table_bytes(p.bits, p.C, !all_std))
        p.g_tab32 = reinterpret_cast<const double2*>(w);
    if (ws.end > ws.counts && w && aligned(w, 16) && workspace_bytes >= ws.end) {
        p.n_full_tiles = (int32_t)ws.n_full_tiles;
        p.bucket_counts = reinterpret_cast<uint32_t*>(w + ws.counts);
        p.hot_list = reinterpret_cast<uint32_t*>(w + ws.list);
        p.hot_cap = (uint32_t)ws.hot_cap;
        p.bucket_entries = reinterpret_cast<uint32_t*>(w + ws.entries);
    }

    enum Candidate { kWide, kStream, kStreamLut, kStaged, kStagedLut, kGeneric, kEnd };
    static constexpr Candidate kCandidates[5][7] = {
        {kWide, kStream, kStreamLut, kStaged, kStagedLut, kGeneric, kEnd},
        {kGeneric, kEnd},
        {kStaged, kStagedLut, kEnd},
        {kWide, kEnd},
        {kStream, kStreamLut, kEnd},
    };
    cudaStream_t s = (cudaStream_t)stream;
    int status = CL_ERR_UNSUPPORTED;
    for (const Candidate* c = kCandidates[a->algo]; *c != kEnd; ++c) {
        int st;
        switch (*c) {
            case kWide: st = try_merge_wide(p, s); break;
            case kStream: st = try_merge_stream(p, s); break;
            case kStreamLut: st = try_merge_stream_lut(p, s); break;
            case kStaged: st = try_merge_staged(p, s); break;
            case kStagedLut: st = try_merge_staged_lut(p, s); break;
            default: st = try_merge_generic(p, workspace, workspace_bytes, s); break;
        }
        if (st == CL_ERR_WORKSPACE) status = st;
        else if (st != CL_ERR_UNSUPPORTED) return st;
    }
    return status;
}

size_t cl_flat_roi_means_workspace_bytes(int height, int width, int channels) {
    (void)height; (void)width;
    return (size_t)cl::kRoiBlocks * 2 * (channels > 0 ? channels : 1) * sizeof(double) + 16;   // partials + ticket
}

int cl_flat_roi_means(const void* flat, int flat_bytes, double max_dn, const double* flat_std,
                      int height, int width, int channels, int r0, int r1, int c0, int c1,
                      double* out_means, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace cl;
    CL_REQUIRE(flat && flat_std && out_means);
    CL_REQUIRE(flat_bytes == 1 || flat_bytes == 2 || flat_bytes == 8);
    CL_REQUIRE(height > 0 && width > 0 && channels >= 1 && channels <= CL_MAX_CHANNELS);
    if (!workspace || workspace_bytes < cl_flat_roi_means_workspace_bytes(height, width, channels))
        return CL_ERR_WORKSPACE;
    // NumPy slice clamping (negative bounds are not produced by the reference formula)
    CL_REQUIRE(r0 >= 0 && c0 >= 0);
    if (r1 > height) r1 = height;
    if (c1 > width) c1 = width;
    const int rh = r1 > r0 ? r1 - r0 : 0, rw = c1 > c0 ? c1 - c0 : 0;
    cudaStream_t s = (cudaStream_t)stream;
    double* partial = reinterpret_cast<double*>(workspace);
    // an empty ROI yields 0/0 = NaN, like np.mean of an empty slice
    auto partial_kernel = channels == 3 ? roi_partial_kernel<3> : channels == 1 ? roi_partial_kernel<1> : roi_partial_kernel<0>;
    unsigned int* ticket = reinterpret_cast<unsigned int*>(partial + (size_t)kRoiBlocks * 2 * channels);
    cudaError_t e = cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s);
    if (e != cudaSuccess) return cuda_status(e);
    partial_kernel<<<kRoiBlocks, kRoiThreads, 0, s>>>(flat, flat_bytes, max_dn, flat_std, width, channels, r0, c0,
                                                     rw > 0 ? rh : 0, rw > 0 ? rw : 1, partial, ticket,
                                                     (double)rh * (double)rw, out_means);
    return launched();
}

int cl_gaussian_weight(const double* val, double* w, double* dw, int64_t n, void* stream) {
    using namespace cl;
    CL_REQUIRE(n >= 0);
    if (n == 0) return CL_OK;
    CL_REQUIRE(val && w);
    gaussian_weight_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(val, w, dw, n);
    return launched();
}

int cl_bad_pixel_filter(const double* val, const double* std, const double* dark_val,
                        double threshold, int kernel, int height, int width, int channels,
                        double* out_val, double* out_std, void* stream) {
    using namespace cl;
    CL_REQUIRE(height >= 0 && width >= 0 && channels >= 1);
    CL_REQUIRE(kernel >= 1 && kernel <= CL_MAX_MEDIAN_KERNEL);
    const int64_t n = (int64_t)height * width * channels;
    if (n == 0) return CL_OK;
    CL_REQUIRE(val && dark_val && out_val && (!std || out_std));
    bad_pixel_filter_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
        val, std, dark_val, threshold, kernel, height, width, channels, out_val, out_std);
    return launched();
}

int cl_flat_field_normalize(const double* val, const double* std, const double* flat_val,
                            const double* flat_std, const double* flat_means, int64_t n, int channels,
                            double* out_val, double* out_std, void* stream) {
    using namespace cl;
    CL_REQUIRE(n >= 0 && channels >= 1 && channels <= CL_MAX_CHANNELS);
    if (n == 0) return CL_OK;
    CL_REQUIRE(val && std && flat_val && flat_std && flat_means && out_val && out_std);
    flat_normalize_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
        val, std, flat_val, flat_std, flat_means, n, channels, out_val, out_std);
    return launched();
}

}  // extern "C"
