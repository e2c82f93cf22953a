// K2 fast path for 8-bit stacks WITHOUT uncertainty images ("algo 2", STD-table variant): the uncertainty of
// every sample is the camera's STD table value STD[dn][c] (image_set.py:228-243, 365-385 -- what the reference
// does whenever no "... STD.tif" exists).  Same bulk-copy staging of the DN bytes as hdr_merge_staged.cu, but no
// float64 stream at all: only N + [dark] + [flat: 9] + 16 bytes per sample cross HBM (and PCIe, in the end-to-end
// path), so this variant is bound by the SM (shared-memory gathers + FP64), not by HBM.
//
// With sigma a function of (dn, c), most of one exposure's contribution is too.  Two lane-replicated shared-memory
// tables per channel hold, per DN,
//     Ta = { w,        Y0 = dICRF * sigma }                   (pass A reads w only)
//     Tb = { P1 = w*g, X  = fma(w * dICRF, sigma, kappa*P1) } (dw*g + w*dg of exposure_series.py:389)
// computed with the very operations merge_accumulate() performs, so the result is BIT-IDENTICAL to the generic
// kernel; per sample-exposure the loop is left with two conflict-free LDS.128 gathers and 8 FP64 instructions.
//
// Bad pixels: the median warp repairs the DN in the staged A buffer as in hdr_merge_staged.cu.  The repaired
// uncertainty is the MEDIAN of the neighbours' table values (the reference filters the uncertainty image it
// built from the unfiltered DNs), which equals STD[median DN] whenever the table is monotone over the
// neighbourhood's DNs -- always, for a physical noise model.  The median warp checks that equality bit for bit
// and files the rare sample where it fails in the fix-up list, which merge_fixup_kernel recomputes in full.
#include "staged_common.cuh"

namespace cl {
namespace {

using namespace staged;

constexpr int kTilePx = kStagedTilePx;
constexpr int kC = 3;
constexpr int kConsumerWarps = kTilePx / 32;
constexpr int kThreads = kTilePx + 64;          // + A-buffer producer and median warps
constexpr int kDnChunk = kTilePx * kC;          // bytes of one exposure's DN tile
constexpr int kCopies = 8;                      // double2 entries: quarter-warp lanes hit 8 distinct bank quads
constexpr size_t kSmemLimit = 227 * 1024;

struct LutLayout {
    uint32_t off_ta, off_tb, off_abuf_dn, off_bucket, off_bars, total;
};

template <int NMAX, bool MONO>
__global__ void __launch_bounds__(kThreads, 1)
merge_staged_lut_kernel(const __grid_constant__ MergeParams p, const LutLayout L, const int n_tiles) {
    constexpr int kCt = MONO ? 1 : kC;           // true channel count
    extern __shared__ __align__(128) unsigned char smem[];
    double2* ta = reinterpret_cast<double2*>(smem + L.off_ta);
    double2* tb = reinterpret_cast<double2*>(smem + L.off_tb);
    uint8_t* abuf_dn = smem + L.off_abuf_dn;
    uint32_t* bucket_s = reinterpret_cast<uint32_t*>(smem + L.off_bucket);
    uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + L.off_bars);
    uint64_t* a_empty = a_full + 1;
    uint64_t* a_ready = a_full + 2;
    const bool patched = p.any_dark != 0;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const bool has_flat = p.flat_bytes != 0;
    const bool flat_u8 = p.flat_bytes == 1;     // flat DN bytes ride in the A buffer (slot n)

    if (tid == 0) {
        mbar_init(a_full, 1);
        mbar_init(a_empty, kConsumerWarps);
        mbar_init(a_ready, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (warp < kConsumerWarps) {
        for (int it = tid; it < 256 * kC; it += kTilePx) {
            const int d = it & 255, c = it >> 8;
            const int cs = MONO ? 0 : c;                     // mono: the single LUT column in every slot
            double w, dw;
            gaussian_weight(__ddiv_rn((double)d, p.max_dn), w, dw);
            const double p1 = w * p.lut[d * kCt + cs];
            const double dgl = p.dlut[d * kCt + cs];
            const double sigma = p.std_lut[d * kCt + cs];
            // the exposure-independent part of merge_accumulate(), same operations in the same order
            const double a = kappa_of((uint32_t)d, p.kappa_scale) * p1;
            const double b = w * dgl;
            const double2 ea = make_double2(w, dgl * sigma);
            const double2 eb = make_double2(p1, fma(b, sigma, a));
#pragma unroll
            for (int r = 0; r < kCopies; ++r) {
                ta[(c * 256 + d) * kCopies + r] = ea;
                tb[(c * 256 + d) * kCopies + r] = eb;
            }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kTilePx) : "memory");    // consumers only
    }

    if (warp == kConsumerWarps) {
        // ===== A-buffer producer: DN bytes of every exposure of one tile (+ flat DN bytes, + bucket) =====
        if (lane == 0) {
            uint32_t ti = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                const size_t off = (size_t)tile * kDnChunk;
                mbar_wait(a_empty, (ti & 1) ^ 1);
                mbar_expect_tx(a_full, (uint32_t)(p.n + (flat_u8 ? 1 : 0)) * kDnChunk +
                                           (patched ? kBucketWords * 4u : 0u));
                if (patched) {
                    bulk_g2s(smem + L.off_bucket, p.bucket_counts + (size_t)tile * 4, 16, a_full);
                    bulk_g2s(smem + L.off_bucket + 16, p.bucket_entries + (size_t)tile * kBucketCap * 4,
                             kBucketCap * 16, a_full);
                }
                for (int k = 0; k < p.n; ++k)
                    bulk_g2s(abuf_dn + k * kDnChunk, reinterpret_cast<const uint8_t*>(p.dn[k]) + off,
                             kDnChunk, a_full);
                if (flat_u8)
                    bulk_g2s(abuf_dn + p.n * kDnChunk, reinterpret_cast<const uint8_t*>(p.flat) + off,
                             kDnChunk, a_full);
            }
        }
    } else if (warp == kConsumerWarps + 1) {
        // ===== median warp: repairs the bad pixels of the NEXT tile while the consumers work =====
        if (patched) {
            uint32_t ti = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                mbar_wait(a_full, ti & 1);
                const uint32_t n_patch = min(bucket_s[0], (uint32_t)kBucketCap);
                if ((uint32_t)lane < n_patch) {
                    const uint32_t meta = bucket_s[4 + 4 * lane];
                    const int pix = (int)(meta & 511u), c = (int)((meta >> 9) & 3u), ke = (int)((meta >> 11) & 31u);
                    const uint32_t tpx = (uint32_t)tile * kTilePx + (uint32_t)pix;
                    const uint32_t px = MONO ? tpx * kC + (uint32_t)c : tpx;
                    const int ct = MONO ? 0 : c;
                    const int y = (int)(px / (uint32_t)p.W), x = (int)(px - (uint32_t)y * (uint32_t)p.W);
                    uint32_t d_new;
                    double s_new;
                    median_pair(reinterpret_cast<const uint8_t*>(p.dn[ke]), (const double*)nullptr, p.std_lut, y, x, ct,
                                p.H, p.W, kCt, p.K, d_new, s_new);
                    abuf_dn[ke * kDnChunk + pix * kC + c] = (uint8_t)d_new;
                    // the consumers will use STD[d_new]; the reference uses the median of the neighbours' STD values
                    const double s_tab = p.std_lut[(int)d_new * kCt + ct];
                    if (__double_as_longlong(s_tab) != __double_as_longlong(s_new)) {
                        const uint32_t g = atomicAdd(&p.hot_list[0], 1u);
                        if (g < p.hot_cap) p.hot_list[kHotListHeader + g] = tpx * kC + (uint32_t)c;
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic writes vs the next bulk refill
                __syncwarp();
                if (lane == 0) mbar_arrive(a_ready);
            }
        }
    } else {
        // ===== consumers: thread tid owns pixel tid of each tile =====
        uint64_t* const c_afull = patched ? a_ready : a_full;
        const double2* myA = ta + (lane & (kCopies - 1));
        const double2* myB = tb + (lane & (kCopies - 1));
        const int a_word = (tid * kC) >> 2;
        const uint32_t a_shift = ((tid * kC) & 3) * 8;
        uint32_t ti = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
            const int64_t i0 = ((int64_t)tile * kTilePx + tid) * kC;
            // the flat field's uncertainty (the only float64 input) straight from global memory, in flight under pass A
            double f0 = 0.0, f1 = 0.0, f2 = 0.0;
            if (has_flat) {
                f0 = __ldcs(p.flat_std + i0 + 0);
                f1 = __ldcs(p.flat_std + i0 + 1);
                f2 = __ldcs(p.flat_std + i0 + 2);
            }
            // ---- pass A: sum of weights; pack the DNs of every exposure into registers ----
            mbar_wait(c_afull, ti & 1);
            uint32_t pk[NMAX];
            double S0 = 0.0, S1 = 0.0, S2 = 0.0;
#pragma unroll
            for (int k = 0; k < NMAX; ++k) {
                if (k < p.n) {
                    const uint32_t* aw = reinterpret_cast<const uint32_t*>(abuf_dn + k * kDnChunk) + a_word;
                    const uint32_t q = __funnelshift_r(aw[0], aw[1], a_shift) & 0xFFFFFFu;
                    const uint32_t d0 = q & 0xFF, d1 = (q >> 8) & 0xFF, d2 = q >> 16;
                    S0 += myA[(0 * 256 + d0) * kCopies].x;
                    S1 += myA[(1 * 256 + d1) * kCopies].x;
                    S2 += myA[(2 * 256 + d2) * kCopies].x;
                    pk[k] = q;
                }
            }
            uint32_t pkf = 0;
            if (flat_u8) {
                const uint32_t* aw = reinterpret_cast<const uint32_t*>(abuf_dn + p.n * kDnChunk) + a_word;
                pkf = __funnelshift_r(aw[0], aw[1], a_shift) & 0xFFFFFFu;
            }
            __syncwarp();
            if (lane == 0 && consumed(S0, S1, S2 + (double)pkf)) mbar_arrive(a_empty);
            const double r0 = 1.0 / S0, r1 = 1.0 / S1, r2 = 1.0 / S2;

            // ---- pass B: registers and tables only ----
            double av0 = 0.0, av1 = 0.0, av2 = 0.0, as0 = 0.0, as1 = 0.0, as2 = 0.0;
#pragma unroll
            for (int k = 0; k < NMAX; ++k) {
                if (k < p.n) {
                    const uint32_t q = pk[k];
                    const uint32_t d0 = q & 0xFF, d1 = (q >> 8) & 0xFF, d2 = q >> 16;
                    const double rt = p.inv_t[k];
                    const double2 a0 = myA[(0 * 256 + d0) * kCopies], b0 = myB[(0 * 256 + d0) * kCopies];
                    const double2 a1 = myA[(1 * 256 + d1) * kCopies], b1 = myB[(1 * 256 + d1) * kCopies];
                    const double2 a2 = myA[(2 * 256 + d2) * kCopies], b2 = myB[(2 * 256 + d2) * kCopies];
                    merge_accumulate_lut(a0.x, b0.x, b0.y, a0.y, kappa_of(d0, p.kappa_scale), r0, rt, av0, as0);
                    merge_accumulate_lut(a1.x, b1.x, b1.y, a1.y, kappa_of(d1, p.kappa_scale), r1, rt, av1, as1);
                    merge_accumulate_lut(a2.x, b2.x, b2.y, a2.y, kappa_of(d2, p.kappa_scale), r2, rt, av2, as2);
                }
            }

            double v0 = av0 * r0, v1 = av1 * r1, v2 = av2 * r2;
            double u0, u1, u2;
            if (has_flat) {
                double rf0, rf1, rf2;
                if (flat_u8) {
                    rf0 = kRecip255.v[pkf & 0xFF];
                    rf1 = kRecip255.v[(pkf >> 8) & 0xFF];
                    rf2 = kRecip255.v[pkf >> 16];
                } else {
                    rf0 = flat_recip(p.flat, p.flat_bytes, i0 + 0, p.max_dn);
                    rf1 = flat_recip(p.flat, p.flat_bytes, i0 + 1, p.max_dn);
                    rf2 = flat_recip(p.flat, p.flat_bytes, i0 + 2, p.max_dn);
                }
                constexpr int c1 = MONO ? 0 : 1, c2 = MONO ? 0 : 2;
                flat_apply(v0, u0, (as0 * r0) * r0, rf0, f0, p.flat_means[0], p.flat_means[kCt + 0]);
                flat_apply(v1, u1, (as1 * r1) * r1, rf1, f1, p.flat_means[c1], p.flat_means[kCt + c1]);
                flat_apply(v2, u2, (as2 * r2) * r2, rf2, f2, p.flat_means[c2], p.flat_means[kCt + c2]);
            } else {
                u0 = sqrt(as0) * r0; u1 = sqrt(as1) * r1; u2 = sqrt(as2) * r2;
            }
            __stcs(p.out_val + i0 + 0, v0); __stcs(p.out_val + i0 + 1, v1); __stcs(p.out_val + i0 + 2, v2);
            __stcs(p.out_std + i0 + 0, u0); __stcs(p.out_std + i0 + 1, u1); __stcs(p.out_std + i0 + 2, u2);
        }
    }
}

bool make_lut_layout(const MergeParams& p, LutLayout& L) {
    uint32_t off = 0;
    L.off_ta = off; off += kC * 256 * kCopies * 16;
    L.off_tb = off; off += kC * 256 * kCopies * 16;
    L.off_abuf_dn = off; off += (uint32_t)(p.n + (p.flat_bytes == 1 ? 1 : 0)) * kDnChunk;
    L.off_bucket = off; off += kBucketWords * 4;      // (also the landing zone of the last pixel's second DN word)
    off = (off + 127) & ~127u;
    L.off_bars = off; off += 128;
    L.total = off;
    return off <= kSmemLimit;
}

}  // namespace

int try_merge_staged_lut(const MergeParams& p, cudaStream_t stream) {
    LutLayout L;
    if (!tile_stack(p, false) || !make_lut_layout(p, L)) return CL_ERR_UNSUPPORTED;
    const bool mono = p.C == 1;
    auto kernel = p.n <= 8 ? (mono ? merge_staged_lut_kernel<8, true> : merge_staged_lut_kernel<8, false>)
                           : (mono ? merge_staged_lut_kernel<16, true> : merge_staged_lut_kernel<16, false>);
    return launch_tile_kernel(p, kernel, kThreads, L, stream);
}

}  // namespace cl
