// K2 single-pass path ("algo 4"): 8-bit RGB / mono stacks with float64 uncertainty images, N >= 2 exposures.
//
// The staged kernel (hdr_merge_staged.cu) is bound by its shared-memory traffic, not by HBM (ncu: LSU shared pipe
// 56-59 %, issue 60 %, HBM 73 %): per warp and exposure it makes 32 shared-memory wavefronts, 8 of them in "pass A",
// which only exists because the reference's variance term needs 1/S = 1/sum(w) INSIDE the square:
//     var = sum_k ((x_k - e_k / S) y_k)^2 ,   x = dw g + w dg,  e = dw w g,  y = dg / t        (exposure_series.py:389)
// Expanding the square makes the sum of weights a post-factor:
//     var = A - 2 B / S + C / S^2 ,   A = sum (x y)^2,  B = sum (x y)(e y),  C = sum (e y)^2 .
// The expansion cancels when one exposure dominates the weight -- but the Gaussian weight never drops below
// w(0) = w(1) = e^-7.5 = 5.5e-4, so with N >= 2 exposures 1 - w_k / S >= 5.5e-4 and the cancellation costs at most
// ~7 decimal digits of the 16: <= 1e-9 relative on the uncertainty in the most adversarial stack (one mid-grey
// exposure, all others black or saturated; measured 3e-11 for N = 2, 3e-13 for N = 16) and ~1e-15 on ordinary data,
// against the 1e-6 the north star allows.  That bound covers the STRUCTURAL cancellation only: where the two parts of
// x - e/S = dw g (1 - w/S) + w dg also cancel each other by accident, the uncertainty itself is anomalously small and
// the expansion's absolute error (~1e-16 A) is large relative to it (1e-3 seen on 0.3 % of the samples of an
// adversarial stack).  The kernel therefore checks q < 1e-6 A per sample and hands those samples to the exact
// two-pass formula through the fix-up work list (merge_fixup_kernel; none on ordinary stacks): every sample is
// within 1.1e-10 of the two-pass kernels (tests assert 1e-9), and the rule is deterministic -- the fix-up pass
// applies the same expansion + check, so a sample gets the same bits whichever kernel computes it.  N = 1 has no
// weight floor and stays on the two-pass kernels.
//
// With S out of the loop there is ONE pass: no A buffer, no packed-DN registers, no pass-A gathers.  A ring stage
// carries everything exposure k of a tile needs -- its 12 KB of uncertainties and its 1.5 KB of DN bytes, two bulk
// copies on one mbarrier -- so the ring is 7 stages deep (the staged kernel: 6 + the A buffer) and a tile needs no
// other hand-off.  16 consumer warps (thread t = pixel t of the 512-pixel tile), one producer warp, a median warp
// (bad pixels: the K x K medians of a tile's bucket from global memory, one or two tiles ahead) and a patcher warp
// (writes the repaired DN byte and sigma over each stage as it lands and only then declares it ready): 608 threads,
// 24 shared-memory wavefronts per warp and exposure instead of 32.
//
// What bounds it (tools/microbench/read_bw.cu: the same ring with the arithmetic removed streams 7.3 TB/s pure read and
// 6.6 TB/s with this kernel's 24 KB of output per 17 stages at 7 stages x 13.8 KB -- the copy figure in
// MEASURED_PEAKS.json, 6.56 TB/s, is not the ceiling of a read-dominated stream): the CONSUMERS.  Capping the ring
// (4 / 5 / 6 / 7 stages: 0.805 / 0.749 / 0.726 / 0.725 ms without corrections) shows the copy side saturating while
// every instruction taken out of the consumer loop still pays:
//   * kappa(dn) rides in the weight table ({w, kappa} as a double2, 8 copies, the same 32 KB) instead of being rebuilt
//     from the DN with an int->double conversion and an FMA per sample-exposure:   0.719 -> 0.685 ms (cfg2, no
//     corrections), 0.834 -> 0.812 with dark frames + flat;
//   * x = fma(w, dg, a) with dg = dICRF sigma shared with y = dg / t (12 instead of 13 FP64 operations): 0.685 -> 0.670 ms
//     = 5.9 TB/s, 91 % of the copy peak.
// Per pixel-exposure the loop is now ~37 FP64 + ~36 other + ~18 ring-bookkeeping instructions.  With corrections
// (0.807 ms) the extras are: dark scan 0.039, the flat stage 0.073 (0.034 of traffic + a second epilogue's worth of
// FP64: ~28 operations and a square root per sample), repairs 0.024 (~11 medians per tile in the bench stack).
#include "staged_common.cuh"

namespace cl {
namespace {

using namespace staged;

constexpr int kTilePx = kStagedTilePx;
constexpr int kC = 3;
constexpr int kConsumerWarps = kTilePx / 32;
constexpr int kThreads = kTilePx + 96;          // + producer, median and patcher warps
constexpr int kDnChunk = kTilePx * kC;          // 1536 B
constexpr int kStdChunk = kTilePx * kC * 8;     // 12288 B
constexpr int kStage = kStdChunk + kDnChunk;    // 13824 B = 108 x 128
constexpr int kLutACopies = 8;
constexpr int kLutBCopies = 8;
constexpr int kMaxStages = 8;
constexpr size_t kSmemLimit = 227 * 1024;

struct StreamLayout {
    int stages;
    uint32_t off_lutA, off_lutB, off_ring, off_bars, off_med, total;
};

// one repaired bad pixel, handed from the median warp to the patcher warp through shared memory
struct MedEntry {
    uint32_t pos;        // sample within the tile (pixel * 3 + channel); 0xFFFFFFFF: no entry
    uint32_t ke_dn;      // exposure << 8 | repaired DN
    double sigma;        // repaired uncertainty
};

// warp-aggregated append to the work list (all 32 lanes of a consumer warp call this together)
__device__ __forceinline__ void flag_cancelled(const MergeParams& p, bool flag, uint32_t sample, int lane) {
    const uint32_t m = __ballot_sync(0xffffffffu, flag);
    if (m == 0u) return;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(&p.hot_list[0], (uint32_t)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (flag) {
        const uint32_t slot = base + (uint32_t)__popc(m & ((1u << lane) - 1u));
        if (slot < p.hot_cap) p.hot_list[kHotListHeader + slot] = sample;
    }
}

template <bool MONO>
__global__ void __launch_bounds__(kThreads, 1)
merge_stream_kernel(const __grid_constant__ MergeParams p, const StreamLayout L, const int n_tiles) {
    constexpr int kCt = MONO ? 1 : kC;           // true channel count
    extern __shared__ __align__(128) unsigned char smem[];
    double2* lutA = reinterpret_cast<double2*>(smem + L.off_lutA);       // [dn][copy] {w, kappa}
    double2* lutB = reinterpret_cast<double2*>(smem + L.off_lutB);
    unsigned char* ring = smem + L.off_ring;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.off_bars);
    uint64_t* full = bars;                    // [stages]  producer -> patch warp / consumers (tx bytes)
    uint64_t* empty = bars + kMaxStages;      // [stages]  consumers -> producer
    uint64_t* ready = bars + 2 * kMaxStages;  // [stages]  patcher -> consumers
    uint64_t* med_full = bars + 3 * kMaxStages;       // [2]  median warp -> patcher (tile parity)
    uint64_t* med_free = med_full + 2;                // [2]  patcher -> median warp
    MedEntry* med = reinterpret_cast<MedEntry*>(smem + L.off_med);   // [2][kBucketCap]
    const bool patched = p.any_dark != 0;
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int stages = L.stages;
    const bool has_flat = p.flat_bytes != 0;
    const bool flat_u8 = p.flat_bytes == 1;
    const int chunks = p.n + (has_flat ? 1 : 0);            // stages per tile

    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumerWarps);
            mbar_init(&ready[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&med_full[b], 1);
            mbar_init(&med_free[b], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();          // the producer starts streaming right away, under the table construction below
    if (warp < kConsumerWarps) {
        for (int it = tid; it < 256 * 4; it += kTilePx) {
            const int d = it >> 2, part = it & 3;            // part 0: w[d]; parts 1..3: channel part-1
            double w, dw;
            gaussian_weight(__ddiv_rn((double)d, p.max_dn), w, dw);
            if (part == 0) {
                const double2 e = make_double2(w, kappa_of((uint32_t)d, p.kappa_scale));
#pragma unroll
                for (int r = 0; r < kLutACopies; ++r) lutA[d * kLutACopies + r] = e;
            } else {
                const int c = part - 1;
                const int cs = MONO ? 0 : c;
                const double2 e = make_double2(w * p.lut[d * kCt + cs], p.dlut[d * kCt + cs]);
#pragma unroll
                for (int r = 0; r < kLutBCopies; ++r) lutB[(c * 256 + d) * kLutBCopies + r] = e;
            }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kTilePx) : "memory");    // consumers only
    }

    if (warp == kConsumerWarps) {
        // ===== producer: one stage per (tile, exposure): sigma chunk + DN chunk; the flat field last =====
        if (lane == 0) {
            int s = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const size_t off = (size_t)tile * kTilePx * kC;   // first sample of the tile
                for (int k = 0; k < chunks; ++k) {
                    const bool is_flat = k == p.n;
                    const bool with_dn = !is_flat || flat_u8;
                    mbar_wait(&empty[s], phase ^ 1);
                    mbar_expect_tx(&full[s], with_dn ? kStage : kStdChunk);
                    unsigned char* dst = ring + (size_t)s * kStage;
                    bulk_g2s(dst, (is_flat ? p.flat_std : p.std[k]) + off, kStdChunk, &full[s]);
                    if (with_dn)
                        bulk_g2s(dst + kStdChunk,
                                 reinterpret_cast<const uint8_t*>(is_flat ? p.flat : p.dn[k]) + off, kDnChunk, &full[s]);
                    if (++s == stages) { s = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kConsumerWarps + 1) {
        // ===== median warp: repairs of the bad pixels of a tile, one or two tiles ahead of the patcher =====
        // lane e owns bucket entry e {pixel, channel, exposure} (filed by dark_scan_kernel); the K x K neighbourhoods
        // come from global memory (~2 us of latency per tile, which must not sit between a stage landing and the
        // consumers seeing it: hence a warp of its own and a double-buffered hand-off).
        if (patched) {
            uint32_t ti = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                const int buf = (int)(ti & 1);
                mbar_wait(&med_free[buf], ((ti >> 1) & 1) ^ 1);
                const uint32_t n_patch = min(__ldcg(p.bucket_counts + (size_t)tile * 4), (uint32_t)kBucketCap);
                MedEntry out;
                out.pos = 0xFFFFFFFFu;
                out.ke_dn = 0u;
                out.sigma = 0.0;
                if ((uint32_t)lane < n_patch) {
                    const uint32_t meta = __ldcg(p.bucket_entries + ((size_t)tile * kBucketCap + lane) * 4);
                    const int pix = (int)(meta & 511u), c = (int)((meta >> 9) & 3u), ke = (int)((meta >> 11) & 31u);
                    const uint32_t tpx = (uint32_t)tile * kTilePx + (uint32_t)pix;
                    const uint32_t px = MONO ? tpx * kC + (uint32_t)c : tpx;
                    const int ct = MONO ? 0 : c;
                    const int y = (int)(px / (uint32_t)p.W), x = (int)(px - (uint32_t)y * (uint32_t)p.W);
                    uint32_t d_new;
                    double s_new;
                    median_pair(reinterpret_cast<const uint8_t*>(p.dn[ke]), p.std[ke], p.std_lut, y, x, ct, p.H, p.W, kCt,
                                p.K, d_new, s_new);
                    out.pos = (uint32_t)(pix * kC + c);
                    out.ke_dn = ((uint32_t)ke << 8) | d_new;
                    out.sigma = s_new;
                }
                med[buf * kBucketCap + lane] = out;
                __syncwarp();
                if (lane == 0) mbar_arrive(&med_full[buf]);
            }
        }
    } else if (warp == kConsumerWarps + 2) {
        // ===== patcher: writes the repaired DN byte and sigma over stage (tile, k) right after it lands =====
        if (patched) {
            int s = 0;
            uint32_t phase = 0, ti = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                const int buf = (int)(ti & 1);
                mbar_wait(&med_full[buf], (ti >> 1) & 1);
                const MedEntry mine = med[buf * kBucketCap + lane];
                __syncwarp();
                if (lane == 0 && consumed(mine.sigma * mine.sigma, (double)mine.pos, 0.0)) mbar_arrive(&med_free[buf]);
                const bool have = mine.pos != 0xFFFFFFFFu;
                const int ke = (int)(mine.ke_dn >> 8);
                for (int k = 0; k < chunks; ++k) {
                    mbar_wait(&full[s], phase);
                    const bool hit = have && ke == k;
                    if (hit) {
                        unsigned char* st = ring + (size_t)s * kStage;
                        reinterpret_cast<double*>(st)[mine.pos] = mine.sigma;
                        st[kStdChunk + mine.pos] = (uint8_t)(mine.ke_dn & 0xFFu);
                    }
                    if (__any_sync(0xffffffffu, hit))
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // before the TMA refill
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&ready[s]);
                    if (++s == stages) { s = 0; phase ^= 1; }
                }
            }
        }
    } else {
        // ===== consumers: thread tid owns pixel tid of each tile; ONE pass over the tile's stages =====
        uint64_t* const c_full = patched ? ready : full;
        const double2* myA = lutA + (lane & (kLutACopies - 1));
        const double2* myB = lutB + (lane & (kLutBCopies - 1));
        // bytes tid*3 .. tid*3+2 of a DN chunk live in words a_word, a_word+1 (the second word of the last pixel lies
        // just past the chunk: inside the next stage or the barrier block, and contributes only the masked-off top byte)
        const int a_word = (tid * kC) >> 2;
        const uint32_t a_shift = ((tid * kC) & 3) * 8;
        uint32_t phase = 0;
        int s = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int64_t i0 = ((int64_t)tile * kTilePx + tid) * kC;
            double S0 = 0.0, S1 = 0.0, S2 = 0.0;
            double av0 = 0.0, av1 = 0.0, av2 = 0.0;
            double A0 = 0.0, A1 = 0.0, A2 = 0.0, B0 = 0.0, B1 = 0.0, B2 = 0.0, C0 = 0.0, C1 = 0.0, C2 = 0.0;
#pragma unroll 2
            for (int k = 0; k < p.n; ++k) {
                mbar_wait(&c_full[s], phase);
                const unsigned char* st = ring + (size_t)s * kStage;
                const double* sp = reinterpret_cast<const double*>(st) + tid * kC;
                const uint32_t* aw = reinterpret_cast<const uint32_t*>(st + kStdChunk) + a_word;
                const double g0 = sp[0], g1 = sp[1], g2 = sp[2];
                const uint32_t q = __funnelshift_r(aw[0], aw[1], a_shift) & 0xFFFFFFu;
                const uint32_t d0 = q & 0xFF, d1 = (q >> 8) & 0xFF, d2 = q >> 16;
                const double rt = p.inv_t[k];
                const double2 w0 = myA[d0 * kLutACopies], w1 = myA[d1 * kLutACopies], w2 = myA[d2 * kLutACopies];
                const double2 e0 = myB[(0 * 256 + d0) * kLutBCopies];
                const double2 e1 = myB[(1 * 256 + d1) * kLutBCopies];
                const double2 e2 = myB[(2 * 256 + d2) * kLutBCopies];
                merge_accumulate_expanded(w0.x, e0.x, e0.y, w0.y, g0, rt, S0, av0, A0, B0, C0);
                merge_accumulate_expanded(w1.x, e1.x, e1.y, w1.y, g1, rt, S1, av1, A1, B1, C1);
                merge_accumulate_expanded(w2.x, e2.x, e2.y, w2.y, g2, rt, S2, av2, A2, B2, C2);
                __syncwarp();
                if (lane == 0 && consumed_nonneg(A0, A1, A2)) mbar_arrive(&empty[s]);
                if (++s == stages) { s = 0; phase ^= 1; }
            }
            // 1 / S and the square roots below are the library's main paths (common.cuh): correctly rounded like the
            // calls they replace, without the six range tests + slow-path branches per pixel that fenced the
            // epilogue's schedule.  A sample that is off a main path joins the cancelled ones on the work list
            // (merge_fixup_kernel recomputes it with the library calls).
            bool k0, k1, k2;
            const double r0 = rcp_main_path(S0, k0), r1 = rcp_main_path(S1, k1), r2 = rcp_main_path(S2, k2);
            double v0 = av0 * r0, v1 = av1 * r1, v2 = av2 * r2;
            const double q0 = expanded_variance(A0, B0, C0, r0), q1 = expanded_variance(A1, B1, C1, r1),
                         q2 = expanded_variance(A2, B2, C2, r2);
            bool f0 = q0 < kStreamCancel * A0 || !k0, f1 = q1 < kStreamCancel * A1 || !k1,
                 f2 = q2 < kStreamCancel * A2 || !k2;
            double u0, u1, u2;
            if (has_flat) {
                mbar_wait(&c_full[s], phase);
                const unsigned char* st = ring + (size_t)s * kStage;
                const double* sp = reinterpret_cast<const double*>(st) + tid * kC;
                const double fs0 = sp[0], fs1 = sp[1], fs2 = sp[2];
                double rf0, rf1, rf2;
                if (flat_u8) {
                    const uint32_t* aw = reinterpret_cast<const uint32_t*>(st + kStdChunk) + a_word;
                    const uint32_t pkf = __funnelshift_r(aw[0], aw[1], a_shift) & 0xFFFFFFu;
                    rf0 = kRecip255.v[pkf & 0xFF];
                    rf1 = kRecip255.v[(pkf >> 8) & 0xFF];
                    rf2 = kRecip255.v[pkf >> 16];
                } else {
                    rf0 = flat_recip(p.flat, p.flat_bytes, i0 + 0, p.max_dn);
                    rf1 = flat_recip(p.flat, p.flat_bytes, i0 + 1, p.max_dn);
                    rf2 = flat_recip(p.flat, p.flat_bytes, i0 + 2, p.max_dn);
                }
                constexpr int c1 = MONO ? 0 : 1, c2 = MONO ? 0 : 2;
                f0 |= !flat_apply_main_path(v0, u0, (q0 * r0) * r0, rf0, fs0, p.flat_means[0], p.flat_means[kCt + 0]);
                f1 |= !flat_apply_main_path(v1, u1, (q1 * r1) * r1, rf1, fs1, p.flat_means[c1], p.flat_means[kCt + c1]);
                f2 |= !flat_apply_main_path(v2, u2, (q2 * r2) * r2, rf2, fs2, p.flat_means[c2], p.flat_means[kCt + c2]);
                __syncwarp();
                if (lane == 0 && consumed(u0, u1, u2 + rf0)) mbar_arrive(&empty[s]);     // (rf: the staged flat bytes)
                if (++s == stages) { s = 0; phase ^= 1; }
            } else {
                bool s0, s1, s2;
                const double t0 = sqrt_main_path(q0, s0), t1 = sqrt_main_path(q1, s1), t2 = sqrt_main_path(q2, s2);
                u0 = (s0 ? t0 : 0.0) * r0; u1 = (s1 ? t1 : 0.0) * r1; u2 = (s2 ? t2 : 0.0) * r2;
                f0 |= !(s0 || q0 == 0.0); f1 |= !(s1 || q1 == 0.0); f2 |= !(s2 || q2 == 0.0);
            }
            // samples whose expansion cancelled (or that left a main path) go to the exact formula (work list ->
            // merge_fixup_kernel); one atomic per warp and channel that has any
            if (__any_sync(0xffffffffu, f0 | f1 | f2)) {
                flag_cancelled(p, f0, (uint32_t)i0 + 0u, lane);
                flag_cancelled(p, f1, (uint32_t)i0 + 1u, lane);
                flag_cancelled(p, f2, (uint32_t)i0 + 2u, lane);
            }
            __stcs(p.out_val + i0 + 0, v0); __stcs(p.out_val + i0 + 1, v1); __stcs(p.out_val + i0 + 2, v2);
            __stcs(p.out_std + i0 + 0, u0); __stcs(p.out_std + i0 + 1, u1); __stcs(p.out_std + i0 + 2, u2);
        }
    }
}

bool make_stream_layout(StreamLayout& L) {
    uint32_t off = 0;
    L.off_lutA = off; off += 256 * kLutACopies * 16;
    L.off_lutB = off; off += kC * 256 * kLutBCopies * 16;
    L.off_ring = off;
    const size_t room = kSmemLimit - 256 - 2 * kBucketCap * sizeof(MedEntry) - off;
    int stages = (int)(room / kStage);
    if (stages > kMaxStages) stages = kMaxStages;
    L.stages = stages;
    off += (uint32_t)stages * kStage;
    L.off_bars = off; off += 256;          // (also absorbs the last pixel's second DN word of the last stage)
    L.off_med = off; off += 2 * kBucketCap * sizeof(MedEntry);
    L.total = off;
    return stages >= 3;
}

}  // namespace

int try_merge_stream(const MergeParams& p_in, cudaStream_t stream) {
    StreamLayout L;
    if (!tile_stack(p_in, true) || p_in.n < 2 || !make_stream_layout(L)) return CL_ERR_UNSUPPORTED;
    MergeParams p = p_in;
    p.stream_mode = 1;
    return launch_tile_kernel(p, p.C == 1 ? merge_stream_kernel<true> : merge_stream_kernel<false>, kThreads, L,
                              stream);
}

}  // namespace cl
