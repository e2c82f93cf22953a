// K2 single-pass path for 8-bit RGB / mono stacks WITHOUT uncertainty images ("algo 4", STD-table variant): the
// uncertainty of every sample is the camera's STD table value STD[dn][c] (image_set.py:228-243, 365-385 -- what the
// reference does whenever no "... STD.tif" exists), N >= 2 exposures.
//
// The two-pass STD-table kernel (hdr_merge_staged_lut.cu) is bound by the SM: 0.85 ms for cfg2 while only 1.0 GB
// cross HBM.  With the variance in expanded form (hdr_merge_stream.cu: var = A - 2 B rS + C rS^2) AND sigma a function
// of (dn, c), everything an exposure contributes is a table value times a power of 1/t:
//     x y = (x dg) / t,   e y = (e dg) / t,    x = dw g + w dg,  e = dw w g,  dg = dICRF sigma
// so two lane-replicated shared-memory tables per channel,
//     T1 = { w, P1 = w g }          T2 = { x dg, e dg }        (lut_products(), hdr_merge.cuh)
// leave per sample-exposure two conflict-free LDS.128 gathers and 7 FP64 instructions (two multiplies by 1/t, five
// accumulations) -- no pass A, no packed-DN registers, no kappa arithmetic.  The DN bytes stream through a ring of
// 6 KB stages holding four exposures of a tile each (one barrier round trip per four exposures).
//
// Cancellation guard, fix-up rule and determinism are those of hdr_merge_stream.cu: a sample whose expanded variance
// kept less than 1e-6 of its largest term goes to the work list and merge_fixup_kernel recomputes it with the exact
// two-pass formula; the fix-up evaluates this kernel's arithmetic (stream_mode 2) for the bad pixels whose bucket
// overflowed, so a sample gets the same bits whichever kernel computes it.
// Bad pixels: median warp + patcher warp as in hdr_merge_stream.cu (only the DN byte is patched); the repaired
// uncertainty is the MEDIAN of the neighbours' table values, which equals STD[median DN] whenever the table is
// monotone over the neighbourhood -- the median warp checks that equality bit for bit and files the rare sample
// where it fails in the work list.
#include "staged_common.cuh"

namespace cl {
namespace {

using namespace staged;

constexpr int kTilePx = kStagedTilePx;
constexpr int kC = 3;
constexpr int kConsumerWarps = kTilePx / 32;
constexpr int kThreads = kTilePx + 96;          // + producer, median and patcher warps
constexpr int kDnChunk = kTilePx * kC;          // 1536 B: one exposure's DN bytes of a tile
constexpr int kGroup = 4;                       // exposures per ring stage
constexpr int kStage = kGroup * kDnChunk;       // 6144 B
constexpr int kCopies = 8;                      // double2 entries: quarter-warp lanes hit 8 distinct bank quads
constexpr int kMaxStages = 8;
constexpr size_t kSmemLimit = 227 * 1024;

struct SLutLayout {
    int stages;
    uint32_t off_t1, off_t2, off_ring, off_bars, off_med, total;
};

// one repaired bad pixel, handed from the median warp to the patcher warp through shared memory
struct MedEntry {
    uint32_t pos;        // sample within the tile (pixel * 3 + channel); 0xFFFFFFFF: no entry
    uint32_t ke_dn;      // exposure << 8 | repaired DN
};

__device__ __forceinline__ void flag_sample(const MergeParams& p, bool flag, uint32_t sample, int lane) {
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
merge_stream_lut_kernel(const __grid_constant__ MergeParams p, const SLutLayout L, const int n_tiles) {
    constexpr int kCt = MONO ? 1 : kC;           // true channel count
    extern __shared__ __align__(128) unsigned char smem[];
    double2* t1 = reinterpret_cast<double2*>(smem + L.off_t1);       // [c][dn][copy] {w, P1}
    double2* t2 = reinterpret_cast<double2*>(smem + L.off_t2);       // [c][dn][copy] {x dg, e dg}
    unsigned char* ring = smem + L.off_ring;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.off_bars);
    uint64_t* full = bars;                    // [stages]  producer -> patcher / consumers (tx bytes)
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
    const bool flat_u8 = p.flat_bytes == 1;                  // the flat's DN bytes ride the ring as one more stage
    const int n_groups = (p.n + kGroup - 1) / kGroup;
    const int chunks = n_groups + (flat_u8 ? 1 : 0);         // stages per tile

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
        for (int it = tid; it < 256 * kC; it += kTilePx) {
            const int d = it & 255, c = it >> 8;
            const int cs = MONO ? 0 : c;                     // mono: the single LUT column in every slot
            double w, dw;
            gaussian_weight(__ddiv_rn((double)d, p.max_dn), w, dw);
            const double p1 = w * p.lut[d * kCt + cs];
            double xu, eu;
            lut_products(w, p1, p.dlut[d * kCt + cs], kappa_of((uint32_t)d, p.kappa_scale), p.std_lut[d * kCt + cs], xu, eu);
            const double2 e1 = make_double2(w, p1), e2 = make_double2(xu, eu);
#pragma unroll
            for (int r = 0; r < kCopies; ++r) {
                t1[(c * 256 + d) * kCopies + r] = e1;
                t2[(c * 256 + d) * kCopies + r] = e2;
            }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kTilePx) : "memory");    // consumers only
    }

    if (warp == kConsumerWarps) {
        // ===== producer: one stage per (tile, group of kGroup exposures): their DN chunks; the flat's DN bytes last =====
        if (lane == 0) {
            int s = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const size_t off = (size_t)tile * kDnChunk;       // first sample of the tile
                for (int g = 0; g < chunks; ++g) {
                    mbar_wait(&empty[s], phase ^ 1);
                    unsigned char* dst = ring + (size_t)s * kStage;
                    if (g == n_groups) {
                        mbar_expect_tx(&full[s], kDnChunk);
                        bulk_g2s(dst, reinterpret_cast<const uint8_t*>(p.flat) + off, kDnChunk, &full[s]);
                    } else {
                        const int k0 = g * kGroup;
                        const int nk = min(kGroup, p.n - k0);
                        mbar_expect_tx(&full[s], (uint32_t)nk * kDnChunk);
                        for (int j = 0; j < nk; ++j)
                            bulk_g2s(dst + j * kDnChunk, reinterpret_cast<const uint8_t*>(p.dn[k0 + j]) + off, kDnChunk,
                                     &full[s]);
                    }
                    if (++s == stages) { s = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kConsumerWarps + 1) {
        // ===== median warp: repairs of the bad pixels of a tile, one or two tiles ahead of the patcher =====
        if (patched) {
            uint32_t ti = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                const int buf = (int)(ti & 1);
                mbar_wait(&med_free[buf], ((ti >> 1) & 1) ^ 1);
                const uint32_t n_patch = min(__ldcg(p.bucket_counts + (size_t)tile * 4), (uint32_t)kBucketCap);
                MedEntry out;
                out.pos = 0xFFFFFFFFu;
                out.ke_dn = 0u;
                if ((uint32_t)lane < n_patch) {
                    const uint32_t meta = __ldcg(p.bucket_entries + ((size_t)tile * kBucketCap + lane) * 4);
                    const int pix = (int)(meta & 511u), c = (int)((meta >> 9) & 3u), ke = (int)((meta >> 11) & 31u);
                    const uint32_t tpx = (uint32_t)tile * kTilePx + (uint32_t)pix;
                    const uint32_t px = MONO ? tpx * kC + (uint32_t)c : tpx;
                    const int ct = MONO ? 0 : c;
                    const int y = (int)(px / (uint32_t)p.W), x = (int)(px - (uint32_t)y * (uint32_t)p.W);
                    uint32_t d_new;
                    double s_new;
                    median_pair(reinterpret_cast<const uint8_t*>(p.dn[ke]), (const double*)nullptr, p.std_lut, y, x, ct,
                                p.H, p.W, kCt, p.K, d_new, s_new);
                    out.pos = (uint32_t)(pix * kC + c);
                    out.ke_dn = ((uint32_t)ke << 8) | d_new;
                    // the consumers will use STD[d_new]; the reference uses the median of the neighbours' STD values
                    const double s_tab = p.std_lut[(int)d_new * kCt + ct];
                    if (__double_as_longlong(s_tab) != __double_as_longlong(s_new)) {
                        const uint32_t gi = atomicAdd(&p.hot_list[0], 1u);
                        if (gi < p.hot_cap) p.hot_list[kHotListHeader + gi] = tpx * kC + (uint32_t)c;
                    }
                }
                med[buf * kBucketCap + lane] = out;
                __syncwarp();
                if (lane == 0) mbar_arrive(&med_full[buf]);
            }
        }
    } else if (warp == kConsumerWarps + 2) {
        // ===== patcher: writes the repaired DN byte over stage (tile, group) right after it lands =====
        if (patched) {
            int s = 0;
            uint32_t phase = 0, ti = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                const int buf = (int)(ti & 1);
                mbar_wait(&med_full[buf], (ti >> 1) & 1);
                const MedEntry mine = med[buf * kBucketCap + lane];
                __syncwarp();
                if (lane == 0 && mine.pos != 0xFFFFFFFEu) mbar_arrive(&med_free[buf]);      // (always true, from the loaded entry)
                const bool have = mine.pos != 0xFFFFFFFFu;
                const int ke = (int)(mine.ke_dn >> 8);
                for (int g = 0; g < chunks; ++g) {
                    mbar_wait(&full[s], phase);
                    const bool hit = have && g < n_groups && ke / kGroup == g;
                    if (hit) ring[(size_t)s * kStage + (ke % kGroup) * kDnChunk + mine.pos] = (uint8_t)(mine.ke_dn & 0xFFu);
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
        const double2* my1 = t1 + (lane & (kCopies - 1));
        const double2* my2 = t2 + (lane & (kCopies - 1));
        // bytes tid*3 .. tid*3+2 of a DN chunk live in words a_word, a_word+1 (the second word of the last pixel lies
        // just past the chunk: inside the next chunk / stage or the barrier block, and contributes only the masked-off
        // top byte)
        const int a_word = (tid * kC) >> 2;
        const uint32_t a_shift = ((tid * kC) & 3) * 8;
        uint32_t phase = 0;
        int s = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int64_t i0 = ((int64_t)tile * kTilePx + tid) * kC;
            // the flat field's uncertainty (the only float64 input) straight from global memory, in flight under the loop
            double f0 = 0.0, f1 = 0.0, f2 = 0.0;
            if (has_flat) {
                f0 = __ldcs(p.flat_std + i0 + 0);
                f1 = __ldcs(p.flat_std + i0 + 1);
                f2 = __ldcs(p.flat_std + i0 + 2);
            }
            double S0 = 0.0, S1 = 0.0, S2 = 0.0;
            double av0 = 0.0, av1 = 0.0, av2 = 0.0;
            double A0 = 0.0, A1 = 0.0, A2 = 0.0, B0 = 0.0, B1 = 0.0, B2 = 0.0, C0 = 0.0, C1 = 0.0, C2 = 0.0;
            for (int g = 0; g < n_groups; ++g) {
                mbar_wait(&c_full[s], phase);
                const unsigned char* st = ring + (size_t)s * kStage;
                const int k0 = g * kGroup;
#pragma unroll
                for (int j = 0; j < kGroup; ++j) {
                    if (j > 0 && k0 + j >= p.n) break;            // (the last group may be partly filled)
                    const uint32_t* aw = reinterpret_cast<const uint32_t*>(st + j * kDnChunk) + a_word;
                    const uint32_t q = __funnelshift_r(aw[0], aw[1], a_shift) & 0xFFFFFFu;
                    const uint32_t d0 = q & 0xFF, d1 = (q >> 8) & 0xFF, d2 = q >> 16;
                    const double rt = p.inv_t[k0 + j];
                    const double2 a0 = my1[(0 * 256 + d0) * kCopies], b0 = my2[(0 * 256 + d0) * kCopies];
                    const double2 a1 = my1[(1 * 256 + d1) * kCopies], b1 = my2[(1 * 256 + d1) * kCopies];
                    const double2 a2 = my1[(2 * 256 + d2) * kCopies], b2 = my2[(2 * 256 + d2) * kCopies];
                    merge_accumulate_expanded_lut(a0.x, a0.y, b0.x, b0.y, rt, S0, av0, A0, B0, C0);
                    merge_accumulate_expanded_lut(a1.x, a1.y, b1.x, b1.y, rt, S1, av1, A1, B1, C1);
                    merge_accumulate_expanded_lut(a2.x, a2.y, b2.x, b2.y, rt, S2, av2, A2, B2, C2);
                }
                __syncwarp();
                if (lane == 0 && consumed_nonneg(A0, A1, A2)) mbar_arrive(&empty[s]);
                if (++s == stages) { s = 0; phase ^= 1; }
            }
            // 1 / S and the square roots: the library's main paths (see merge_stream_kernel); a sample off them joins
            // the cancelled ones on the work list
            bool k0, k1, k2;
            const double r0 = rcp_main_path(S0, k0), r1 = rcp_main_path(S1, k1), r2 = rcp_main_path(S2, k2);
            double v0 = av0 * r0, v1 = av1 * r1, v2 = av2 * r2;
            const double q0 = expanded_variance(A0, B0, C0, r0), q1 = expanded_variance(A1, B1, C1, r1),
                         q2 = expanded_variance(A2, B2, C2, r2);
            bool c0 = q0 < kStreamCancel * A0 || !k0, c1f = q1 < kStreamCancel * A1 || !k1,
                 c2f = q2 < kStreamCancel * A2 || !k2;
            double u0, u1, u2;
            if (has_flat) {
                double rf0, rf1, rf2;
                if (flat_u8) {
                    mbar_wait(&c_full[s], phase);
                    const uint32_t* aw = reinterpret_cast<const uint32_t*>(ring + (size_t)s * kStage) + a_word;
                    const uint32_t pkf = __funnelshift_r(aw[0], aw[1], a_shift) & 0xFFFFFFu;
                    rf0 = kRecip255.v[pkf & 0xFF];
                    rf1 = kRecip255.v[(pkf >> 8) & 0xFF];
                    rf2 = kRecip255.v[pkf >> 16];
                    __syncwarp();
                    if (lane == 0 && consumed(rf0, rf1, rf2)) mbar_arrive(&empty[s]);     // (1/flat >= 0, or +inf)
                    if (++s == stages) { s = 0; phase ^= 1; }
                } else {
                    rf0 = flat_recip(p.flat, p.flat_bytes, i0 + 0, p.max_dn);
                    rf1 = flat_recip(p.flat, p.flat_bytes, i0 + 1, p.max_dn);
                    rf2 = flat_recip(p.flat, p.flat_bytes, i0 + 2, p.max_dn);
                }
                constexpr int c1 = MONO ? 0 : 1, c2 = MONO ? 0 : 2;
                c0 |= !flat_apply_main_path(v0, u0, (q0 * r0) * r0, rf0, f0, p.flat_means[0], p.flat_means[kCt + 0]);
                c1f |= !flat_apply_main_path(v1, u1, (q1 * r1) * r1, rf1, f1, p.flat_means[c1], p.flat_means[kCt + c1]);
                c2f |= !flat_apply_main_path(v2, u2, (q2 * r2) * r2, rf2, f2, p.flat_means[c2], p.flat_means[kCt + c2]);
            } else {
                bool s0, s1, s2;
                const double t0 = sqrt_main_path(q0, s0), t1 = sqrt_main_path(q1, s1), t2 = sqrt_main_path(q2, s2);
                u0 = (s0 ? t0 : 0.0) * r0; u1 = (s1 ? t1 : 0.0) * r1; u2 = (s2 ? t2 : 0.0) * r2;
                c0 |= !(s0 || q0 == 0.0); c1f |= !(s1 || q1 == 0.0); c2f |= !(s2 || q2 == 0.0);
            }
            // samples whose expansion cancelled (or that left a main path) go to the exact formula (work list ->
            // merge_fixup_kernel)
            if (__any_sync(0xffffffffu, c0 | c1f | c2f)) {
                flag_sample(p, c0, (uint32_t)i0 + 0u, lane);
                flag_sample(p, c1f, (uint32_t)i0 + 1u, lane);
                flag_sample(p, c2f, (uint32_t)i0 + 2u, lane);
            }
            __stcs(p.out_val + i0 + 0, v0); __stcs(p.out_val + i0 + 1, v1); __stcs(p.out_val + i0 + 2, v2);
            __stcs(p.out_std + i0 + 0, u0); __stcs(p.out_std + i0 + 1, u1); __stcs(p.out_std + i0 + 2, u2);
        }
    }
}

bool make_slut_layout(SLutLayout& L) {
    uint32_t off = 0;
    L.off_t1 = off; off += kC * 256 * kCopies * 16;
    L.off_t2 = off; off += kC * 256 * kCopies * 16;
    L.off_ring = off;
    const size_t room = kSmemLimit - 256 - 2 * kBucketCap * sizeof(MedEntry) - off;
    int stages = (int)(room / kStage);
    if (stages > kMaxStages) stages = kMaxStages;
    L.stages = stages;
    off += (uint32_t)stages * kStage;
    L.off_bars = off; off += 256;          // (also absorbs the last pixel's second DN word of the last stage)
    L.off_med = off; off += 2 * kBucketCap * sizeof(MedEntry);
    L.total = off;
    return stages >= 2;
}

}  // namespace

int try_merge_stream_lut(const MergeParams& p_in, cudaStream_t stream) {
    SLutLayout L;
    if (!tile_stack(p_in, false) || p_in.n < 2 || !make_slut_layout(L)) return CL_ERR_UNSUPPORTED;
    MergeParams p = p_in;
    p.stream_mode = 2;
    return launch_tile_kernel(p, p.C == 1 ? merge_stream_lut_kernel<true> : merge_stream_lut_kernel<false>, kThreads,
                              L, stream);
}

}  // namespace cl
