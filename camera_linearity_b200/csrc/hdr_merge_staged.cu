// K2 fast path ("algo 2"): bulk-copy staged HDR merge for 8-bit, 3-channel stacks on sm_100a -- and for
// 8-bit mono stacks, which run through the same kernel as "virtual RGB": samples are independent, so a
// (H, W, 1) image is processed as H*W/3 three-sample pixels with the one LUT column in all three table
// slots; only the bad-pixel median (true neighbourhood geometry) and the flat-field means (one channel)
// look at the real channel count.
//
// One persistent CTA per SM (grid = #SMs), 16 consumer warps + 2 producer warps + median warp + patcher warp:
//   * producer warp 0 streams the float64 uncertainty images through a ring of shared-memory
//     stages with cp.async.bulk (the TMA engine's 1-D bulk copy, SASS UBLKCP) and mbarrier
//     transaction counts -- one 12 KB chunk per (tile, exposure);
//   * producer warp 1 bulk-copies the DN bytes of ALL exposures of the next tile (+ flat DN bytes and
//     the tile's bad-pixel bucket) into the "A buffer" while the consumers are still in pass B of
//     the current tile;
//   * consumer thread t owns pixel t of the 512-pixel tile (3 interleaved samples).  Pass A sums
//     the Gaussian weights from the A buffer and packs the DNs into one register per exposure;
//     pass B consumes one ring stage per exposure.
// Bad pixels (dark frame above threshold, ~0.1 % of the samples) never touch the consumers' loops:
// a median gather inside the streaming loop stalls the whole CTA through the ring (measured: 37 us
// per tile instead of 5).  `dark_scan_kernel` streams the dark frames once and files every bad
// (sample, exposure) in a per-tile bucket.  Inside this kernel the MEDIAN warp takes the bucket of
// the NEXT tile as soon as its A buffer has landed, gathers the K x K neighbourhoods from global
// memory (one lane per bad pixel), writes the repaired DN over the staged byte and the repaired
// sigma into the bucket; the PATCHER warp writes that sigma over ring stage (tile, k) right after
// it lands.  Only then are a_ready / ready[s] signalled to the consumers.  Tiles with more than 32
// bad pairs spill to a global list that `merge_fixup_kernel` recomputes in full afterwards.
// Shared-memory tables are replicated per lane so that the random, DN-indexed gathers are bank-
// conflict free: w[dn] as 16 copies of a double (LDS.64: half-warp lanes hit 16 distinct bank
// pairs), {w*g, dICRF}[c][dn] as 8 copies of a double2 (LDS.128: quarter-warp lanes hit 8
// distinct bank quads).  Without the replication a random 8-bit gather costs ~3 wavefronts per
// half-warp and the kernel is shared-memory bound well below the HBM roofline (DESIGN.md).
// Every input byte crosses HBM once: 9 B per sample-exposure (+1 with a dark frame), 16 B out
// (+ ~1.5 KB of scattered re-reads per bad sample in the fix-up).
#include "staged_common.cuh"

namespace cl {
namespace {

constexpr int kTilePx = kStagedTilePx;
constexpr int kC = 3;
constexpr int kConsumerWarps = kTilePx / 32;
constexpr int kThreads = kTilePx + 128;         // + ring producer, A-buffer producer, median and patcher warps
constexpr int kDnChunk = kTilePx * kC;          // bytes of one exposure's DN tile
constexpr int kStdChunk = kTilePx * kC * 8;     // bytes of one exposure's std tile
constexpr int kLutACopies = 16;
constexpr int kLutBCopies = 8;
constexpr int kMaxStages = 8;
constexpr size_t kSmemLimit = 227 * 1024;

struct StagedLayout {
    int stages;
    uint32_t off_lutA, off_lutB, off_abuf_dn, off_bucket, off_ring, off_bars, total;
};

using namespace staged;      // PTX wrappers + stage-release predicates (staged_common.cuh)

// MONO: the stack has one channel and is processed as virtual RGB (see the file header); a template
// parameter so that the RGB instantiation is exactly the code it was before mono support
template <int NMAX, bool MONO>
__global__ void __launch_bounds__(kThreads, 1)
merge_staged_kernel(const __grid_constant__ MergeParams p, const StagedLayout L, const int n_tiles) {
    constexpr int kCt = MONO ? 1 : kC;           // true channel count
    extern __shared__ __align__(128) unsigned char smem[];
    double* lutA = reinterpret_cast<double*>(smem + L.off_lutA);
    double2* lutB = reinterpret_cast<double2*>(smem + L.off_lutB);
    uint8_t* abuf_dn = smem + L.off_abuf_dn;
    uint32_t* bucket_s = reinterpret_cast<uint32_t*>(smem + L.off_bucket);               // [kBucketWords]
    const bool patched = p.any_dark != 0;
    unsigned char* ring = smem + L.off_ring;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.off_bars);
    uint64_t* full = bars;                    // [stages]  producer -> consumers (tx bytes)
    uint64_t* empty = bars + kMaxStages;      // [stages]  consumers -> producer
    uint64_t* ready = bars + 2 * kMaxStages;  // [stages]  patcher -> consumers (bad-pixel patches applied)
    uint64_t* a_full = bars + 3 * kMaxStages;
    uint64_t* a_empty = a_full + 1;
    uint64_t* a_ready = a_full + 2;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const int stages = L.stages;
    const bool has_flat = p.flat_bytes != 0;
    const bool flat_u8 = p.flat_bytes == 1;     // flat DN bytes ride in the A buffer (slot n)

    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumerWarps);
            mbar_init(&ready[s], 1);
        }
        mbar_init(a_full, 1);
        mbar_init(a_empty, kConsumerWarps + (patched ? 1 : 0));   // + the patcher warp (it reads the bucket)
        mbar_init(a_ready, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();          // barriers are initialised: the producer warps start streaming right away,
                              // under the table construction below (only the consumers use the tables)
    if (warp < kConsumerWarps) {
        // replicated tables (see file header): the work is spread over all 512 consumer threads
        for (int it = tid; it < 256 * 4; it += kTilePx) {
            const int d = it >> 2, part = it & 3;            // part 0: w[d]; parts 1..3: channel part-1
            double w, dw;
            gaussian_weight(__ddiv_rn((double)d, p.max_dn), w, dw);
            if (part == 0) {
#pragma unroll
                for (int r = 0; r < kLutACopies; ++r) lutA[d * kLutACopies + r] = w;
            } else {
                const int c = part - 1;
                const int cs = MONO ? 0 : c;                 // mono: the single LUT column in every slot
                const double2 e = make_double2(w * p.lut[d * kCt + cs], p.dlut[d * kCt + cs]);
#pragma unroll
                for (int r = 0; r < kLutBCopies; ++r) lutB[(c * 256 + d) * kLutBCopies + r] = e;
            }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kTilePx) : "memory");    // consumers only
    }

    if (warp == kConsumerWarps) {
        // ===== ring producer: std chunks (tile-major, exposure-minor; flat std last) =====
        if (lane == 0) {
            int s = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const size_t off = (size_t)tile * kTilePx * kC;   // first sample of the tile
                const int chunks = p.n + (has_flat ? 1 : 0);
                for (int k = 0; k < chunks; ++k) {
                    mbar_wait(&empty[s], phase ^ 1);
                    mbar_expect_tx(&full[s], kStdChunk);
                    const double* src = (k < p.n ? p.std[k] : p.flat_std) + off;
                    bulk_g2s(ring + (size_t)s * kStdChunk, src, kStdChunk, &full[s]);
                    if (++s == stages) { s = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == kConsumerWarps + 1) {
        // ===== A-buffer producer: DN bytes of every exposure of one tile =====
        if (lane == 0) {
            uint32_t ti = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                const size_t off = (size_t)tile * kDnChunk;
                mbar_wait(a_empty, (ti & 1) ^ 1);
                mbar_expect_tx(a_full, (uint32_t)(p.n + (flat_u8 ? 1 : 0)) * kDnChunk +
                                           (patched ? kBucketWords * 4u : 0u));
                if (patched) {          // count block (16 B) + entries (512 B) land back to back
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
    } else if (warp == kConsumerWarps + 2) {
        // ===== median warp: repairs the bad pixels of the NEXT tile while the consumers work =====
        // lane e owns bucket entry e {pixel, channel, exposure} (filed by dark_scan_kernel).  It gathers
        // the K x K neighbourhoods from global memory, writes the median DN over the staged byte in the
        // A buffer and the median sigma into the bucket entry, then declares the A buffer ready.
        if (patched) {
            uint32_t ti = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                mbar_wait(a_full, ti & 1);
                const uint32_t n_patch = min(bucket_s[0], (uint32_t)kBucketCap);
                if ((uint32_t)lane < n_patch) {
                    const uint32_t meta = bucket_s[4 + 4 * lane];
                    const int pix = (int)(meta & 511u), c = (int)((meta >> 9) & 3u), ke = (int)((meta >> 11) & 31u);
                    // true image coordinates of the sample (mono: every sample is a pixel)
                    // (32-bit arithmetic: this warp's latency gates a_ready, and the staged path has < 2^32 samples)
                    const uint32_t tpx = (uint32_t)tile * kTilePx + (uint32_t)pix;
                    const uint32_t px = MONO ? tpx * kC + (uint32_t)c : tpx;
                    const int ct = MONO ? 0 : c;
                    const int y = (int)(px / (uint32_t)p.W), x = (int)(px - (uint32_t)y * (uint32_t)p.W);
                    const uint8_t* img = reinterpret_cast<const uint8_t*>(p.dn[ke]);
                    uint32_t d_new;
                    double s_new;
                    median_pair(img, p.std[ke], p.std_lut, y, x, ct, p.H, p.W, kCt, p.K, d_new, s_new);
                    abuf_dn[ke * kDnChunk + pix * kC + c] = (uint8_t)d_new;
                    *reinterpret_cast<double*>(bucket_s + 4 + 4 * lane + 2) = s_new;
                }
                // generic-proxy writes into buffers the TMA engine refills later
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(a_ready);
            }
        }
    } else if (warp == kConsumerWarps + 3) {
        // ===== patcher: writes the repaired sigmas over ring stage (tile, k) right after it lands =====
        // consumers wait on a_ready / ready[] instead of a_full / full[], so their loops carry no
        // patch code and stay exact.
        if (patched) {
            uint32_t ti = 0, phase = 0;
            int s = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
                mbar_wait(a_ready, ti & 1);
                const uint32_t n_patch = min(bucket_s[0], (uint32_t)kBucketCap);
                const bool mine = (uint32_t)lane < n_patch;
                const uint32_t meta = mine ? bucket_s[4 + 4 * lane] : 0u;
                const double sig = mine ? *reinterpret_cast<const double*>(bucket_s + 4 + 4 * lane + 2) : 0.0;
                const uint32_t pos = (meta & 511u) * kC + ((meta >> 9) & 3u);     // sample within the tile
                const int ke = (int)((meta >> 11) & 31u);
                __syncwarp();
                // the bucket is in registers now: let the A-buffer producer refill (with the consumers)
                if (lane == 0 && consumed(sig * sig, (double)meta, 0.0)) mbar_arrive(a_empty);
                const int chunks = p.n + (has_flat ? 1 : 0);
                for (int k = 0; k < chunks; ++k) {
                    mbar_wait(&full[s], phase);
                    const bool hit = mine && ke == k;
                    if (hit) reinterpret_cast<double*>(ring + (size_t)s * kStdChunk)[pos] = sig;
                    if (__any_sync(0xffffffffu, hit))
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // before the TMA refill
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&ready[s]);
                    if (++s == stages) { s = 0; phase ^= 1; }
                }
            }
        }
    } else {
        // ===== consumers: thread tid owns pixel tid of each tile =====
        uint64_t* const c_full = patched ? ready : full;          // what "stage is ready" means
        uint64_t* const c_afull = patched ? a_ready : a_full;
        const double* myA = lutA + (lane & (kLutACopies - 1));
        const double2* myB = lutB + (lane & (kLutBCopies - 1));
        // bytes tid*3 .. tid*3+2 of a DN chunk live in words a_word, a_word+1 (the second word of the last
        // pixel lies just past the chunk -- still inside the A buffer / the bucket that follows it -- and
        // contributes only the masked-off top byte)
        const int a_word = (tid * kC) >> 2;
        const uint32_t a_shift = ((tid * kC) & 3) * 8;
        uint32_t ti = 0, phase = 0;
        int s = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++ti) {
            const int64_t px = (int64_t)tile * kTilePx + tid;
            // ---- pass A: sum of weights; pack the DNs of every exposure into registers ----
            mbar_wait(c_afull, ti & 1);
            uint32_t pk[NMAX];
            double S0 = 0.0, S1 = 0.0, S2 = 0.0;
#pragma unroll
            for (int k = 0; k < NMAX; ++k) {
                if (k < p.n) {
                    // the pixel's 3 DN bytes out of two aligned words (2 shared loads instead of 3 byte loads)
                    const uint32_t* aw = reinterpret_cast<const uint32_t*>(abuf_dn + k * kDnChunk) + a_word;
                    const uint32_t q = __funnelshift_r(aw[0], aw[1], a_shift) & 0xFFFFFFu;
                    const uint32_t d0 = q & 0xFF, d1 = (q >> 8) & 0xFF, d2 = q >> 16;
                    S0 += myA[d0 * kLutACopies];
                    S1 += myA[d1 * kLutACopies];
                    S2 += myA[d2 * kLutACopies];
                    pk[k] = q;
                }
            }
            uint32_t pkf = 0;
            if (flat_u8) {
                const uint32_t* aw = reinterpret_cast<const uint32_t*>(abuf_dn + p.n * kDnChunk) + a_word;
                pkf = __funnelshift_r(aw[0], aw[1], a_shift) & 0xFFFFFFu;
            }
            // release the A buffer; consumed(S) ties the release to the arithmetic that used its bytes
            __syncwarp();
            if (lane == 0 && consumed(S0, S1, S2 + (double)pkf)) mbar_arrive(a_empty);   // pkf >= 0
            const double r0 = 1.0 / S0, r1 = 1.0 / S1, r2 = 1.0 / S2;

            // ---- pass B: one ring stage per exposure ----
            double av0 = 0.0, av1 = 0.0, av2 = 0.0, as0 = 0.0, as1 = 0.0, as2 = 0.0;
#pragma unroll
            for (int k = 0; k < NMAX; ++k) {
                if (k < p.n) {
                    mbar_wait(&c_full[s], phase);
                    const double* sp = reinterpret_cast<const double*>(ring + (size_t)s * kStdChunk) + tid * kC;
                    const double g0 = sp[0], g1 = sp[1], g2 = sp[2];
                    const uint32_t q = pk[k];
                    const uint32_t d0 = q & 0xFF, d1 = (q >> 8) & 0xFF, d2 = q >> 16;
                    const double rt = p.inv_t[k];
                    const double w0 = myA[d0 * kLutACopies], w1 = myA[d1 * kLutACopies], w2 = myA[d2 * kLutACopies];
                    const double2 e0 = myB[(0 * 256 + d0) * kLutBCopies];
                    const double2 e1 = myB[(1 * 256 + d1) * kLutBCopies];
                    const double2 e2 = myB[(2 * 256 + d2) * kLutBCopies];
                    merge_accumulate(w0, e0.x, e0.y, kappa_of(d0, p.kappa_scale), g0, r0, rt, av0, as0);
                    merge_accumulate(w1, e1.x, e1.y, kappa_of(d1, p.kappa_scale), g1, r1, rt, av1, as1);
                    merge_accumulate(w2, e2.x, e2.y, kappa_of(d2, p.kappa_scale), g2, r2, rt, av2, as2);
                    __syncwarp();
                    if (lane == 0 && consumed_nonneg(as0, as1, as2)) mbar_arrive(&empty[s]);
                    if (++s == stages) { s = 0; phase ^= 1; }
                }
            }

            double v0 = av0 * r0, v1 = av1 * r1, v2 = av2 * r2;
            double u0, u1, u2;
            const int64_t i0 = px * kC;
            if (has_flat) {
                mbar_wait(&c_full[s], phase);
                const double* sp = reinterpret_cast<const double*>(ring + (size_t)s * kStdChunk) + tid * kC;
                const double f0 = sp[0], f1 = sp[1], f2 = sp[2];
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
                constexpr int c1 = MONO ? 0 : 1, c2 = MONO ? 0 : 2;           // flat_means = [C means | C std means]
                flat_apply(v0, u0, (as0 * r0) * r0, rf0, f0, p.flat_means[0], p.flat_means[kCt + 0]);
                flat_apply(v1, u1, (as1 * r1) * r1, rf1, f1, p.flat_means[c1], p.flat_means[kCt + c1]);
                flat_apply(v2, u2, (as2 * r2) * r2, rf2, f2, p.flat_means[c2], p.flat_means[kCt + c2]);
                __syncwarp();
                if (lane == 0 && consumed(u0, u1, u2)) mbar_arrive(&empty[s]);
                if (++s == stages) { s = 0; phase ^= 1; }
            } else {
                u0 = sqrt(as0) * r0; u1 = sqrt(as1) * r1; u2 = sqrt(as2) * r2;
            }
            __stcs(p.out_val + i0 + 0, v0); __stcs(p.out_val + i0 + 1, v1); __stcs(p.out_val + i0 + 2, v2);
            __stcs(p.out_std + i0 + 0, u0); __stcs(p.out_std + i0 + 1, u1); __stcs(p.out_std + i0 + 2, u2);
        }
    }
}

bool make_layout(const MergeParams& p, StagedLayout& L) {
    uint32_t off = 0;
    L.off_lutA = off; off += 256 * kLutACopies * 8;
    L.off_lutB = off; off += kC * 256 * kLutBCopies * 16;
    L.off_abuf_dn = off; off += (uint32_t)(p.n + (p.flat_bytes == 1 ? 1 : 0)) * kDnChunk;
    L.off_bucket = off; if (p.any_dark) off += kBucketWords * 4;
    off = (off + 127) & ~127u;
    L.off_ring = off;
    const size_t room = kSmemLimit - 256 - off;
    int stages = (int)(room / kStdChunk);
    if (stages > kMaxStages) stages = kMaxStages;
    L.stages = stages;
    off += (uint32_t)stages * kStdChunk;
    L.off_bars = off; off += 256;
    L.total = off;
    return stages >= 3;
}

}  // namespace

int try_merge_staged(const MergeParams& p, cudaStream_t stream) {
    StagedLayout L;
    if (!tile_stack(p, true) || !make_layout(p, L)) return CL_ERR_UNSUPPORTED;
    const bool mono = p.C == 1;
    auto kernel = p.n <= 8    ? (mono ? merge_staged_kernel<8, true> : merge_staged_kernel<8, false>)
                  : p.n <= 16 ? (mono ? merge_staged_kernel<16, true> : merge_staged_kernel<16, false>)
                              : (mono ? merge_staged_kernel<32, true> : merge_staged_kernel<32, false>);
    return launch_tile_kernel(p, kernel, kThreads, L, stream);
}

}  // namespace cl
