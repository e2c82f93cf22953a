// K4: ICRF calibration objective for a whole differential-evolution population in one launch.
// Replaces ICRF_calibration_exposure.py:20-44, 66-201 and general_functions.py:149-176.
//
// Mapping: one LANE per candidate curve (32 candidates per warp), one WARP-ITERATION per pixel.
// The pixel's N digital numbers are warp-uniform, so the candidate tables are laid out
// [dn][candidate] and every gather `table[dn_k][lane]` is a contiguous, conflict-free 256-byte
// row of shared memory.  Two tables per candidate group: I (the curve value, NaN where the range
// mask of :97-98 applies -- the mask depends only on the DN) and R = 1/I.  Each lane keeps the
// per-exposure-pair numerator / denominator of ITS candidate in registers, so no cross-lane
// reduction is needed at all; warps are combined through shared memory and CTAs in a fixed order
// (deterministic).
//
// Arithmetic per pixel: with A_i = I_i / t_i and B_j = t_j / I_j (2N multiplies per pixel) the relative
// difference of pair (i, j),  |I_i - r I_j| / (r I_j)  with r = t_i / t_j (:101-121), is |A_i B_j - 1|: ONE
// FMA per pair, its absolute value is a source modifier of the accumulating add, the NaN test runs on the
// integer pipe and the valid count is an integer add -- 2 FP64-pipe instructions per pair instead of 6.
//
// Range masks without per-lane work: a candidate that passes the gates is STRICTLY INCREASING (:178), so
// "I < curve[lower] or I > curve[upper]" (:97-98) is exactly "dn < lower or dn > upper" -- the same for every
// candidate, warp-uniform, and a gated candidate's energy is +inf whatever its sums are.  With lower >= 1 every
// unmasked I is > 0, so no NaN / inf can arise: masked table entries are stored as 0 (A_i B_j - 1 = -1, |.| = 1
// exactly), the pair sums are accumulated unconditionally and each lane subtracts the number of masked pairs at
// the end (a lane sees a few hundred pixels, so the subtraction costs ~1e-14 relative); the valid counts are
// kept by lane q for pair q from the warp-uniform DN range bits.  The kernel is issue bound (80 % issue-slot
// utilisation, FP64 pipe 30 %): this took the pixel loop from ~125 to ~80 instructions.  lower == 0 keeps the
// NaN-checking path (0/0 at DN 0 must be skipped, x/0 = inf kept, as np.nanmean does).
//
// Multi-GPU: pixels are sharded over the ranks; `energy_tail_kernel` reduces this rank's CTAs, PUSHES the
// (S x pairs x 2) sums into every peer's exchange buffer over NVLink (plain stores to peer memory), raises a
// flag on each peer, waits for the peers' flags and sums the W contributions in rank order -- so every rank
// finalises identical numbers without an NCCL launch (one fused kernel instead of reduce + all-reduce +
// finalize).  Bound: FP64 pipe + shared-memory gathers; the 2-18 MB of pixel data stay in L2.
//
// 16-bit cameras (uint16 samples, curves of up to 65536 points): the curves are built by one thread-block cluster per
// candidate and the partial kernel gathers its table rows from global memory (L1 / L2) instead of shared memory --
// see curves_wide_kernel and GLOBAL_TABLES below.
#include "de_common.cuh"

#include <cooperative_groups.h>

#include <cstring>

namespace cl {
namespace {

constexpr int kGroup = 32;            // candidates per warp
constexpr int kMaxN = CL_MAX_PAIR_EXPOSURES;

__host__ __device__ inline int n_pairs(int n) { return n * (n - 1) / 2; }

// see the file header: lower >= 1 makes the range masks a property of the DN alone.  Swapped limits (upper < lower)
// mask every sample of a candidate that passes the gates; the NaN-checking path gives that +inf, while the uniform
// pixel loop's unsigned span test would wrap and count the DNs outside (upper, lower) as valid.
__host__ __device__ inline bool uniform_masks(const cl_icrf_problem& p) { return p.lower >= 1 && p.lower <= p.upper; }

struct ExposureScales {
    double inv_t[kMaxN];              // 1 / t_k
    double t[kMaxN];
};

// R-table entry of an unmasked point on the uniform path.  A subnormal curve value has 1/v = inf, and the weighted
// loop's fma(|u - 1|, w = 0, num) would turn the whole pair sum into NaN; the reference gives such a pair the weight
// 0 (its propagated sigma overflows), which R = 0 reproduces exactly: u = t1 = t2 = 0, so var = 0 and w = 0.
__device__ __forceinline__ double reciprocal(const cl_icrf_problem& prob, double v) {
    const double r = 1.0 / v;
    return prob.use_std && isinf(r) ? 0.0 : r;
}

// ---- candidate curves, gates and tables -----------------------------------------------------------
// One CTA per candidate, one thread per curve point.  `p` points at the candidate's parameters (global or
// shared memory).  Tables: tab[0 .. S*D) = I, tab[S*D .. 2*S*D) = R, each laid out [group][dn][lane].
__device__ __forceinline__ void build_curve(const cl_icrf_problem& prob, const double* __restrict__ mean_icrf,
                                            const double* __restrict__ pca, const double* p, int s,
                                            double* __restrict__ curves, int32_t* __restrict__ valid,
                                            double* __restrict__ tables, double* sc /* shared [256] */) {
    const int d = threadIdx.x, D = prob.datapoints;
    const int n_pc = prob.use_mean_icrf ? prob.n_params : prob.n_params - 1;
    const double* coef = prob.use_mean_icrf ? p : p + 1;
    double v = 0.0;
    if (d < D) {
        double acc = 0.0;                       // matmul(PCA_array, params), :38-40
        for (int k = 0; k < n_pc; ++k) acc = __dadd_rn(acc, __dmul_rn(pca[d * n_pc + k], coef[k]));
        double base;
        if (prob.use_mean_icrf) {
            base = mean_icrf[d];
        } else {                                // linspace(0, 1, BITS) ** p[0], :37
            const double x = (d == D - 1) ? 1.0 : __dmul_rn((double)d, __ddiv_rn(1.0, (double)(D - 1)));
            base = pow(x, p[0]);
        }
        v = __dadd_rn(base, acc);
        sc[d] = v;
    }
    __syncthreads();
    const double shift = __dsub_rn(1.0, sc[D - 1]);     // ICRF += 1 - ICRF[-1], :167
    __syncthreads();
    if (d < D) {
        v = __dadd_rn(v, shift);
        if (d == 0) v = 0.0;                             // ICRF[0] = 0, :168
        sc[d] = v;
    }
    __syncthreads();
    int bad = 0;
    if (d < D) {
        if (v > 1.0 || v < 0.0) bad = 1;                 // :174  (NaN compares false, like NumPy max)
        if (d > 0 && !(v > sc[d - 1])) bad = 1;          // :178  strictly increasing
        if (v != v) bad = 1;                             // NaN: np.max -> NaN, comparisons False, then
                                                         // `all(nan > ..)` is False -> inf as well
    }
    bad = __syncthreads_or(bad);
    if (d < D) {
        curves[(int64_t)s * D + d] = v;
        const double lo = sc[prob.lower], hi = sc[prob.upper];      // :182-183
        const bool masked = v < lo || v > hi;                                                   // :97-98
        const int64_t at = ((int64_t)(s / kGroup) * D + d) * kGroup + (s % kGroup);
        if (uniform_masks(prob)) {          // masked entries contribute |0 * x - 1| = 1, subtracted by the kernel
            // A gated candidate's energy is +inf whatever its sums are, and its curve need not be monotone, so its
            // own mask could zero entries INSIDE the DN range; the weighted pixel loop would take those for
            // zero-variance pairs and walk its pixels a second time.  It gets the benign table 1 on [lower, upper].
            const bool inside = d >= prob.lower && d <= prob.upper;
            tables[at] = bad ? (inside ? 1.0 : 0.0) : (masked ? 0.0 : v);
            tables[(int64_t)prob.n_candidates * D + at] = bad ? (inside ? 1.0 : 0.0) : (masked ? 0.0 : reciprocal(prob, v));
        } else {
            const double m = masked ? __longlong_as_double(0x7ff8000000000000LL) : v;
            tables[at] = m;
            tables[(int64_t)prob.n_candidates * D + at] = 1.0 / m;
        }
    }
    if (d == 0) valid[s] = bad ? 0 : 1;
}

__global__ void curves_kernel(const cl_icrf_problem prob, const double* __restrict__ mean_icrf,
                              const double* __restrict__ pca, const double* __restrict__ params,
                              double* __restrict__ curves, int32_t* __restrict__ valid, double* __restrict__ tables) {
    __shared__ double sc[256];
    build_curve(prob, mean_icrf, pca, params + (int64_t)blockIdx.x * prob.n_params, blockIdx.x, curves, valid, tables, sc);
}

// DE trial step (de_common.cuh) fused with the curve construction: CTA s draws member s's trial vector, keeps
// the scaled parameters in shared memory and builds the candidate's curve and tables from them.
__global__ void de_trial_curves_kernel(const cl_icrf_problem prob, const double* __restrict__ pop, int n_members,
                                       const de::TrialConfig cfg, const int64_t* __restrict__ generation,
                                       const double* __restrict__ lo, const double* __restrict__ hi,
                                       double* __restrict__ trial, double* __restrict__ params,
                                       const double* __restrict__ mean_icrf, const double* __restrict__ pca,
                                       double* __restrict__ curves, int32_t* __restrict__ valid,
                                       double* __restrict__ tables) {
    __shared__ double sc[256];
    __shared__ double sp[64];
    const int s = blockIdx.x, P = prob.n_params;
    if ((int)threadIdx.x < P) {
        double tv = 0.0, pv = 0.0;
        if (s < n_members) {
            de::trial_component(pop, n_members, P, cfg, (uint64_t)generation[0], s, threadIdx.x, lo, hi, tv, pv);
            trial[s * P + threadIdx.x] = tv;
        }
        params[s * P + threadIdx.x] = pv;              // padding members (s >= n_members) evaluate the zero vector
        sp[threadIdx.x] = pv;
    }
    __syncthreads();
    build_curve(prob, mean_icrf, pca, sp, s, curves, valid, tables, sc);
}

// ---- candidate curves for 256 < D <= 65536 (16-bit cameras: D = 65536; 12-bit data in uint16: D = 4096) ----------
// One thread-block cluster per candidate: CTA r of the cluster owns the points [r * chunk, (r + 1) * chunk).  Every
// CTA recomputes the few points it needs from elsewhere -- curve[D-1] (the shift), curve[lower], curve[upper] and the
// left neighbour of its first point -- with build_curve's arithmetic, so it gets the same bits.  The gates of the
// eight CTAs meet through distributed shared memory and a cluster barrier; only then are the table rows written
// (a gated candidate gets the benign table).  One launch, no scratch to clear: capturable in a CUDA graph.
constexpr int kWideCluster = 8, kWideThreads = 1024;
constexpr int kMaxSharedDatapoints = 256;      // tables staged in shared memory up to this curve length
constexpr int kMaxDatapoints = 65536;

__host__ __device__ inline int wide_chunk(int D) { return (D + kWideCluster - 1) / kWideCluster; }
inline size_t wide_curve_smem(int D) { return (size_t)(wide_chunk(D) + 1) * sizeof(double); }

// curve[d] before the shift (:34-44): matmul(PCA_array, params) summed in order, plus the mean ICRF or linspace ** p[0].
// The same operations as build_curve, which keeps its own copy so that the D <= 256 kernels compile as before.
__device__ __forceinline__ double raw_point(const cl_icrf_problem& prob, const double* __restrict__ mean_icrf,
                                            const double* __restrict__ pca, const double* p, int d) {
    const int D = prob.datapoints;
    const int n_pc = prob.use_mean_icrf ? prob.n_params : prob.n_params - 1;
    const double* coef = prob.use_mean_icrf ? p : p + 1;
    double acc = 0.0;                       // matmul(PCA_array, params), :38-40
    for (int k = 0; k < n_pc; ++k) acc = __dadd_rn(acc, __dmul_rn(pca[d * n_pc + k], coef[k]));
    double base;
    if (prob.use_mean_icrf) {
        base = mean_icrf[d];
    } else {                                // linspace(0, 1, BITS) ** p[0], :37
        const double x = (d == D - 1) ? 1.0 : __dmul_rn((double)d, __ddiv_rn(1.0, (double)(D - 1)));
        base = pow(x, p[0]);
    }
    return __dadd_rn(base, acc);
}

// Curve point d of candidate s (value v, its gate decision `bad`, the curve's values lo / hi at the data limits) into
// `curves` and the I / R tables.
__device__ __forceinline__ void store_point(const cl_icrf_problem& prob, int s, int d, double v, int bad, double lo,
                                            double hi, double* __restrict__ curves, double* __restrict__ tables) {
    const int D = prob.datapoints;
    curves[(int64_t)s * D + d] = v;
    const bool masked = v < lo || v > hi;                                                   // :97-98
    const int64_t at = ((int64_t)(s / kGroup) * D + d) * kGroup + (s % kGroup);
    if (uniform_masks(prob)) {          // masked entries contribute |0 * x - 1| = 1, subtracted by the kernel
        // A gated candidate's energy is +inf whatever its sums are, and its curve need not be monotone, so its
        // own mask could zero entries INSIDE the DN range; the weighted pixel loop would take those for
        // zero-variance pairs and walk its pixels a second time.  It gets the benign table 1 on [lower, upper].
        const bool inside = d >= prob.lower && d <= prob.upper;
        tables[at] = bad ? (inside ? 1.0 : 0.0) : (masked ? 0.0 : v);
        tables[(int64_t)prob.n_candidates * D + at] = bad ? (inside ? 1.0 : 0.0) : (masked ? 0.0 : reciprocal(prob, v));
    } else {
        const double m = masked ? __longlong_as_double(0x7ff8000000000000LL) : v;
        tables[at] = m;
        tables[(int64_t)prob.n_candidates * D + at] = 1.0 / m;
    }
}

__device__ __forceinline__ void build_curve_wide(const cl_icrf_problem& prob, const double* __restrict__ mean_icrf,
                                                 const double* __restrict__ pca, const double* p, int s,
                                                 double* __restrict__ curves, int32_t* __restrict__ valid,
                                                 double* __restrict__ tables,
                                                 double* sc /* shared [chunk + 1] */, int* gate /* shared */) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int D = prob.datapoints, rank = (int)cluster.block_rank();
    const int first = rank * wide_chunk(D), end = min(D, first + wide_chunk(D));
    const double shift = __dsub_rn(1.0, raw_point(prob, mean_icrf, pca, p, D - 1));    // ICRF += 1 - ICRF[-1], :167
    auto point = [&](int d) {                                                           // ICRF[0] = 0, :168
        return d == 0 ? 0.0 : __dadd_rn(raw_point(prob, mean_icrf, pca, p, d), shift);
    };
    double* v = sc + 1;                          // v[i] = curve[first + i], sc[0] = curve[first - 1]
    for (int i = threadIdx.x; first + i < end; i += blockDim.x) v[i] = point(first + i);
    if (threadIdx.x == 0 && first > 0) sc[0] = point(first - 1);
    __syncthreads();
    int bad = 0;
    for (int i = threadIdx.x; first + i < end; i += blockDim.x) {
        const double x = v[i];
        if (x > 1.0 || x < 0.0) bad = 1;                        // :174
        if (first + i > 0 && !(x > v[i - 1])) bad = 1;          // :178, across the CTA boundary through sc[0]
        if (x != x) bad = 1;
    }
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) *gate = bad;
    cluster.sync();                              // every CTA's gate is in its shared memory
    int any = 0;
    if ((int)threadIdx.x < kWideCluster) any = *cluster.map_shared_rank(gate, (unsigned)threadIdx.x);
    any = __syncthreads_or(any);
    cluster.sync();                              // the peers' gates are read before any CTA of the cluster exits
    const double lo = point(prob.lower), hi = point(prob.upper);                        // :182-183
    for (int i = threadIdx.x; first + i < end; i += blockDim.x)
        store_point(prob, s, first + i, v[i], any, lo, hi, curves, tables);
    if (rank == 0 && threadIdx.x == 0) valid[s] = any ? 0 : 1;
}

__global__ void __cluster_dims__(kWideCluster, 1, 1) __launch_bounds__(kWideThreads, 1)
curves_wide_kernel(const cl_icrf_problem prob, const double* __restrict__ mean_icrf, const double* __restrict__ pca,
                   const double* __restrict__ params, double* __restrict__ curves, int32_t* __restrict__ valid,
                   double* __restrict__ tables) {
    extern __shared__ double sc_wide[];
    __shared__ int gate;
    const int s = blockIdx.x / kWideCluster;
    build_curve_wide(prob, mean_icrf, pca, params + (int64_t)s * prob.n_params, s, curves, valid, tables, sc_wide, &gate);
}

// de_trial_curves_kernel for D > 256: the draws are counter based, so every CTA of the cluster re-derives its
// member's trial vector; CTA 0 of the cluster writes `trial` / `params`.
__global__ void __cluster_dims__(kWideCluster, 1, 1) __launch_bounds__(kWideThreads, 1)
de_trial_curves_wide_kernel(const cl_icrf_problem prob, const double* __restrict__ pop, int n_members,
                            const de::TrialConfig cfg, const int64_t* __restrict__ generation,
                            const double* __restrict__ lo, const double* __restrict__ hi, double* __restrict__ trial,
                            double* __restrict__ params, const double* __restrict__ mean_icrf,
                            const double* __restrict__ pca, double* __restrict__ curves, int32_t* __restrict__ valid,
                            double* __restrict__ tables) {
    extern __shared__ double sc_wide[];
    __shared__ double sp[64];
    __shared__ int gate;
    const int s = blockIdx.x / kWideCluster, P = prob.n_params;
    const bool writer = blockIdx.x % kWideCluster == 0;
    if ((int)threadIdx.x < P) {
        double tv = 0.0, pv = 0.0;
        if (s < n_members) {
            de::trial_component(pop, n_members, P, cfg, (uint64_t)generation[0], s, threadIdx.x, lo, hi, tv, pv);
            if (writer) trial[s * P + threadIdx.x] = tv;
        }
        if (writer) params[s * P + threadIdx.x] = pv;  // padding members (s >= n_members) evaluate the zero vector
        sp[threadIdx.x] = pv;
    }
    __syncthreads();
    build_curve_wide(prob, mean_icrf, pca, sp, s, curves, valid, tables, sc_wide, &gate);
}

// ---- partial energies -----------------------------------------------------------------------------
// One pixel per warp-iteration, two pixels in flight (the DN / sigma loads of the next pixel are
// issued before the arithmetic of the current one).
template <int N, bool USE_STD>
struct PixelData {
    int bin[N];
    double sg[USE_STD ? N : 1];
};

template <int N, bool USE_STD, typename DN>
__device__ __forceinline__ void load_pixel(PixelData<N, USE_STD>& d, const DN* __restrict__ dn,
                                           const double* __restrict__ sd, int64_t px, int D) {
#pragma unroll
    for (int k = 0; k < N; ++k) {
        d.bin[k] = min((int)__ldg(dn + px * N + k), D - 1);        // callers guarantee dn < D
        if (USE_STD) d.sg[USE_STD ? k : 0] = __ldg(sd + px * N + k);
    }
}

// UNIFORM (lower >= 1): `vmask` bit k = exposure k of this pixel is inside [lower, upper] (warp-uniform)
template <int N, bool USE_STD, int P>
__device__ __forceinline__ void accumulate_pixel_uniform(const PixelData<N, USE_STD>& d, uint32_t vmask,
                                                         const double* __restrict__ tabI,
                                                         const double* __restrict__ tabR, int lane,
                                                         const ExposureScales& sc, double (&num)[P], double (&den)[P]) {
    double A[N], B[N], C[USE_STD ? N : 1], Dj[USE_STD ? N : 1];
#pragma unroll
    for (int k = 0; k < N; ++k) {
        if (k < N - 1) A[k] = tabI[d.bin[k] * kGroup + lane] * sc.inv_t[k];
        if (k > 0) {
            const double r = tabR[d.bin[k] * kGroup + lane];
            B[k] = r * sc.t[k];
            if (USE_STD) Dj[USE_STD ? k : 0] = d.sg[USE_STD ? k : 0] * r;
        }
        if (USE_STD && k < N - 1) C[USE_STD ? k : 0] = d.sg[USE_STD ? k : 0] * sc.inv_t[k];
    }
    int q = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = i + 1; j < N; ++j, ++q) {
            if (!USE_STD) {
                num[q] += fabs(fma(A[i], B[j], -1.0));        // masked pair: exactly 1 (removed at the end)
            } else {
                const double u = A[i] * B[j];
                const double a = fabs(u - 1.0);
                const double t1 = C[USE_STD ? i : 0] * B[j];
                const double t2 = u * Dj[USE_STD ? j : 0];
                const double var = fma(t1, t1, t2 * t2);
                // pair inside the range (warp-uniform bit) and sigma != 0 (:134); |d| is finite here.  The weight is
                // the main path of rsqrt() without its range test and slow-path branch: ten of those per pixel
                // fenced the schedule (same-box A/B, ms per population: library rsqrt 0.375; main path with a
                // rare-case branch per PAIR 0.401, per PIXEL 0.361, with a per-pair "odd" flag and the rare cases
                // after the loop 0.361; no bookkeeping in the loop at all 0.332).  A pair that is out of range or
                // whose variance is not a normal positive number gets weight 0 and adds exact zeros.  Whether such
                // a pair CAN exist is decided before the loop from the sigmas alone (see `wild` in the kernel).
                const bool in_range = (vmask >> i) & (vmask >> j) & 1u;
                const bool fast = in_range && normal_positive(var);
                double w = rsqrt_main_path(var);
                w = fast ? w : 0.0;
                num[q] = fma(a, w, num[q]);
                den[q] += w;
            }
        }
    }
}

// Second visit of a pixel (CTAs whose sigmas are `wild` only): pairs inside the range whose variance is not a normal
// positive number -- zero / NaN (the pair is skipped, :134) or denormal (library rsqrt).  Only the latter add something.
template <int N, int P>
__device__ __forceinline__ void fix_pixel_uniform(const PixelData<N, true>& d, uint32_t vmask,
                                                  const double* __restrict__ tabI, const double* __restrict__ tabR,
                                                  int lane, const ExposureScales& sc, double (&num)[P], double (&den)[P]) {
    double A2[N], B2[N], C2[N], D2[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
        A2[k] = tabI[d.bin[k] * kGroup + lane] * sc.inv_t[k];
        const double r = tabR[d.bin[k] * kGroup + lane];
        B2[k] = r * sc.t[k];
        D2[k] = d.sg[k] * r;
        C2[k] = d.sg[k] * sc.inv_t[k];
    }
    int q = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = i + 1; j < N; ++j, ++q) {
            const double u = A2[i] * B2[j];
            const double t1 = C2[i] * B2[j];
            const double t2 = u * D2[j];
            const double var = fma(t1, t1, t2 * t2);
            if (((vmask >> i) & (vmask >> j) & 1u) && !normal_positive(var) && var > 0.0) {
                const double w = rsqrt(var);
                num[q] = fma(fabs(u - 1.0), w, num[q]);
                den[q] += w;
            }
        }
    }
}

// two pixels at once: all gathers first, then the two arithmetic chains interleaved by the compiler
template <int N, bool USE_STD, int P>
__device__ __forceinline__ void accumulate_two_pixels_uniform(const PixelData<N, USE_STD>& d0,
                                                              const PixelData<N, USE_STD>& d1, uint32_t vm0,
                                                              uint32_t vm1, const double* __restrict__ tabI,
                                                              const double* __restrict__ tabR, int lane,
                                                              const ExposureScales& sc, double (&num)[P],
                                                              double (&den)[P]) {
    if (USE_STD) {                      // (FP64 bound already: no gain from the wider window, and no registers for it)
        accumulate_pixel_uniform<N, USE_STD, P>(d0, vm0, tabI, tabR, lane, sc, num, den);
        accumulate_pixel_uniform<N, USE_STD, P>(d1, vm1, tabI, tabR, lane, sc, num, den);
        return;
    }
    double A0[N], B0[N], A1[N], B1[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
        if (k < N - 1) {
            A0[k] = tabI[d0.bin[k] * kGroup + lane];
            A1[k] = tabI[d1.bin[k] * kGroup + lane];
        }
        if (k > 0) {
            B0[k] = tabR[d0.bin[k] * kGroup + lane];
            B1[k] = tabR[d1.bin[k] * kGroup + lane];
        }
    }
#pragma unroll
    for (int k = 0; k < N; ++k) {
        if (k < N - 1) { A0[k] *= sc.inv_t[k]; A1[k] *= sc.inv_t[k]; }
        if (k > 0) { B0[k] *= sc.t[k]; B1[k] *= sc.t[k]; }
    }
    int q = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = i + 1; j < N; ++j, ++q) {
            const double a0 = fabs(fma(A0[i], B0[j], -1.0));
            const double a1 = fabs(fma(A1[i], B1[j], -1.0));
            num[q] += a0;                                   // same order as one pixel at a time
            num[q] += a1;
        }
    }
}

template <int N, bool USE_STD, int P>
__device__ __forceinline__ void accumulate_pixel(const PixelData<N, USE_STD>& d, const double* __restrict__ tabI,
                                                 const double* __restrict__ tabR, int lane,
                                                 const ExposureScales& sc, double (&num)[P], double (&den)[P],
                                                 int (&cnt)[P]) {
    double A[N], B[N], C[USE_STD ? N : 1], Dj[USE_STD ? N : 1];
#pragma unroll
    for (int k = 0; k < N; ++k) {
        if (k < N - 1) A[k] = tabI[d.bin[k] * kGroup + lane] * sc.inv_t[k];          // I_k / t_k   (exposure i of a pair)
        if (k > 0) {
            const double r = tabR[d.bin[k] * kGroup + lane];
            B[k] = r * sc.t[k];                                                      // t_k / I_k   (exposure j of a pair)
            if (USE_STD) Dj[USE_STD ? k : 0] = d.sg[USE_STD ? k : 0] * r;            // sigma_k / I_k
        }
        if (USE_STD && k < N - 1) C[USE_STD ? k : 0] = d.sg[USE_STD ? k : 0] * sc.inv_t[k];   // sigma_k / t_k
    }
    int q = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = i + 1; j < N; ++j, ++q) {
            if (!USE_STD) {
                // |I_i - scaled| / scaled = |I_i / scaled - 1|, :115-121.  nanmean (:139) skips NaN and keeps inf:
                // with quiet NaNs only, "not NaN" <=> high word (sign cleared) <= 0x7ff00000 -- integer pipe.
                const double a0 = fma(A[i], B[j], -1.0);
                const bool ok = (uint32_t)(__double2hiint(a0) & 0x7fffffff) <= 0x7ff00000u;
                if (ok) {
                    num[q] += fabs(a0);
                    cnt[q] += 1;
                }
            } else {
                const double u = A[i] * B[j];                                  // I_i / scaled
                const double a0 = u - 1.0;
                const double t1 = C[USE_STD ? i : 0] * B[j];                   // sigma_i / scaled
                const double t2 = u * Dj[USE_STD ? j : 0];                     // I_i sigma_j / (r I_j^2)
                const double var = fma(t1, t1, t2 * t2);                       // :128
                // finite |d|, sigma != 0, weight 1/sigma not NaN (:134-135, gf.nanaverage)
                const bool ok = ((uint32_t)(__double2hiint(a0) & 0x7fffffff) < 0x7ff00000u) && (var > 0.0);
                const double w = rsqrt(ok ? var : 1.0);        // (a NaN operand would send the whole warp down rsqrt's slow path)
                if (ok) {
                    num[q] = fma(fabs(a0), w, num[q]);
                    den[q] += w;
                }
            }
        }
    }
}

// DN: uint8_t or uint16_t samples.  GLOBAL_TABLES (D > 256): the candidate group's [dn][lane] tables stay in global
// memory -- 2 x D x 32 x 8 B is 32 MB at D = 65536 -- and every gather is still one contiguous 256-byte row per warp,
// served by L1 / L2 (the whole blob, 2 x S x D x 8 B = 64 MiB at S = 64, fits the 126 MB L2 next to the pixels).
template <int N, bool USE_STD, int WARPS, bool UNIFORM, typename DN = uint8_t, bool GLOBAL_TABLES = false>
__global__ void __launch_bounds__(WARPS * 32, 1)
energy_partial_kernel(const double* __restrict__ tables, int D, int S, const DN* __restrict__ dn,
                      const double* __restrict__ sd, int64_t n_pixels, int64_t px_per_cta,
                      const __grid_constant__ ExposureScales sc, int lower, int upper,
                      double* __restrict__ cta_partial /* [cta][S][pairs][2] */) {
    constexpr int P = N * (N - 1) / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int group = blockIdx.y;
    const double* srcI = tables + (int64_t)group * D * kGroup;
    const double* srcR = srcI + (int64_t)S * D;
    const double* tabI;
    const double* tabR;
    if constexpr (GLOBAL_TABLES) {
        tabI = srcI;                                               // [D][32], D * 32 < 2^31
        tabR = srcR;
    } else {
        double* stI = reinterpret_cast<double*>(smem_raw);         // [D][32]
        double* stR = stI + D * kGroup;                            // [D][32]
        for (int i = threadIdx.x; i < D * kGroup; i += WARPS * 32) {
            stI[i] = srcI[i];
            stR[i] = srcR[i];
        }
        tabI = stI;
        tabR = stR;
    }
    const int64_t first = (int64_t)blockIdx.x * px_per_cta;
    const int64_t last = min(n_pixels, first + px_per_cta);
    // `wild`: can a pair of this CTA's pixels have a variance that is not a normal positive number?  With every
    // sigma in [2^-332, 2^332], exposure-time ratios in [1e-50, 1e50] and 1/I >= 1 (a candidate that passes the
    // gates has I <= 1; a gated one has the table 1) the first variance term is >= (2^-332 * 1e-50)^2 ~ 1e-300:
    // normal, or +inf by overflow, whose exact weight is the 0 the loop adds.  So one streaming look at the CTA's
    // sigmas (L2-hot for the loop that follows) replaces any bookkeeping inside the loop; a wild CTA -- a zero, NaN,
    // negative or denormal-scale sigma somewhere -- walks its pixels a second time with the exact routine.
    int wild = 0;
    if (USE_STD && UNIFORM) {
        const double* sdc = sd + first * N;
        const int64_t count = (last - first) * N;
        for (int64_t e = threadIdx.x; e < count; e += WARPS * 32)
            wild |= !((uint32_t)(__double2hiint(__ldg(sdc + e)) - 0x2B300000) < 0x29800000u);
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
            for (int j = i + 1; j < N; ++j) {
                const double r = sc.t[j] * sc.inv_t[i];
                wild |= !(r >= 1e-50 && r <= 1e50);
            }
    }
    wild = __syncthreads_or(wild);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double num[P], den[P];
    int cnt[P];
#pragma unroll
    for (int q = 0; q < P; ++q) { num[q] = 0.0; den[q] = 0.0; cnt[q] = 0; }
    int64_t px = first + warp;
    PixelData<N, USE_STD> cur, nxt;
    if (px < last) load_pixel<N, USE_STD>(cur, dn, sd, px, D);
    if (UNIFORM) {
        // lane q (< P) counts the valid pixels of pair q = (pi, pj) from the warp-uniform range bits
        int pi = 0, pj = 1;
        {
            int q = 0;
            for (int i = 0; i < N; ++i)
                for (int j = i + 1; j < N; ++j, ++q)
                    if (q == lane) { pi = i; pj = j; }
        }
        const uint32_t span = (uint32_t)(upper - lower);
        int my_valid = 0, n_px = 0;
        // two pixels per iteration (px and px + WARPS): two independent gather -> multiply -> FMA -> add chains in
        // flight per warp -- with 4 warps per scheduler one chain left the issue slots ~25 % empty
        if (USE_STD) {                  // FP64 bound: one pixel per iteration (the second window only costs registers)
            for (; px < last; px += WARPS) {
                if (px + WARPS < last) load_pixel<N, USE_STD>(nxt, dn, sd, px + WARPS, D);     // prefetch
                uint32_t vmask = 0;
#pragma unroll
                for (int k = 0; k < N; ++k) vmask |= ((uint32_t)(cur.bin[k] - lower) <= span ? 1u : 0u) << k;
                accumulate_pixel_uniform<N, USE_STD, P>(cur, vmask, tabI, tabR, lane, sc, num, den);
                cur = nxt;
            }
            if constexpr (USE_STD) {
                if (wild) {             // rare: zero / NaN / denormal-scale sigmas in this CTA -- walk the pixels again
                    for (px = first + warp; px < last; px += WARPS) {
                        load_pixel<N, USE_STD>(cur, dn, sd, px, D);
                        uint32_t vmask = 0;
#pragma unroll
                        for (int k = 0; k < N; ++k) vmask |= ((uint32_t)(cur.bin[k] - lower) <= span ? 1u : 0u) << k;
                        fix_pixel_uniform<N, P>(cur, vmask, tabI, tabR, lane, sc, num, den);
                    }
                }
            }
        }
        PixelData<N, USE_STD> cur2, nxt2;
        if (!USE_STD && px + WARPS < last) load_pixel<N, USE_STD>(cur2, dn, sd, px + WARPS, D);
        for (; !USE_STD && px < last; px += 2 * WARPS) {
            const bool second = px + WARPS < last;
            if (px + 2 * WARPS < last) load_pixel<N, USE_STD>(nxt, dn, sd, px + 2 * WARPS, D);     // prefetch
            if (px + 3 * WARPS < last) load_pixel<N, USE_STD>(nxt2, dn, sd, px + 3 * WARPS, D);
            uint32_t vmask = 0, vmask2 = 0;
#pragma unroll
            for (int k = 0; k < N; ++k) {
                vmask |= ((uint32_t)(cur.bin[k] - lower) <= span ? 1u : 0u) << k;
                vmask2 |= ((uint32_t)(cur2.bin[k] - lower) <= span ? 1u : 0u) << k;
            }
            my_valid += (int)((vmask >> pi) & (vmask >> pj) & 1u);
            ++n_px;
            if (second) {
                my_valid += (int)((vmask2 >> pi) & (vmask2 >> pj) & 1u);
                ++n_px;
                accumulate_two_pixels_uniform<N, USE_STD, P>(cur, cur2, vmask, vmask2, tabI, tabR, lane, sc, num, den);
            } else {
                accumulate_pixel_uniform<N, USE_STD, P>(cur, vmask, tabI, tabR, lane, sc, num, den);
            }
            cur = nxt;
            cur2 = nxt2;
        }
        if (!USE_STD) {
#pragma unroll
            for (int q = 0; q < P; ++q) {
                const int valid = __shfl_sync(0xffffffffu, my_valid, q);
                num[q] -= (double)(n_px - valid);      // every masked pair added exactly 1.0
                den[q] = (double)valid;
            }
        }
    } else {
        for (; px < last; px += WARPS) {
            const int64_t pn = px + WARPS;
            if (pn < last) load_pixel<N, USE_STD>(nxt, dn, sd, pn, D);     // prefetch
            accumulate_pixel<N, USE_STD, P>(cur, tabI, tabR, lane, sc, num, den, cnt);
            cur = nxt;
        }
        if (!USE_STD) {
#pragma unroll
            for (int q = 0; q < P; ++q) den[q] = (double)cnt[q];           // exact (< 2^31 pixels per warp)
        }
    }

    // combine the CTA's warps with a fixed-order tree through shared memory (table space reused)
    double* red = reinterpret_cast<double*>(smem_raw);             // [half][2P][32]
    for (int half = WARPS / 2; half >= 1; half >>= 1) {
        __syncthreads();
        if (warp >= half && warp < 2 * half) {
#pragma unroll
            for (int q = 0; q < P; ++q) {
                red[(((warp - half) * 2 * P) + 2 * q) * 32 + lane] = num[q];
                red[(((warp - half) * 2 * P) + 2 * q + 1) * 32 + lane] = den[q];
            }
        }
        __syncthreads();
        if (warp < half) {
#pragma unroll
            for (int q = 0; q < P; ++q) {
                num[q] += red[((warp * 2 * P) + 2 * q) * 32 + lane];
                den[q] += red[((warp * 2 * P) + 2 * q + 1) * 32 + lane];
            }
        }
    }
    if (warp == 0) {
        const int s = group * kGroup + lane;
        double* out = cta_partial + (((int64_t)blockIdx.x * S + s) * P) * 2;
#pragma unroll
        for (int q = 0; q < P; ++q) {
            out[2 * q] = num[q];
            out[2 * q + 1] = den[q];
        }
    }
}

// One warp per output: lanes stride over the CTAs, then an xor tree -- a fixed order, so the result is
// deterministic (a single thread walking all CTAs' partials took 13 us of a 150 us evaluation).
__device__ __forceinline__ double reduce_over_ctas(const double* __restrict__ cta_partial, int n_ctas, int64_t per_cta,
                                                   int64_t i, int lane) {
    double s = 0.0;
#pragma unroll 4
    for (int c = lane; c < n_ctas; c += 32) s += __ldcg(cta_partial + (int64_t)c * per_cta + i);
    return warp_sum(s);
}

__global__ void reduce_ctas_kernel(const double* __restrict__ cta_partial, int n_ctas, int64_t per_cta,
                                   double* __restrict__ out) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= per_cta) return;
    const double s = reduce_over_ctas(cta_partial, n_ctas, per_cta, i, lane);
    if (lane == 0) out[i] = s;
}

__device__ __forceinline__ double energy_of(const double* __restrict__ acc /* [P][2] */, int P, int is_valid) {
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    if (!is_valid) return inf;
    double sum = 0.0;
    int cnt = 0;
    for (int q = 0; q < P; ++q) {
        const double num = acc[2 * q], den = acc[2 * q + 1];
        if (den == 0.0) continue;                    // empty pair -> NaN -> skipped by nanmean
        const double r = num / den;
        if (r != r) continue;
        sum += r;
        ++cnt;
    }
    double e = inf;
    if (cnt > 0) e = sum / (double)cnt;               // np.nanmean(linearity_data), :196
    if (e != e) e = inf;                              // :197-198
    return e;
}

__global__ void finalize_kernel(const double* __restrict__ pair_acc, const int32_t* __restrict__ valid,
                                int S, int P, double* __restrict__ energy) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    energy[s] = energy_of(pair_acc + (int64_t)s * P * 2, P, valid[s]);
}

// ---- fused tail: CTA reduction + cross-GPU exchange over peer memory + finalize -----------------------
// Exchange buffer of one rank (cl_icrf_exchange_bytes): [parity 0/1][source rank][S*P*2 doubles], then
// [source rank] uint64 flags (the sequence number of the last generation that rank has delivered).  Two
// parities: a rank can only be one generation ahead of a peer (it needs that peer's flag to go on), so the
// slot it overwrites was consumed before the peer sent the flag it has already seen.
constexpr int kTailThreads = 1024;

struct PeerGroup {
    int32_t world, rank;
    unsigned char* buf[CL_MAX_PEERS];
};

// optional DE selection run by the last block right after the finalize (cl_de_select fused in): pop == nullptr: none
struct SelectArgs {
    double* pop;
    double* energies;
    const double* trial;
    int32_t n_members, n_params;
    double tol, atol;
    int64_t* generation;
    int32_t* status;
    double* best;
};

__device__ __forceinline__ uint64_t ld_acquire_sys(const uint64_t* p) {
    uint64_t v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(kTailThreads, 1)
energy_tail_kernel(const double* __restrict__ cta_partial, int n_ctas, int S, int P, const int32_t* __restrict__ valid,
                   double* __restrict__ pair_acc, double* __restrict__ energy, const __grid_constant__ PeerGroup pg,
                   uint64_t* __restrict__ seq_counter, unsigned int* __restrict__ ticket, const SelectArgs sel) {
    const int64_t per_rank = (int64_t)S * P * 2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int warps = kTailThreads / 32;
    const int W = pg.world;
    const uint64_t seq = *seq_counter + 1;                   // (incremented by the last block, at the very end)
    const int parity = (int)(seq & 1);
    __shared__ double vals[warps];
    __shared__ bool last;
    // phase 1 (all blocks): this rank's sums, fixed order.  Warp w of a block reduces output base + w; warp 0 then
    // writes the block's 32 consecutive values -- locally, or into every rank's exchange buffer (256-byte stores
    // over NVLink) -- and fences ONCE per block (a system-scope fence per warp made this kernel 20 us long).
    for (int64_t base = (int64_t)blockIdx.x * warps; base < per_rank; base += (int64_t)gridDim.x * warps) {
        const int64_t i = base + warp;
        const double v = i < per_rank ? reduce_over_ctas(cta_partial, n_ctas, per_rank, i, lane) : 0.0;
        __syncthreads();                                      // (vals of the previous round have been read)
        if (lane == 0) vals[warp] = v;
        __syncthreads();
        if (warp == 0 && base + lane < per_rank) {
            const double mine = vals[lane];
            if (W == 1) {
                pair_acc[base + lane] = mine;
            } else {
                for (int r = 0; r < W; ++r)
                    reinterpret_cast<double*>(pg.buf[r])[((int64_t)parity * W + pg.rank) * per_rank + base + lane] = mine;
            }
        }
    }
    if (warp == 0) {
        if (W > 1) __threadfence_system(); else __threadfence();
        __syncwarp();
        if (lane == 0) last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    if (W > 1) __threadfence_system(); else __threadfence();
    if (W > 1) {
        // phase 2 (last block): flags out, flags in, sum the W contributions in rank order
        const int64_t flags_off = 2 * (int64_t)W * per_rank * (int64_t)sizeof(double);
        if ((int)threadIdx.x < W) {
            uint64_t* peer_flag = reinterpret_cast<uint64_t*>(pg.buf[threadIdx.x] + flags_off) + pg.rank;
            asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(peer_flag), "l"(seq) : "memory");
            const uint64_t* my_flag = reinterpret_cast<const uint64_t*>(pg.buf[pg.rank] + flags_off) + threadIdx.x;
            const long long t0 = clock64();
            while (ld_acquire_sys(my_flag) < seq) {
                if (clock64() - t0 > 40000000000LL) __trap();          // ~20 s: a peer died
            }
        }
        __syncthreads();
        const double* mine = reinterpret_cast<const double*>(pg.buf[pg.rank]) + (int64_t)parity * W * per_rank;
        for (int64_t i = threadIdx.x; i < per_rank; i += kTailThreads) {
            double s = 0.0;
            for (int r = 0; r < W; ++r) s += __ldcv(mine + (int64_t)r * per_rank + i);
            pair_acc[i] = s;
        }
    }
    __syncthreads();
    for (int s = threadIdx.x; s < S; s += kTailThreads) energy[s] = energy_of(pair_acc + (int64_t)s * P * 2, P, valid[s]);
    if (threadIdx.x == 0) {
        *seq_counter = seq;
        *ticket = 0;                                          // self-cleaning for the next launch
    }
    if (sel.pop) {                                            // the DE selection of this generation, same block
        __syncthreads();
        de::select_block(sel.pop, sel.energies, sel.trial, energy, sel.n_members, sel.n_params, sel.tol, sel.atol,
                         sel.generation, sel.status, sel.best);
    }
}

struct Plan {
    int groups, chunks;
    int64_t px_per_cta;
};

// CTAs per SM of the partial kernel when its tables stay in global memory (D > 256): nothing to stage, so several
// CTAs share an SM and hide the L2 latency of the gathers (see DESIGN.md, K4 for D > 256).
#ifndef CL_K4_GLOBAL_CTAS_PER_SM
#define CL_K4_GLOBAL_CTAS_PER_SM 2
#endif
constexpr int kGlobalCtasPerSm = CL_K4_GLOBAL_CTAS_PER_SM;

inline bool global_tables(const cl_icrf_problem& p) { return p.datapoints > kMaxSharedDatapoints; }

inline Plan make_plan(const cl_icrf_problem& p, int64_t n_pixels) {
    Plan pl;
    pl.groups = p.n_candidates / kGroup;
    int chunks = (global_tables(p) ? kGlobalCtasPerSm : 1) * sm_count() / (pl.groups > 0 ? pl.groups : 1);
    if (chunks < 1) chunks = 1;
    const int64_t min_px = 16 * 8;         // do not split tiny problems into idle CTAs
    if ((int64_t)chunks * min_px > n_pixels) chunks = (int)((n_pixels + min_px - 1) / min_px);
    if (chunks < 1) chunks = 1;
    pl.chunks = chunks;
    pl.px_per_cta = (n_pixels + chunks - 1) / chunks;
    return pl;
}

// max_datapoints: 256 for the uint8 entry points, 65536 for the others
inline bool problem_ok(const cl_icrf_problem* p, int max_datapoints = kMaxDatapoints) {
    return p && p->n_candidates >= kGroup && p->n_candidates % kGroup == 0 && p->n_params >= 1 &&
           p->n_params <= 64 && p->datapoints >= 2 && p->datapoints <= max_datapoints && p->lower >= 0 &&
           p->lower < p->datapoints && p->upper >= 0 && p->upper < p->datapoints && p->n_exposures >= 2 &&
           p->n_exposures <= kMaxN && (p->use_mean_icrf || p->n_params >= 2);
}

// D > 256: tables read from global memory, shared memory only for the warp reduction
template <int N, typename DN>
int launch_partial_global(const cl_icrf_problem& p, const Plan& pl, const double* tables, const DN* dn,
                          const double* sd, int64_t n_pixels, const ExposureScales& sc, double* cta_partial,
                          cudaStream_t stream) {
    // registers: 2P accumulators per lane; no spills at N = 6 with std needs more than 128 (a register cap for two
    // resident CTAs spills the accumulators at every N >= 4)
    constexpr int WARPS = N <= 5 ? 16 : 8;
    const size_t smem = (size_t)(WARPS / 2) * 2 * n_pairs(N) * 32 * sizeof(double);
    dim3 grid(pl.chunks, pl.groups);
    auto go = [&](auto kernel) -> int {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
        kernel<<<grid, WARPS * 32, smem, stream>>>(tables, p.datapoints, p.n_candidates, dn, sd, n_pixels,
                                                   pl.px_per_cta, sc, p.lower, p.upper, cta_partial);
        return launched();
    };
    if (uniform_masks(p))
        return sd ? go(energy_partial_kernel<N, true, WARPS, true, DN, true>)
                  : go(energy_partial_kernel<N, false, WARPS, true, DN, true>);
    return sd ? go(energy_partial_kernel<N, true, WARPS, false, DN, true>)
              : go(energy_partial_kernel<N, false, WARPS, false, DN, true>);
}

template <int N, typename DN>
int launch_partial(const cl_icrf_problem& p, const Plan& pl, const double* tables, const DN* dn,
                   const double* sd, int64_t n_pixels, const ExposureScales& sc, double* cta_partial,
                   cudaStream_t stream) {
    constexpr int WARPS = N <= 6 ? 16 : 8;         // registers: 2P accumulators per lane
    if constexpr (sizeof(DN) > 1)                 // (the uint8 entry points accept D <= 256 only)
        if (global_tables(p)) return launch_partial_global<N>(p, pl, tables, dn, sd, n_pixels, sc, cta_partial, stream);
    const size_t tab_bytes = (size_t)p.datapoints * kGroup * 2 * sizeof(double);
    const size_t red_bytes = (size_t)(WARPS / 2) * 2 * n_pairs(N) * 32 * sizeof(double);
    const size_t smem = tab_bytes > red_bytes ? tab_bytes : red_bytes;
    dim3 grid(pl.chunks, pl.groups);
    auto go = [&](auto kernel) -> int {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
        kernel<<<grid, WARPS * 32, smem, stream>>>(tables, p.datapoints, p.n_candidates, dn, sd, n_pixels,
                                                   pl.px_per_cta, sc, p.lower, p.upper, cta_partial);
        return launched();
    };
    if (uniform_masks(p))
        return sd ? go(energy_partial_kernel<N, true, WARPS, true, DN>)
                  : go(energy_partial_kernel<N, false, WARPS, true, DN>);
    return sd ? go(energy_partial_kernel<N, true, WARPS, false, DN>)
              : go(energy_partial_kernel<N, false, WARPS, false, DN>);
}

template <typename DN>
int run_partial(const cl_icrf_problem* p, const void* tables, const DN* dn, const double* std,
                const double* exposure_s, int64_t n_pixels, double* cta_partial, const Plan& pl, cudaStream_t s) {
    const int N = p->n_exposures;
    ExposureScales sc;
    for (int k = 0; k < kMaxN; ++k) {
        sc.t[k] = k < N ? exposure_s[k] : 0.0;
        sc.inv_t[k] = k < N ? 1.0 / exposure_s[k] : 0.0;
    }
    const double* tab = reinterpret_cast<const double*>(tables);
    switch (N) {
        case 2: return launch_partial<2>(*p, pl, tab, dn, std, n_pixels, sc, cta_partial, s);
        case 3: return launch_partial<3>(*p, pl, tab, dn, std, n_pixels, sc, cta_partial, s);
        case 4: return launch_partial<4>(*p, pl, tab, dn, std, n_pixels, sc, cta_partial, s);
        case 5: return launch_partial<5>(*p, pl, tab, dn, std, n_pixels, sc, cta_partial, s);
        case 6: return launch_partial<6>(*p, pl, tab, dn, std, n_pixels, sc, cta_partial, s);
        case 7: return launch_partial<7>(*p, pl, tab, dn, std, n_pixels, sc, cta_partial, s);
        case 8: return launch_partial<8>(*p, pl, tab, dn, std, n_pixels, sc, cta_partial, s);
        default: return CL_ERR_UNSUPPORTED;
    }
}

// workspace: [cta partials: chunks x S x P x 2 doubles][ticket, 16 bytes]
inline size_t partial_bytes(const cl_icrf_problem& p, const Plan& pl) {
    return (size_t)pl.chunks * p.n_candidates * n_pairs(p.n_exposures) * 2 * sizeof(double);
}

}  // namespace
}  // namespace cl

extern "C" size_t cl_icrf_energy_workspace_bytes(const cl_icrf_problem* p, int64_t n_pixels);

namespace cl {
namespace {

template <typename DN>
int energy_partial(const cl_icrf_problem* p, int max_datapoints, const void* tables, const DN* dn, const double* std,
                   const double* exposure_s, int64_t n_pixels, double* pair_acc, void* workspace,
                   size_t workspace_bytes, void* stream) {
    if (!problem_ok(p, max_datapoints)) return CL_ERR_INVALID_ARGUMENT;
    CL_REQUIRE(tables && exposure_s && pair_acc && n_pixels >= 0);
    CL_REQUIRE(n_pixels == 0 || dn);
    CL_REQUIRE((p->use_std != 0) == (std != nullptr) || n_pixels == 0);
    if (!workspace || workspace_bytes < cl_icrf_energy_workspace_bytes(p, n_pixels)) return CL_ERR_WORKSPACE;
    if (!aligned(workspace, 16) || !aligned(tables, 16)) return CL_ERR_ALIGNMENT;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t per_cta = (int64_t)p->n_candidates * n_pairs(p->n_exposures) * 2;
    if (n_pixels == 0) return cuda_status(cudaMemsetAsync(pair_acc, 0, per_cta * sizeof(double), s));
    double* cta_partial = reinterpret_cast<double*>(workspace);
    const Plan pl = make_plan(*p, n_pixels);
    int st = run_partial(p, tables, dn, std, exposure_s, n_pixels, cta_partial, pl, s);
    if (st != CL_OK) return st;
    reduce_ctas_kernel<<<(unsigned)((per_cta * 32 + 255) / 256), 256, 0, s>>>(cta_partial, pl.chunks, per_cta,
                                                                             pair_acc);
    return launched();
}

template <typename DN>
int energy_population(const cl_icrf_problem* p, int max_datapoints, const void* tables, const DN* dn,
                      const double* std, const double* exposure_s, int64_t n_pixels, const int32_t* valid,
                      double* pair_acc, double* energy, void* workspace, size_t workspace_bytes,
                      const cl_peer_group* peers, const cl_de_select_args* select, void* stream) {
    if (!problem_ok(p, max_datapoints)) return CL_ERR_INVALID_ARGUMENT;
    CL_REQUIRE(tables && exposure_s && valid && pair_acc && energy && n_pixels >= 1 && dn && peers);
    CL_REQUIRE((p->use_std != 0) == (std != nullptr));
    CL_REQUIRE(peers->world >= 1 && peers->world <= CL_MAX_PEERS && peers->rank >= 0 && peers->rank < peers->world);
    if (!workspace || workspace_bytes < cl_icrf_energy_workspace_bytes(p, n_pixels)) return CL_ERR_WORKSPACE;
    if (!aligned(workspace, 16) || !aligned(tables, 16)) return CL_ERR_ALIGNMENT;
    PeerGroup pg;
    pg.world = peers->world;
    pg.rank = peers->rank;
    for (int r = 0; r < CL_MAX_PEERS; ++r) {
        pg.buf[r] = r < pg.world ? reinterpret_cast<unsigned char*>(peers->buffers[r]) : nullptr;
        if (r < pg.world) CL_REQUIRE(pg.buf[r] != nullptr && aligned(pg.buf[r], 16));
    }
    cudaStream_t s = (cudaStream_t)stream;
    const int P = n_pairs(p->n_exposures);
    const Plan pl = make_plan(*p, n_pixels);
    double* cta_partial = reinterpret_cast<double*>(workspace);
    int st = run_partial(p, tables, dn, std, exposure_s, n_pixels, cta_partial, pl, s);
    if (st != CL_OK) return st;
    // seq counter and ticket live behind the flags of this rank's exchange buffer (zeroed by cl_peer_alloc)
    const size_t per_rank = (size_t)p->n_candidates * P * 2 * sizeof(double);
    unsigned char* tail = pg.buf[pg.rank] + 2 * (size_t)pg.world * per_rank + (size_t)CL_MAX_PEERS * sizeof(uint64_t);
    const int64_t outputs = (int64_t)p->n_candidates * P * 2;
    int blocks = (int)((outputs + (kTailThreads / 32) - 1) / (kTailThreads / 32));
    if (blocks > 148) blocks = 148;
    SelectArgs sel;
    memset(&sel, 0, sizeof(sel));
    if (select) {
        CL_REQUIRE(select->pop && select->energies && select->trial && select->generation && select->status && select->best);
        CL_REQUIRE(select->n_members >= 4 && select->n_members <= p->n_candidates && select->n_params == p->n_params);
        sel.pop = select->pop; sel.energies = select->energies; sel.trial = select->trial;
        sel.n_members = select->n_members; sel.n_params = select->n_params; sel.tol = select->tol; sel.atol = select->atol;
        sel.generation = select->generation; sel.status = select->status; sel.best = select->best;
    }
    energy_tail_kernel<<<blocks, kTailThreads, 0, s>>>(cta_partial, pl.chunks, p->n_candidates, P, valid, pair_acc, energy,
                                                       pg, reinterpret_cast<uint64_t*>(tail),
                                                       reinterpret_cast<unsigned int*>(tail + 8), sel);
    return launched();
}

}  // namespace
}  // namespace cl

extern "C" {

size_t cl_icrf_tables_bytes(const cl_icrf_problem* p) {
    if (!cl::problem_ok(p)) return 0;
    return (size_t)p->n_candidates * p->datapoints * 2 * sizeof(double);
}

int cl_icrf_curves(const cl_icrf_problem* p, const double* mean_icrf, const double* pca,
                   const double* params, double* curves, int32_t* valid, void* tables, void* stream) {
    using namespace cl;
    if (!problem_ok(p)) return CL_ERR_INVALID_ARGUMENT;
    CL_REQUIRE(pca && params && curves && valid && tables);
    CL_REQUIRE(mean_icrf || !p->use_mean_icrf);
    if (!aligned(tables, 16)) return CL_ERR_ALIGNMENT;
    if (p->datapoints > kMaxSharedDatapoints) {
        const size_t smem = wide_curve_smem(p->datapoints);
        cudaError_t e = cudaFuncSetAttribute(curves_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
        curves_wide_kernel<<<p->n_candidates * kWideCluster, kWideThreads, smem, (cudaStream_t)stream>>>(
            *p, mean_icrf, pca, params, curves, valid, reinterpret_cast<double*>(tables));
        return launched();
    }
    curves_kernel<<<p->n_candidates, 256, 0, (cudaStream_t)stream>>>(
        *p, mean_icrf, pca, params, curves, valid, reinterpret_cast<double*>(tables));
    return launched();
}

int cl_de_trial_curves(const cl_icrf_problem* p, const double* pop, int n_members, double dither_lo, double dither_hi,
                       double crossover, uint64_t seed, const int64_t* generation, const double* lower,
                       const double* upper, double* trial, double* params, const double* mean_icrf,
                       const double* pca, double* curves, int32_t* valid, void* tables, void* stream) {
    using namespace cl;
    if (!problem_ok(p)) return CL_ERR_INVALID_ARGUMENT;
    CL_REQUIRE(pop && generation && lower && upper && trial && params && pca && curves && valid && tables);
    CL_REQUIRE(mean_icrf || !p->use_mean_icrf);
    CL_REQUIRE(n_members >= 4 && n_members <= p->n_candidates);
    CL_REQUIRE(dither_lo <= dither_hi && crossover >= 0.0 && crossover <= 1.0);
    if (!aligned(tables, 16)) return CL_ERR_ALIGNMENT;
    const de::TrialConfig cfg{dither_lo, dither_hi, crossover, seed};
    if (p->datapoints > kMaxSharedDatapoints) {
        const size_t smem = wide_curve_smem(p->datapoints);
        cudaError_t e =
            cudaFuncSetAttribute(de_trial_curves_wide_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_status(e);
        de_trial_curves_wide_kernel<<<p->n_candidates * kWideCluster, kWideThreads, smem, (cudaStream_t)stream>>>(
            *p, pop, n_members, cfg, generation, lower, upper, trial, params, mean_icrf, pca, curves, valid,
            reinterpret_cast<double*>(tables));
        return launched();
    }
    de_trial_curves_kernel<<<p->n_candidates, 256, 0, (cudaStream_t)stream>>>(
        *p, pop, n_members, cfg, generation, lower, upper, trial, params, mean_icrf, pca, curves, valid,
        reinterpret_cast<double*>(tables));
    return launched();
}

size_t cl_icrf_energy_workspace_bytes(const cl_icrf_problem* p, int64_t n_pixels) {
    if (!cl::problem_ok(p) || n_pixels < 0) return 0;
    const cl::Plan pl = cl::make_plan(*p, n_pixels > 0 ? n_pixels : 1);
    return cl::partial_bytes(*p, pl) + 16;
}

int cl_icrf_energy_partial(const cl_icrf_problem* p, const void* tables, const uint8_t* dn,
                           const double* std, const double* exposure_s, int64_t n_pixels,
                           double* pair_acc, void* workspace, size_t workspace_bytes, void* stream) {
    return cl::energy_partial(p, cl::kMaxSharedDatapoints, tables, dn, std, exposure_s, n_pixels, pair_acc, workspace,
                              workspace_bytes, stream);
}

int cl_icrf_energy_partial_u16(const cl_icrf_problem* p, const void* tables, const uint16_t* dn,
                               const double* std, const double* exposure_s, int64_t n_pixels,
                               double* pair_acc, void* workspace, size_t workspace_bytes, void* stream) {
    return cl::energy_partial(p, cl::kMaxDatapoints, tables, dn, std, exposure_s, n_pixels, pair_acc, workspace,
                              workspace_bytes, stream);
}

int cl_icrf_energy_finalize(const cl_icrf_problem* p, const double* pair_acc, const int32_t* valid,
                            double* energy, void* stream) {
    using namespace cl;
    if (!problem_ok(p)) return CL_ERR_INVALID_ARGUMENT;
    CL_REQUIRE(pair_acc && valid && energy);
    finalize_kernel<<<(p->n_candidates + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        pair_acc, valid, p->n_candidates, n_pairs(p->n_exposures), energy);
    return launched();
}

size_t cl_icrf_exchange_bytes(const cl_icrf_problem* p, int world) {
    if (!cl::problem_ok(p) || world < 1 || world > CL_MAX_PEERS) return 0;
    const size_t per_rank = (size_t)p->n_candidates * cl::n_pairs(p->n_exposures) * 2 * sizeof(double);
    return 2 * (size_t)world * per_rank + (size_t)CL_MAX_PEERS * sizeof(uint64_t) + 64;   // slots, flags, seq + ticket
}

int cl_icrf_energy_population(const cl_icrf_problem* p, const void* tables, const uint8_t* dn, const double* std,
                              const double* exposure_s, int64_t n_pixels, const int32_t* valid, double* pair_acc,
                              double* energy, void* workspace, size_t workspace_bytes, const cl_peer_group* peers,
                              const cl_de_select_args* select, void* stream) {
    return cl::energy_population(p, cl::kMaxSharedDatapoints, tables, dn, std, exposure_s, n_pixels, valid, pair_acc,
                                 energy, workspace, workspace_bytes, peers, select, stream);
}

int cl_icrf_energy_population_u16(const cl_icrf_problem* p, const void* tables, const uint16_t* dn, const double* std,
                                  const double* exposure_s, int64_t n_pixels, const int32_t* valid, double* pair_acc,
                                  double* energy, void* workspace, size_t workspace_bytes, const cl_peer_group* peers,
                                  const cl_de_select_args* select, void* stream) {
    return cl::energy_population(p, cl::kMaxDatapoints, tables, dn, std, exposure_s, n_pixels, valid, pair_acc,
                                 energy, workspace, workspace_bytes, peers, select, stream);
}

// ---- peer-visible device buffers (CUDA IPC) for the exchange above ------------------------------------
int cl_peer_alloc(size_t bytes, void** dev_ptr, cl_ipc_handle* handle) {
    using namespace cl;
    CL_REQUIRE(dev_ptr && handle && bytes > 0);
    static_assert(sizeof(cudaIpcMemHandle_t) <= sizeof(cl_ipc_handle), "handle size");
    void* ptr = nullptr;
    cudaError_t e = cudaMalloc(&ptr, bytes);
    if (e != cudaSuccess) return cuda_status(e);
    e = cudaMemset(ptr, 0, bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, ptr);
    if (e != cudaSuccess) {
        cudaFree(ptr);
        return cuda_status(e);
    }
    memset(handle, 0, sizeof(*handle));
    memcpy(handle, &h, sizeof(h));
    *dev_ptr = ptr;
    return CL_OK;
}

int cl_peer_open(const cl_ipc_handle* handle, void** dev_ptr) {
    using namespace cl;
    CL_REQUIRE(handle && dev_ptr);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    return cuda_status(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
}

int cl_peer_close(void* dev_ptr) { return cl::cuda_status(cudaIpcCloseMemHandle(dev_ptr)); }

int cl_peer_free(void* dev_ptr) { return cl::cuda_status(cudaFree(dev_ptr)); }

}  // extern "C"
