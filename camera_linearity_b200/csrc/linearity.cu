// Linearity analysis of one exposure pair (SURVEY.md 8f, rank 1): thresholds -> scaled difference
// -> per-channel statistics over the two spatial axes, fused.
// Replaces apply_thresholds (measurand.py:375-428), compute_difference (:620-655) and
// compute_dimension_statistics(axis=(0,1)) (:318-350) as ExposureSeries.process_linearity chains
// them (exposure_series.py:421-446): the reference materialises the absolute and relative
// difference images with their uncertainties (4 full float64 images per pair) and then reduces
// them; here ONE streaming pass over the four inputs (32 B/sample) produces the 6 x C numbers.
//
// Per channel and for the absolute and the relative difference the pass accumulates
//   weighted:   sum(w), sum(v*w) with w = 1/sigma   (np.nansum semantics: NaN terms are skipped
//               individually), sum(sigma), count(sigma) for the mean uncertainty;
//   unweighted: count, sum(v);
//   and, for the variance sum(w*(v-mean)^2), the SHIFTED moments T0 = sum(w), T1 = sum(w*d), T2 = sum(w*d^2)
//   with d = v - K over the samples the variance counts:  sum(w*(v-mean)^2) = T2 - 2(mean-K) T1 + (mean-K)^2 T0.
// K (per channel, abs and rel) is the plain mean of the samples the variance counts in the first of a few chunks of a
// few thousand samples (the image's first, then chunks spread over the image) that holds one -- every block derives
// it from the same L2-hot chunks in the same order, so it is one number and costs no launch; with K within a few
// standard errors of the mean the expansion loses nothing (round 1 made a second pass over the inputs, 64 B per
// sample, only to centre the variance).  Block partials are combined in a fixed order (deterministic); the
// reference's pairwise summation differs at the 1e-13 level.
#include <math.h>

#include "common.cuh"

namespace cl {
namespace {

constexpr int kThreads = 256;
constexpr int kBlocks = 296;  // 148 SMs x 2 resident CTAs; fixed (not sm_count) so the summation order is machine-independent
constexpr int kQ1 = 8;    // sums per channel: {sw, svw, ssig, nsig} x {abs, rel}
constexpr int kQ = 14;    // + the shifted moments {T0, T1, T2} x {abs, rel}
constexpr int kShiftSamples = 16;   // per thread: the provisional mean K comes from a chunk of 16 * lanes_used samples
constexpr int kShiftChunks = 8;     // chunks, at j/8 of the image, scanned for one the variance counts a sample of
                                    // before K falls back to 0: a channel with no such sample (thresholded away) costs
                                    // each thread 8 * 16 extra samples

struct PairArgs {
    const double* x_val;
    const double* x_std;
    const double* y_val;
    const double* y_std;
    double multiplier;
    double t2_multiplier;    // the m of the general routine's rcp * m: 1 when m = 0, so that sigma_y*x / (m*y*y) is +-inf
                             // there as in NumPy, not inf * 0 = NaN (the lean routine never runs with m = 0)
    double lower[CL_MAX_CHANNELS], upper[CL_MAX_CHANNELS];
    int has_thr;
    int64_t n;
    int C;
};

struct Diff {
    double a, r, sa, sr;     // absolute / relative difference and their uncertainties
    double wa, wr;           // 1/sa, 1/sr
    double qa, qr;           // sa^2, sr^2
    bool bad_v, bad_sa, bad_sr;   // the reference's value would be NaN here (thresholded or NaN input)
};

struct Raw {
    double x, y, xs, ys;
};

constexpr int kUnroll = 4;   // independent samples in flight per thread (the loads of all of them issue first)

__device__ __forceinline__ Raw load_raw(const PairArgs& p, int64_t i) {
    Raw r;
    r.x = __ldcs(p.x_val + i);
    r.y = __ldcs(p.y_val + i);
    r.xs = p.x_std ? __ldcs(p.x_std + i) : 0.0;
    r.ys = p.y_std ? __ldcs(p.y_std + i) : 0.0;
    return r;
}

__device__ __forceinline__ Diff difference(const PairArgs& p, const Raw& raw, double lo, double hi, bool use_std) {
    double x = raw.x, y = raw.y, xs = raw.xs, ys = raw.ys;
    // apply_thresholds (measurand.py:418-428) turns out-of-range values and their std into NaN.  NaN
    // samples would send every lane's rcp / rsqrt through its slow path, so the NaN-ness is carried in
    // flags (exactly where IEEE propagation would put it) and the arithmetic runs on 1.0 instead.
    const bool tx = p.has_thr && (x < lo || x > hi), ty = p.has_thr && (y < lo || y > hi);
    const bool nx = tx || x != x, ny = ty || y != y;
    const bool nxs = (tx && p.x_std) || xs != xs, nys = (ty && p.y_std) || ys != ys;
    x = nx ? 1.0 : x;  y = ny ? 1.0 : y;  xs = nxs ? 1.0 : xs;  ys = nys ? 1.0 : ys;
    Diff d;
    // One reciprocal and two reciprocal square roots replace the reference's five divisions and two
    // square roots (a/s = a*(1/s), 1/sqrt(q) = rsqrt(q), sqrt(q) = q*rsqrt(q)): each element moves by
    // <= 2 ulp, far inside the reduction's own reordering error, and the 0 / inf cases match.
    const double scale = __dmul_rn(p.multiplier, y);     // measurand.py:634-636
    const double inv = __drcp_rn(scale);
    d.a = __dsub_rn(x, scale);
    d.r = __dmul_rn(d.a, inv);
    d.bad_v = nx || ny;
    d.sa = d.sr = d.wa = d.wr = d.qa = d.qr = 0.0;
    d.bad_sa = d.bad_sr = false;
    if (use_std) {                                       // :652-653
        const double inf = __longlong_as_double(0x7ff0000000000000LL);
        const double my = __dmul_rn(p.multiplier, ys);
        const double qa = __dadd_rn(__dmul_rn(xs, xs), __dmul_rn(my, my));
        d.wa = rsqrt(qa);                                // weights = 1 / stds
        d.sa = (qa > 0.0 && qa < inf) ? __dmul_rn(qa, d.wa) : qa;
        const double t1 = __dmul_rn(xs, inv);
        const double t2 = __dmul_rn(__dmul_rn(__dmul_rn(ys, x), inv), __dmul_rn(inv, p.t2_multiplier));   // ys*x / (m*y*y)
        const double qr = __dadd_rn(__dmul_rn(t1, t1), __dmul_rn(t2, t2));
        d.wr = rsqrt(qr);
        d.sr = (qr > 0.0 && qr < inf) ? __dmul_rn(qr, d.wr) : qr;
        d.bad_sa = nxs || nys;
        d.bad_sr = nxs || nys || nx || ny;
        d.qa = qa;
        d.qr = qr;
    }
    return d;
}

__device__ __forceinline__ bool not_nan(double v) { return v == v; }

// np.nansum semantics: every term is skipped individually when it is NaN.
template <bool USE_STD>
__device__ __forceinline__ void accumulate1(double (&acc)[8], const Diff& d) {
    if (USE_STD) {
        const double va = __dmul_rn(d.a, d.wa), vr = __dmul_rn(d.r, d.wr);
        if (!d.bad_sa && not_nan(d.wa)) acc[0] += d.wa;
        if (!d.bad_sa && !d.bad_v && not_nan(va)) acc[1] += va;
        if (!d.bad_sa && not_nan(d.sa)) { acc[2] += d.sa; acc[3] += 1.0; }
        if (!d.bad_sr && not_nan(d.wr)) acc[4] += d.wr;
        if (!d.bad_sr && not_nan(vr)) acc[5] += vr;            // (bad_sr includes bad_v)
        if (!d.bad_sr && not_nan(d.sr)) { acc[6] += d.sr; acc[7] += 1.0; }
    } else {
        if (!d.bad_v && not_nan(d.a)) { acc[0] += 1.0; acc[1] += d.a; }
        if (!d.bad_v && not_nan(d.r)) { acc[4] += 1.0; acc[5] += d.r; }
    }
}

// shifted moments of the variance set (the samples round 1's second pass counted)
template <bool USE_STD>
__device__ __forceinline__ void accumulate_shifted(double (&acc)[kQ], const Diff& d, double ka, double kr) {
    const double da = __dsub_rn(d.a, ka), dr = __dsub_rn(d.r, kr);
    double wa = 1.0, wr = 1.0;
    bool bad_a = d.bad_v, bad_r = d.bad_v;
    if (USE_STD) {
        // An infinite value makes the weighted mean infinite (or NaN), and then its own term (inf - mean)^2 is NaN
        // in np.nansum: leaving it out keeps T0 the weight of the samples with finite values, which decides
        // whether the variance about an infinite mean is inf or 0.  With a finite mean no such sample exists.
        const double inf = __longlong_as_double(0x7ff0000000000000LL);
        wa = d.wa;
        wr = d.wr;
        bad_a = bad_a || d.bad_sa || !(fabs(d.a) < inf);
        bad_r = d.bad_sr || !(fabs(d.r) < inf);
    }
    const double ta = __dmul_rn(wa, __dmul_rn(da, da)), tr = __dmul_rn(wr, __dmul_rn(dr, dr));
    if (!bad_a && not_nan(ta)) { acc[8] += wa; acc[9] = fma(wa, da, acc[9]); acc[10] += ta; }
    if (!bad_r && not_nan(tr)) { acc[11] += wr; acc[12] = fma(wr, dr, acc[12]); acc[13] += tr; }
}

// ---------------------------------------------------------------------------------------------------------
// Lean per-sample routine (both uncertainty images present).  The general routine above spends ~210
// instructions per sample, two thirds of them on bookkeeping: every one of the 14 sums carries its own "is this
// term NaN" predicate (a compare and two selects each) because np.nansum skips terms individually.  But a sample
// is almost always in one of two states: ORDINARY (nothing thresholded, nothing NaN, every term finite) -- all
// 14 terms count -- or DROPPED (value and uncertainty of one side thresholded: every term is skipped).  So:
//   * the arithmetic runs once, without per-term checks (dropped samples compute on 1.0 so it stays finite);
//   * ONE predicate zeroes the sample's four weights / uncertainties and its count (9 selects), and the 14 sums
//     are updated unconditionally -- a dropped sample adds exact zeros;
//   * a sample in any other state (a NaN in only the value or only the uncertainty image, a zero / denormal /
//     infinite variance, an infinite ratio) adds zeros here and goes through the general routine instead.
// Ordinary samples execute the same operations in the same order as the general routine: the statistics are
// bit-identical to the all-general kernel (CL_PAIR_GENERAL_ONLY builds it for the A/B).
// (normal_positive, rsqrt_main_path, rcp_main_path: common.cuh)
__device__ __forceinline__ bool lean_sample(const PairArgs& p, const Raw& raw, double lo, double hi, double ka,
                                            double kr, double (&acc)[kQ]) {
    double x = raw.x, y = raw.y, xs = raw.xs, ys = raw.ys;
    const bool tx = p.has_thr && (x < lo || x > hi), ty = p.has_thr && (y < lo || y > hi);
    const bool bad_v = tx || ty || x != x || y != y;               // the reference's value is NaN
    const bool bad_s = tx || ty || xs != xs || ys != ys;           // ... its uncertainty is NaN
    const bool any_bad = bad_v || bad_s;
    x = any_bad ? 1.0 : x;  y = any_bad ? 1.0 : y;  xs = any_bad ? 1.0 : xs;  ys = any_bad ? 1.0 : ys;
    const double scale = __dmul_rn(p.multiplier, y);
    bool rcp_ok;
    const double inv = rcp_main_path(scale, rcp_ok);
    double a = __dsub_rn(x, scale);
    double r = __dmul_rn(a, inv);
    const double my = __dmul_rn(p.multiplier, ys);
    const double qa = __dadd_rn(__dmul_rn(xs, xs), __dmul_rn(my, my));
    double wa = rsqrt_main_path(qa);
    double sa = __dmul_rn(qa, wa);
    const double t1 = __dmul_rn(xs, inv);
    const double t2 = __dmul_rn(__dmul_rn(__dmul_rn(ys, x), inv), __dmul_rn(inv, p.multiplier));
    const double qr = __dadd_rn(__dmul_rn(t1, t1), __dmul_rn(t2, t2));
    double wr = rsqrt_main_path(qr);
    double sr = __dmul_rn(qr, wr);
    const bool ordinary = !any_bad && rcp_ok && normal_positive(qa) && normal_positive(qr) &&
                          fabs(r) < __longlong_as_double(0x7ff0000000000000LL);
    const bool dropped = bad_v && bad_s;
    // everything a non-ordinary sample computed may be garbage (NaN, inf): selects, not multiplications by zero
    a = ordinary ? a : 0.0;    r = ordinary ? r : 0.0;
    wa = ordinary ? wa : 0.0;  wr = ordinary ? wr : 0.0;
    sa = ordinary ? sa : 0.0;  sr = ordinary ? sr : 0.0;
    const double one = ordinary ? 1.0 : 0.0;
    const double da = __dsub_rn(a, ka), dr = __dsub_rn(r, kr);
    acc[0] += wa;
    acc[1] += __dmul_rn(a, wa);
    acc[2] += sa;
    acc[3] += one;
    acc[4] += wr;
    acc[5] += __dmul_rn(r, wr);
    acc[6] += sr;
    acc[7] += one;
    acc[8] += wa;
    acc[9] = fma(wa, da, acc[9]);
    acc[10] += __dmul_rn(wa, __dmul_rn(da, da));
    acc[11] += wr;
    acc[12] = fma(wr, dr, acc[12]);
    acc[13] += __dmul_rn(wr, __dmul_rn(dr, dr));
    return !(ordinary || dropped);                                 // true: the general routine must count this sample
}

template <bool USE_STD, bool LEAN>
__device__ __forceinline__ void count_sample(const PairArgs& p, const Raw& raw, double lo, double hi, double ka,
                                             double kr, double (&acc)[kQ]) {
    if (LEAN) {
        if (!lean_sample(p, raw, lo, hi, ka, kr, acc)) return;
    }
    const Diff d = difference(p, raw, lo, hi, USE_STD);
    double (&a8)[8] = reinterpret_cast<double (&)[8]>(acc);
    accumulate1<USE_STD>(a8, d);
    accumulate_shifted<USE_STD>(acc, d, ka, kr);
}

// Deterministic block reduction of per-thread accumulators: thread t owns channel (t % C) because
// the grid stride is a multiple of C.  acc -> shared [Q][kThreads]; then Q*C threads sum their
// column in index order.
template <int Q>
__device__ __forceinline__ void block_reduce(const double (&acc)[Q], int C, int lanes_used, double* out) {
    __shared__ double sh[Q][kThreads];
#pragma unroll
    for (int q = 0; q < Q; ++q) sh[q][threadIdx.x] = acc[q];
    __syncthreads();
    if (threadIdx.x < Q * C) {
        const int q = threadIdx.x / C, c = threadIdx.x % C;
        double s = 0.0;
        for (int t = c; t < lanes_used; t += C) s += sh[q][t];
        out[q * C + c] = s;
    }
    __syncthreads();
}

__device__ __forceinline__ double ka_of(const double (&shift)[4][CL_MAX_CHANNELS], int c) {
    return shift[1][c] > 0.0 ? shift[0][c] / shift[1][c] : 0.0;
}
__device__ __forceinline__ double kr_of(const double (&shift)[4][CL_MAX_CHANNELS], int c) {
    return shift[3][c] > 0.0 ? shift[2][c] / shift[3][c] : 0.0;
}

template <bool USE_STD, bool LEAN>
__global__ void __launch_bounds__(kThreads, 2)
pair_stats_kernel(const PairArgs p, double* __restrict__ partial /* [blocks][kQ][C] */) {
    const int C = p.C;
    const int lanes_used = (kThreads / C) * C;               // threads beyond that idle: keeps t % C fixed
    const int64_t stride = (int64_t)gridDim.x * lanes_used;
    __shared__ double shift[4][CL_MAX_CHANNELS];             // {sum a, count a, sum r, count r} -> K
    double acc[kQ];
#pragma unroll
    for (int q = 0; q < kQ; ++q) acc[q] = 0.0;
    const bool active = (int)threadIdx.x < lanes_used;
    const int c = threadIdx.x % C;                           // (block offset and stride are multiples of C)
    const double lo = p.lower[c], hi = p.upper[c];
    // ---- provisional means K (identical in every block) ----
    // K is the plain mean of the samples the variance counts -- a finite value and, with uncertainty images, a finite
    // positive weight -- in the first chunk of kShiftSamples * lanes_used samples that holds one, found separately
    // per channel and for the absolute and the relative difference.  Chunk j starts at j/kShiftChunks of the image
    // (rounded down to a multiple of lanes_used, so thread t keeps channel t % C): dark or saturated top rows do not
    // hide the rest of the image.  Every block scans the same chunks in the same order; a channel none of them
    // counts a sample of keeps K = 0.
    {
        const double inf = __longlong_as_double(0x7ff0000000000000LL);
        __shared__ double sh4[4][kThreads];
        if (threadIdx.x < 4 * CL_MAX_CHANNELS) shift[threadIdx.x / CL_MAX_CHANNELS][threadIdx.x % CL_MAX_CHANNELS] = 0.0;
        for (int chunk = 0; chunk < kShiftChunks; ++chunk) {
            const int64_t base = chunk * (p.n / kShiftChunks) / lanes_used * lanes_used;
            if (base >= p.n) break;
            double pa[4] = {0, 0, 0, 0};
            if (active) {
                for (int u = 0; u < kShiftSamples; ++u) {
                    const int64_t i = base + (int64_t)u * lanes_used + threadIdx.x;
                    if (i >= p.n) break;
                    const Diff d = difference(p, load_raw(p, i), lo, hi, USE_STD);
                    bool fa = !d.bad_v && fabs(d.a) < inf, fr = !d.bad_v && fabs(d.r) < inf;
                    if (USE_STD) {                       // the weight 1/sqrt(q) is finite and positive
                        fa = fa && !d.bad_sa && d.qa > 0.0 && d.qa < inf;
                        fr = fr && !d.bad_sr && d.qr > 0.0 && d.qr < inf;
                    }
                    if (fa) { pa[0] += d.a; pa[1] += 1.0; }
                    if (fr) { pa[2] += d.r; pa[3] += 1.0; }
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) sh4[q][threadIdx.x] = pa[q];
            __syncthreads();
            bool pending = false;
            if (threadIdx.x < 2 * C) {                       // (which, channel): the first chunk with a count wins
                const int q = 2 * (threadIdx.x / C), cc = threadIdx.x % C;
                double s = 0.0, k = 0.0;
                for (int l = cc; l < lanes_used; l += C) { s += sh4[q][l]; k += sh4[q + 1][l]; }
                if (shift[q + 1][cc] == 0.0) { shift[q][cc] = s; shift[q + 1][cc] = k; }
                pending = shift[q + 1][cc] == 0.0;
            }
            if (!__syncthreads_or(pending)) break;
        }
        __syncthreads();
    }
    const double ka = ka_of(shift, c), kr = kr_of(shift, c);
    if (active) {
        int64_t i = (int64_t)blockIdx.x * lanes_used + threadIdx.x;
        for (; i + (kUnroll - 1) * stride < p.n; i += kUnroll * stride) {
            Raw raw[kUnroll];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) raw[u] = load_raw(p, i + u * stride);
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) count_sample<USE_STD, LEAN>(p, raw[u], lo, hi, ka, kr, acc);
        }
        for (; i < p.n; i += stride) count_sample<USE_STD, LEAN>(p, load_raw(p, i), lo, hi, ka, kr, acc);
    }
    block_reduce<kQ>(acc, C, lanes_used, partial + (int64_t)blockIdx.x * kQ * C);
    if (blockIdx.x == 0 && threadIdx.x < 2 * C)              // the shifts, for the final kernel
        partial[(int64_t)gridDim.x * kQ * C + threadIdx.x] = threadIdx.x < C ? ka_of(shift, threadIdx.x) : kr_of(shift, threadIdx.x - C);
}

// Fixed-order sum of one column of the per-block partials by one warp: lanes stride over the blocks, then
// an xor tree (deterministic; a single thread walking 444 dependent loads took 40 us).
__device__ __forceinline__ double column_sum(const double* __restrict__ partial, int n_blocks, int row_len, int col) {
    const int lane = threadIdx.x & 31;
    double s = 0.0;
#pragma unroll 4
    for (int b = lane; b < n_blocks; b += 32) s += partial[(int64_t)b * row_len + col];
    return warp_sum(s);
}

// stats[which][k][c]: which 0 = absolute, 1 = relative; k 0 = mean, 1 = std, 2 = error.  One block: a warp per
// column total, then one thread per (which, c).
__global__ void pair_final_kernel(const double* __restrict__ partial, int n_blocks, int C, int use_std,
                                  double* __restrict__ stats) {
    __shared__ double totals[kQ * CL_MAX_CHANNELS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int o = warp; o < kQ * C; o += (int)(blockDim.x >> 5)) {
        const double s = column_sum(partial, n_blocks, kQ * C, o);
        if (lane == 0) totals[o] = s;
    }
    __syncthreads();
    const int t = threadIdx.x;
    if (t >= 2 * C) return;
    const int which = t / C, c = t % C;
    const double K = partial[(int64_t)n_blocks * kQ * C + t];
    const double denom = totals[(which * 4 + 0) * C + c];                     // sum of weights / count
    const double mean = totals[(which * 4 + 1) * C + c] / denom;
    const double T0 = totals[(8 + which * 3 + 0) * C + c], T1 = totals[(8 + which * 3 + 1) * C + c],
                 T2 = totals[(8 + which * 3 + 2) * C + c];
    const double dm = mean - K;
    double q = fma(dm * dm, T0, fma(-2.0 * dm, T1, T2));                      // sum w (v - mean)^2
    if (q < 0.0) q = 0.0;
    // degenerate means, as np.nansum sees them: (v - NaN)^2 is NaN for every sample -> an empty sum; (v - inf)^2 is
    // inf for every finite v and NaN for v = inf, and T0 is the weight of the samples with finite values.  Without
    // uncertainty images np.nanstd's plain sum keeps the NaN of inf - inf or of a NaN mean: the std is NaN.  (This
    // takes the infinity to come from an infinite sample.  A mean that overflows from finite values, |v| ~ 1e305,
    // gives NaN here where np.nanstd gives inf; the sums cannot tell the two apart.)
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    if (mean != mean) q = 0.0;
    else if (fabs(mean) == inf) q = T0 > 0.0 ? inf : 0.0;
    if (!use_std && !(fabs(mean) < inf)) q = __longlong_as_double(0x7ff8000000000000LL);
    stats[(which * 3 + 0) * C + c] = mean;
    stats[(which * 3 + 1) * C + c] = sqrt(q / denom);
    stats[(which * 3 + 2) * C + c] = use_std ? totals[(which * 4 + 2) * C + c] / totals[(which * 4 + 3) * C + c]
                                             : __longlong_as_double(0x7ff8000000000000LL);
}

}  // namespace
}  // namespace cl

extern "C" {

size_t cl_pair_statistics_workspace_bytes(int channels) {
    const size_t c = channels > 0 ? channels : 1;
    return ((size_t)cl::kBlocks * cl::kQ * c + 2 * c) * sizeof(double);     // block partials + the two shifts per channel
}

int cl_pair_statistics(const double* x_val, const double* x_std, const double* y_val, const double* y_std,
                       double multiplier, const double* lower, const double* upper, int64_t n_samples,
                       int channels, double* stats, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace cl;
    CL_REQUIRE(n_samples >= 0 && channels >= 1 && channels <= CL_MAX_CHANNELS);
    CL_REQUIRE(x_val && y_val && stats);
    CL_REQUIRE(n_samples % channels == 0);
    CL_REQUIRE((lower == nullptr) == (upper == nullptr));
    if (!workspace || workspace_bytes < cl_pair_statistics_workspace_bytes(channels)) return CL_ERR_WORKSPACE;
    PairArgs p;
    p.x_val = x_val; p.x_std = x_std; p.y_val = y_val; p.y_std = y_std;
    p.multiplier = multiplier; p.n = n_samples; p.C = channels;
    p.t2_multiplier = multiplier == 0.0 ? 1.0 : multiplier;
    p.has_thr = lower != nullptr;
    for (int c = 0; c < CL_MAX_CHANNELS; ++c) {      // HOST arrays of per-channel limits
        p.lower[c] = (lower && c < channels) ? lower[c] : 0.0;
        p.upper[c] = (upper && c < channels) ? upper[c] : 0.0;
    }
    const bool use_std = x_std != nullptr || y_std != nullptr;
    cudaStream_t s = (cudaStream_t)stream;
    double* partial = reinterpret_cast<double*>(workspace);
    // the lean routine needs both uncertainty images and a multiplier whose products stay finite on 1.0
    bool lean = x_std && y_std && multiplier == multiplier && fabs(multiplier) >= 1e-100 && fabs(multiplier) <= 1e100;
#ifdef CL_PAIR_GENERAL_ONLY
    lean = false;
#endif
    if (lean) pair_stats_kernel<true, true><<<kBlocks, kThreads, 0, s>>>(p, partial);
    else if (use_std) pair_stats_kernel<true, false><<<kBlocks, kThreads, 0, s>>>(p, partial);
    else pair_stats_kernel<false, false><<<kBlocks, kThreads, 0, s>>>(p, partial);
    int st = launched();
    if (st != CL_OK) return st;
    pair_final_kernel<<<1, 1024, 0, s>>>(partial, kBlocks, channels, use_std ? 1 : 0, stats);
    return launched();
}

}  // extern "C"
