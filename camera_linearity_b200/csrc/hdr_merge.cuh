// K2 shared definitions: kernel parameter block, per-exposure accumulation, median replace and
// the flat-field epilogue, used by every HDR-merge kernel.  The two-pass kernels run the same
// arithmetic in the same order, so their outputs are bit-identical; the single-pass kernels'
// expanded variance is checked against them (tests/test_gpu_hdr_merge.py).
#pragma once

#include "common.cuh"

namespace cl {

struct MergeParams {
    const void* dn[CL_MAX_EXPOSURES];
    const double* std[CL_MAX_EXPOSURES];
    const void* dark[CL_MAX_EXPOSURES];
    double inv_t[CL_MAX_EXPOSURES];          // 1 / exposure time
    uint32_t hot_dn[CL_MAX_EXPOSURES];       // smallest dark DN counted as a bad pixel
    int32_t n, H, W, C, bits, K;
    double max_dn;
    double kappa_scale;                      // -60 / max_dn : dw/w = kappa_scale*dn + 30
    const double* lut;
    const double* dlut;
    const double* std_lut;
    const void* flat;
    const double* flat_std;
    const double* flat_means;
    int32_t flat_bytes;
    int32_t any_dark;
    double* out_val;
    double* out_std;
    // tables in global memory (16-bit path): wt[bits], pb[bits][C] = {w*g, dlut}
    const double* g_wt;
    const double2* g_pb;
    // interleaved tables of the 16-bit kernel (hdr_merge_wide.cu): [bits][C] x {lut, dlut}
    const double2* g_tab32;
    // bad-pixel work list of the staged path (see hdr_merge_staged.cu): sample indices whose dark
    // frame exceeds the threshold in at least one exposure; hot_list[0] is the counter
    uint32_t* hot_list;
    uint32_t hot_cap;
    int32_t n_full_tiles;      // 512-pixel tiles handled by the staged kernel
    // per-tile bad-pixel patch buckets (staged path): counts [tile]{count, pad x3} sit right in front of
    // the hot-list header (one memset clears both), entries [tile][kBucketCap]{meta, pad, sigma}
    uint32_t* bucket_counts;
    uint32_t* bucket_entries;
    // exposures whose dark frame can flag a bad pixel (dark[k] set and hot_dn[k] <= max DN), in order
    int32_t n_dark;
    uint8_t dark_k[CL_MAX_EXPOSURES];
    int32_t stream_mode;       // a single-pass kernel runs and the fix-up pass applies its rule: 1 = uncertainty images
                               // (hdr_merge_stream.cu), 2 = STD table (hdr_merge_stream_lut.cu)
};

// single-pass kernel: a sample whose expanded variance q kept less than this fraction of its largest term A has
// cancelled by more than 6 digits and is recomputed with the exact two-pass formula; above it the expansion is within
// 1.1e-16 / kStreamCancel = 1.1e-10 of the two-pass result
constexpr double kStreamCancel = 1e-6;

constexpr size_t kHotListHeader = 4;   // uint32 entries reserved in front of the list (counter + pad)
constexpr int kStagedTilePx = 512;     // pixels per tile of the staged kernel
constexpr int kBucketCap = 32;         // patch entries per tile; more -> the sample goes to the fix-up list
constexpr int kBucketWords = 4 + 4 * kBucketCap;   // uint32 words per bucket in shared memory: count block + entries (528 bytes)
// entry meta word: pixel-in-tile [0,9) | channel [9,11) | exposure [11,16)

// One exposure's contribution for one sample.  With S = sum of weights and rS = 1/S:
//   val = rS * sum_k (w g) / t_k                                   exposure_series.py:388
//   std = rS * sqrt( sum_k ( (dw g + w dg - dw w g rS) dg / t_k )^2 )              :389,394
// where P1 = w*g and dgl = dlut[dn] come from the tables, dw = kappa*w, dg = dgl*sigma.
__device__ __forceinline__ void merge_accumulate(double w, double p1, double dgl, double kappa,
                                                 double sigma, double rS, double rt, double& acc_val,
                                                 double& acc_var) {
    const double a = kappa * p1;        // dw * g
    const double b = w * dgl;           // w * dICRF
    const double e = a * w;             // dw * w * g
    const double x = fma(b, sigma, a);  // dw*g + w*dg
    const double z = fma(-e, rS, x);
    const double y = (dgl * sigma) * rt;
    const double q = z * y;
    acc_var = fma(q, q, acc_var);
    acc_val = fma(p1, rt, acc_val);
}

// The same contribution when sigma comes from the camera's STD table (a function of the DN): the caller has
// tabulated  X = fma(w*dgl, sigma, kappa*p1)  and  Y0 = dgl*sigma  per DN with the operations above, what is left
// per exposure is below -- every intermediate is the bit pattern merge_accumulate() produces.
__device__ __forceinline__ void merge_accumulate_lut(double w, double p1, double X, double Y0, double kappa,
                                                     double rS, double rt, double& acc_val, double& acc_var) {
    const double a = kappa * p1;        // dw * g
    const double e = a * w;             // dw * w * g
    const double z = fma(-e, rS, X);
    const double y = Y0 * rt;
    const double q = z * y;
    acc_var = fma(q, q, acc_var);
    acc_val = fma(p1, rt, acc_val);
}

// Single-pass form (hdr_merge_stream.cu): the square expanded so that 1/S is a post-factor,
//   var = A - 2 B rS + C rS^2,  A = sum (x y)^2,  B = sum (x y)(e y),  C = sum (e y)^2,  x = dw g + w dg,  e = dw w g.
__device__ __forceinline__ void merge_accumulate_expanded(double w, double p1, double dgl, double kappa, double sigma,
                                                          double rt, double& S, double& acc_val, double& A, double& B,
                                                          double& C) {
    const double a = kappa * p1;        // dw * g
    const double e = a * w;             // dw * w * g
    const double u = dgl * sigma;       // dg
    const double x = fma(w, u, a);      // dw*g + w*dg
    const double y = u * rt;
    const double X = x * y, E = e * y;
    A = fma(X, X, A);
    B = fma(X, E, B);
    C = fma(E, E, C);
    acc_val = fma(p1, rt, acc_val);
    S += w;
}

// The single-pass form when sigma comes from the camera's STD table (hdr_merge_stream_lut.cu): x y = (x dg) / t and
// e y = (e dg) / t, and both products are functions of (dn, c) alone -- tabulated per DN by lut_products(), the
// exposure contributes two multiplies by 1/t and the five accumulations.
__device__ __forceinline__ void lut_products(double w, double p1, double dgl, double kappa, double sigma, double& xu,
                                             double& eu) {
    const double a = kappa * p1;        // dw * g
    const double e = a * w;             // dw * w * g
    const double u = dgl * sigma;       // dg
    const double x = fma(w, u, a);      // dw*g + w*dg
    xu = x * u;
    eu = e * u;
}
__device__ __forceinline__ void merge_accumulate_expanded_lut(double w, double p1, double xu, double eu, double rt,
                                                              double& S, double& acc_val, double& A, double& B,
                                                              double& C) {
    const double X = xu * rt, E = eu * rt;
    A = fma(X, X, A);
    B = fma(X, E, B);
    C = fma(E, E, C);
    acc_val = fma(p1, rt, acc_val);
    S += w;
}

// sum_k ((x - e rS) y)^2 from the expanded sums; rounding can leave a tiny negative where the true value is ~0
__device__ __forceinline__ double expanded_variance(double A, double B, double C, double rS) {
    const double q = fma(rS * rS, C, fma(-2.0 * rS, B, A));
    return q < 0.0 ? 0.0 : q;           // (NaN compares false and is kept)
}

__device__ __forceinline__ double kappa_of(uint32_t d, double kappa_scale) {
    return fma(u32_to_double(d), kappa_scale, 30.0);
}

template <typename DN>
__device__ __noinline__ uint32_t median_dn(const DN* __restrict__ img, int y, int x, int c, int H,
                                              int W, int C, int K) {
    uint32_t win[CL_MAX_MEDIAN_KERNEL * CL_MAX_MEDIAN_KERNEL];
    const int lo = K / 2;
    int m = 0;
    for (int dy = -lo; dy < K - lo; ++dy) {
        const int yy = reflect_index(y + dy, H);
        for (int dx = -lo; dx < K - lo; ++dx) {
            const int xx = reflect_index(x + dx, W);
            win[m++] = (uint32_t)img[((int64_t)yy * W + xx) * C + c];
        }
    }
    return select_rank(win, m, (K * K) / 2);
}

// Median of the uncertainty image; when there is no image the uncertainty of a neighbour is the
// STD-table value of ITS (unfiltered) DN (image_set.py:228-243, 365-385).
template <typename DN>
__device__ __noinline__ double median_std(const double* __restrict__ std_img,
                                             const DN* __restrict__ dn_img,
                                             const double* __restrict__ std_lut, int y, int x, int c,
                                             int H, int W, int C, int K) {
    double win[CL_MAX_MEDIAN_KERNEL * CL_MAX_MEDIAN_KERNEL];
    const int lo = K / 2;
    int m = 0;
    for (int dy = -lo; dy < K - lo; ++dy) {
        const int yy = reflect_index(y + dy, H);
        for (int dx = -lo; dx < K - lo; ++dx) {
            const int xx = reflect_index(x + dx, W);
            const int64_t j = ((int64_t)yy * W + xx) * C + c;
            win[m++] = std_img ? std_img[j] : std_lut[(int64_t)dn_img[j] * C + c];
        }
    }
    return select_rank(win, m, (K * K) / 2);
}

// 3 x 3 fast path (the reference's default kernel size): all 18 neighbourhood loads are issued
// together and the two medians come out of a 19-exchange selection network in registers --
// one memory round trip instead of two plus local-memory sorting.
template <typename T>
__device__ __forceinline__ void cswap(T& a, T& b) {
    const T lo = a < b ? a : b;
    const T hi = a < b ? b : a;
    a = lo;
    b = hi;
}
template <typename T>
__device__ __forceinline__ T median9(T (&v)[9]) {
    cswap(v[1], v[2]); cswap(v[4], v[5]); cswap(v[7], v[8]);
    cswap(v[0], v[1]); cswap(v[3], v[4]); cswap(v[6], v[7]);
    cswap(v[1], v[2]); cswap(v[4], v[5]); cswap(v[7], v[8]);
    cswap(v[0], v[3]); cswap(v[5], v[8]); cswap(v[4], v[7]);
    cswap(v[3], v[6]); cswap(v[1], v[4]); cswap(v[2], v[5]);
    cswap(v[4], v[7]); cswap(v[4], v[2]); cswap(v[6], v[4]);
    cswap(v[4], v[2]);
    return v[4];
}

template <typename DN>
__device__ __forceinline__ void median_pair(const DN* __restrict__ img, const double* __restrict__ std_img,
                                            const double* __restrict__ std_lut, int y, int x, int c, int H,
                                            int W, int C, int K, uint32_t& d_med, double& s_med) {
    if (K == 3) {
        uint32_t d[9];
        double s[9];
        int64_t idx[9];
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy) {
            const int yy = reflect_index(y + dy, H);
#pragma unroll
            for (int dx = -1; dx <= 1; ++dx)
                idx[(dy + 1) * 3 + dx + 1] = ((int64_t)yy * W + reflect_index(x + dx, W)) * C + c;
        }
#pragma unroll
        for (int i = 0; i < 9; ++i) d[i] = (uint32_t)img[idx[i]];
        if (std_img) {
#pragma unroll
            for (int i = 0; i < 9; ++i) s[i] = std_img[idx[i]];
        } else {
#pragma unroll
            for (int i = 0; i < 9; ++i) s[i] = std_lut[(int64_t)d[i] * C + c];
        }
        d_med = median9(d);
        s_med = median9(s);
    } else {
        d_med = median_dn(img, y, x, c, H, W, C, K);
        s_med = median_std(std_img, img, std_lut, y, x, c, H, W, C, K);
    }
}

// normalize_by_map, measurand.py:586-602, in variance form with rf = 1/flat:
//   val' = val*rf*m ;  std' = sqrt( var*(rf*m)^2 + (val*rf^2*fs*m)^2 + (val*rf*ms)^2 ),  var = std^2
// The reference's three quotients share the divisor, so one reciprocal serves all of them, and the
// merge kernels pass var = acc*rS^2 directly: one square root per sample instead of two.
__device__ __forceinline__ void flat_apply(double& val, double& sd_out, double var, double rf, double fs,
                                           double m, double ms) {
    const double vr = val * rf;            // val / flat
    const double k1 = rf * m;
    const double t2 = ((vr * rf) * fs) * m;
    const double t3 = vr * ms;
    sd_out = sqrt(fma(var, k1 * k1, fma(t2, t2, t3 * t3)));
    val = vr * m;
}

// flat_apply with sqrt()'s main path (common.cuh): same bits wherever the radicand is on it; returns false when the
// caller must have the sample recomputed (a zero radicand is selected and fine).
__device__ __forceinline__ bool flat_apply_main_path(double& val, double& sd_out, double var, double rf, double fs,
                                                     double m, double ms) {
    const double vr = val * rf;
    const double k1 = rf * m;
    const double t2 = ((vr * rf) * fs) * m;
    const double t3 = vr * ms;
    const double rad = fma(var, k1 * k1, fma(t2, t2, t3 * t3));
    bool ok;
    const double root = sqrt_main_path(rad, ok);
    sd_out = ok ? root : 0.0;
    val = vr * m;
    return ok || rad == 0.0;
}

// 1 / (dn / 255) for 8-bit flats, correctly rounded at compile time (identical to the two device
// divisions it replaces); dn = 0 -> +inf like IEEE division.
struct RecipTable {
    double v[256];
};
constexpr RecipTable make_recip255() {
    RecipTable t{};
    t.v[0] = __builtin_huge_val();
    for (int d = 1; d < 256; ++d) t.v[d] = 1.0 / (static_cast<double>(d) / 255.0);
    return t;
}
static __device__ const RecipTable kRecip255 = make_recip255();

__device__ __forceinline__ double flat_value(const void* flat, int flat_bytes, int64_t i,
                                             double max_dn) {
    if (flat_bytes == 8) return reinterpret_cast<const double*>(flat)[i];
    if (flat_bytes == 2) return __ddiv_rn((double)reinterpret_cast<const uint16_t*>(flat)[i], max_dn);
    return __ddiv_rn((double)reinterpret_cast<const uint8_t*>(flat)[i], max_dn);
}

// reciprocal of the flat value of sample i (the compile-time table is 1/(d/255): only for max_dn == 255, so
// that a uint8 flat next to a 16-bit stack is scaled by the same max_dn as flat_value / the ROI means)
__device__ __forceinline__ double flat_recip(const void* flat, int flat_bytes, int64_t i, double max_dn) {
    if (flat_bytes == 1 && max_dn == 255.0) return kRecip255.v[reinterpret_cast<const uint8_t*>(flat)[i]];
    return 1.0 / flat_value(flat, flat_bytes, i, max_dn);
}

// Full recomputation of one sample with the bad-pixel repair, same arithmetic (and the same
// table values, recomputed on the fly) as the streaming kernels -> bit-identical to inline repair.
template <typename DN>
__device__ __noinline__ void recompute_sample(const MergeParams& p, int64_t i) {
    const int C = p.C;
    const int c = (int)(i % C);
    const int64_t px = i / C;
    const int y = (int)(px / p.W), x = (int)(px - (int64_t)y * p.W);
    double S = 0.0;
    uint32_t hot = 0;
    for (int k = 0; k < p.n; ++k) {
        const DN* img = reinterpret_cast<const DN*>(p.dn[k]);
        uint32_t d = img[i];
        if (p.dark[k] && (uint32_t) reinterpret_cast<const DN*>(p.dark[k])[i] >= p.hot_dn[k]) {
            d = median_dn(img, y, x, c, p.H, p.W, C, p.K);
            hot |= 1u << k;
        }
        double w, dw;
        gaussian_weight(__ddiv_rn((double)d, p.max_dn), w, dw);
        S += w;
    }
    const double rS = 1.0 / S;
    double av = 0.0, as = 0.0;
    for (int k = 0; k < p.n; ++k) {
        const DN* img = reinterpret_cast<const DN*>(p.dn[k]);
        uint32_t d = img[i];
        double sg;
        if (hot & (1u << k)) {
            d = median_dn(img, y, x, c, p.H, p.W, C, p.K);
            sg = median_std(p.std[k], img, p.std_lut, y, x, c, p.H, p.W, C, p.K);
        } else {
            sg = p.std[k] ? p.std[k][i] : p.std_lut[(int64_t)d * C + c];
        }
        double w, dw;
        gaussian_weight(__ddiv_rn((double)d, p.max_dn), w, dw);
        const double p1 = w * p.lut[(int64_t)d * C + c];
        merge_accumulate(w, p1, p.dlut[(int64_t)d * C + c], kappa_of(d, p.kappa_scale), sg, rS, p.inv_t[k],
                         av, as);
    }
    double ov = av * rS, os;
    if (p.flat_bytes)
        flat_apply(ov, os, (as * rS) * rS, flat_recip(p.flat, p.flat_bytes, i, p.max_dn), p.flat_std[i],
                   p.flat_means[c], p.flat_means[C + c]);
    else
        os = sqrt(as) * rS;
    p.out_val[i] = ov;
    p.out_std[i] = os;
}

// One "try" per kernel family (the selection table is in hdr_merge.cu): CL_ERR_UNSUPPORTED when the kernel does not
// handle the stack, CL_ERR_WORKSPACE when only its part of the workspace is missing -- both before anything is
// enqueued -- otherwise the status of its launches.
int try_merge_wide(const MergeParams& p, cudaStream_t stream);         // hdr_merge_wide.cu
int try_merge_stream(const MergeParams& p, cudaStream_t stream);       // hdr_merge_stream.cu
int try_merge_stream_lut(const MergeParams& p, cudaStream_t stream);   // hdr_merge_stream_lut.cu
int try_merge_staged(const MergeParams& p, cudaStream_t stream);       // hdr_merge_staged.cu
int try_merge_staged_lut(const MergeParams& p, cudaStream_t stream);   // hdr_merge_staged_lut.cu
size_t wide_table_bytes(int bits, int C, bool with_std_lut);            // hdr_merge_wide.cu
// hdr_merge.cu
int launch_merge_generic_range(const MergeParams& p, int64_t first_item, cudaStream_t stream);
int launch_dark_scan(const MergeParams& p, cudaStream_t stream);
int launch_merge_fixup(const MergeParams& p, cudaStream_t stream);
int clear_hot_list(const MergeParams& p, cudaStream_t stream);

}  // namespace cl
