/*
 * camera_linearity_b200 -- C ABI of the B200 (sm_100a) imaging hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference
 * (samivout/camera_linearity) has no FFI: its "plugin API" is the AbstractMeasurand
 * backend contract (modules/measurand.py:26-32, 684-714).  Every entry point below replaces
 * the NumPy/CuPy body of one reference method; the file:line it replaces is cited on the
 * declaration.  INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.
 *   - All image pointers are DEVICE pointers to C-contiguous, channel-interleaved (H, W, C)
 *     arrays ("samples" = H*W*C elements), unless a parameter says HOST.
 *   - Nothing here allocates device memory, synchronises the device or keeps global state.
 *     Scratch space is caller-provided (cl_*_workspace_bytes tells how much).  Work is
 *     enqueued on `stream` (a cudaStream_t passed as void*; NULL = the legacy default stream).
 *   - Return value: CL_OK (0) or a negative cl_status.  cl_status_string() names it.
 *   - Integer results (LUT bins, masks, uint8 means, valid-sample counts) are bit-exact with
 *     the reference NumPy path; float64 results agree to <= 1e-6 relative (typically ~1e-15).
 */
#ifndef CAMERA_LINEARITY_B200_H
#define CAMERA_LINEARITY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CL_ABI_VERSION 1
#define CL_MAX_EXPOSURES 32   /* exposures per cl_hdr_merge call   */
#define CL_MAX_CHANNELS 8     /* channels (last image dimension)    */
#define CL_MAX_MEDIAN_KERNEL 7
#define CL_MAX_PAIR_EXPOSURES 8 /* exposures per calibration stack (28 pairs) */

typedef enum cl_status {
    CL_OK = 0,
    CL_ERR_INVALID_ARGUMENT = -1, /* NULL pointer, non-positive size, bad enum        */
    CL_ERR_UNSUPPORTED = -2,      /* valid request outside the implemented envelope   */
    CL_ERR_WORKSPACE = -3,        /* workspace missing or too small                   */
    CL_ERR_ALIGNMENT = -4,        /* pointer not aligned to the element size          */
    CL_ERR_CUDA = -100            /* -(100 + cudaError_t) : CUDA runtime failure      */
} cl_status;

int cl_abi_version(void);
const char* cl_status_string(int status);
/* Number of kernel launches enqueued by this library in this process (for bench accounting). */
uint64_t cl_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * K1  ICRF linearisation -- replaces AbstractMeasurand.linearize / _linearize_channel /
 *     _linearize_single (modules/measurand.py:471-541), called from ImageSet.linearize
 *     (image_set.py:102-115), ExposureSeries.linearize (exposure_series.py:226-250) and
 *     ImageSet.calculate_numerical_STD (image_set.py:365-385, the table passed as `lut`).
 *
 *   out_val[i] = lut[bin(i) * C + (i % C)]
 *   out_std[i] = dlut[bin(i) * C + (i % C)] * std_in[i]        (only if all three are non-NULL)
 *
 *   cl_linearize_dn : bin(i) = dn[i]; dn_bytes = 1 (uint8) or 2 (uint16).  Bins >= bits are an
 *                     error the caller must rule out (NumPy would raise IndexError).
 *   cl_linearize_f64: bin(i) = wrap(rint(val[i] * max_dn)) -- round-half-even then the wrapping
 *                     cast of measurand.py:503,531 (to uint8 when bits <= 256, else uint16).
 *   bin_out (nullable) receives the bins as uint16 for bit-exactness checks.
 * ------------------------------------------------------------------------------------------- */
int cl_linearize_dn(const void* dn, int dn_bytes, const double* std_in, const double* lut,
                    const double* dlut, double* out_val, double* out_std, int64_t n_samples,
                    int channels, int bits, void* stream);
int cl_linearize_f64(const double* val, double max_dn, const double* std_in, const double* lut,
                     const double* dlut, double* out_val, double* out_std, uint16_t* bin_out,
                     int64_t n_samples, int channels, int bits, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2  Fused weighted HDR merge -- replaces ExposureSeries._precalculate_sum_of_weights
 *     (exposure_series.py:317-345), _compute_HDR_image_set (:347-397) and the Measurand methods
 *     they call per exposure: apply_gaussian_weight (measurand.py:606-618), linearize (:471-541),
 *     filter_larger_than_by_map (:543-557, via ImageSet.bad_pixel_filter image_set.py:387-400),
 *     and the normalize_by_map epilogue (:559-604, via ImageSet.flat_field_correction
 *     image_set.py:402-421).  One launch streams every input byte once.
 *
 *   For each sample, with v_k = dn_k / max_dn, w = e^(-30 (v-0.5)^2), dw = -60 (v-0.5) w,
 *   g = lut[dn_k], dg = dlut[dn_k] * std_k, S = sum_k w_k:
 *     val = sum_k (w g) / (S t_k)
 *     std = sqrt( sum_k ( ((dw g + w dg)/S - (dw w g)/S^2) * dg / t_k )^2 )
 *   Bad pixels: where dark_k * dark_scale_k / max_dn > dark_threshold, dn_k and std_k are first
 *   replaced by their K x K per-channel median (scipy 'reflect' boundary, rank K*K/2).
 *   Flat field (optional): val' = val/flat*m,  std' per measurand.py:586-599, with the ROI means
 *   m[c], ms[c] in flat_means[0..C) and [C..2C) (see cl_flat_roi_means).
 * ------------------------------------------------------------------------------------------- */
typedef struct cl_hdr_merge_args {
    int32_t n_exposures;          /* 1..CL_MAX_EXPOSURES                                    */
    int32_t height, width, channels;
    int32_t dn_bytes;             /* 1 = uint8 images, 2 = uint16                           */
    int32_t bits;                 /* LUT rows: 256 or 65536                                 */
    const void* const* dn;        /* HOST array [n] of device pointers, (H,W,C) dn_bytes    */
    const double* const* std;     /* HOST array [n] of device pointers, (H,W,C) f64; an
                                     entry (or the array) may be NULL when std_lut is given  */
    const double* exposure_s;     /* HOST array [n], seconds                                */
    const double* lut;            /* device [bits][C]  ICRF                                 */
    const double* dlut;           /* device [bits][C]  ICRF derivative                      */
    const double* std_lut;        /* device [bits][C] or NULL: std_k = std_lut[dn_k]
                                     (image_set.py:365-385) where std[k] is NULL            */
    const void* const* dark;      /* HOST array [n] of device pointers or NULL; entry NULL =
                                     no dark frame for that exposure (image_set.py:157-198)  */
    const double* dark_scale;     /* HOST array [n] or NULL (= 1.0): target_t / dark_t      */
    double dark_threshold;        /* gs.DARK_THRESHOLD as used by measurand.py:545           */
    int32_t median_kernel;        /* gs.MEDIAN_FILTER_KERNEL_SIZE, 1..CL_MAX_MEDIAN_KERNEL   */
    int32_t flat_bytes;           /* 0 = no flat; 1/2 = integer DN (val = dn/max_dn); 8 = f64 */
    const void* flat;             /* device (H,W,C)                                         */
    const double* flat_std;       /* device (H,W,C) f64                                     */
    const double* flat_means;     /* device [2C]: ROI mean of flat value, then of flat std  */
    double* out_val;              /* device (H,W,C) f64                                     */
    double* out_std;              /* device (H,W,C) f64                                     */
    int32_t algo;                 /* 0 = auto, 1 = generic register kernel,
                                     2 = bulk-copy staged two-pass kernel (uint8, C = 3 / 1; with std_lut
                                         and no uncertainty images: its STD-table variant),
                                     3 = fused-table kernel (uint16, N <= 16; software-pipelined, bit-identical to the
                                         generic kernel) -- what auto picks for uint16 stacks,
                                     4 = single-pass streaming kernels (uint8, C = 3 / 1, N >= 2, either
                                         uncertainty images for every exposure or std_lut and none;
                                         expanded variance, <= 1e-9 from the others) -- what auto picks
                                         whenever it applies                                   */
    int32_t reserved;
} cl_hdr_merge_args;

size_t cl_hdr_merge_workspace_bytes(const cl_hdr_merge_args* args);
int cl_hdr_merge(const cl_hdr_merge_args* args, void* workspace, size_t workspace_bytes,
                 void* stream);

/* ROI means for the flat-field epilogue -- flat_field_mean() inside normalize_by_map
 * (measurand.py:561-583).  Rows [r0, r1) x cols [c0, c1), clamped like a NumPy slice.
 * out_means[0..C) = mean of the flat value (dn / max_dn for integer flats), [C..2C) = mean of
 * flat_std.  Deterministic two-stage reduction. */
size_t cl_flat_roi_means_workspace_bytes(int height, int width, int channels);
int cl_flat_roi_means(const void* flat, int flat_bytes, double max_dn, const double* flat_std,
                      int height, int width, int channels, int r0, int r1, int c0, int c1,
                      double* out_means, void* workspace, size_t workspace_bytes, void* stream);

/* Stand-alone Measurand methods (same formulae as inside cl_hdr_merge). */
/* apply_gaussian_weight, measurand.py:606-618 */
int cl_gaussian_weight(const double* val, double* w, double* dw, int64_t n_samples, void* stream);
/* filter_larger_than_by_map, measurand.py:543-557 (+ repairs R5/R6): float64 images */
int cl_bad_pixel_filter(const double* val, const double* std, const double* dark_val,
                        double threshold, int kernel, int height, int width, int channels,
                        double* out_val, double* out_std, void* stream);
/* normalize_by_map, measurand.py:559-604 (+ repair R7) */
int cl_flat_field_normalize(const double* val, const double* std, const double* flat_val,
                            const double* flat_std, const double* flat_means, int64_t n_samples,
                            int channels, double* out_val, double* out_std, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K3  Welford mean / standard-error frames -- replaces welford_algorithm
 *     (modules/video_processing.py:161-219).
 *
 *   Streaming form (bit-identical float64 state to the reference's sequential recurrence,
 *   video_processing.py:205-208, no FMA contraction):
 *     cl_welford_update   : folds F frames [F][n_samples] uint8 into (mean, m2), starting at
 *                           frame number count0 + 1.  lut (nullable, [256][C]) linearises each
 *                           frame first (video_processing.py:200-201, repair R9).
 *     cl_welford_finalize : sem = sqrt(m2/(n-1))/sqrt(n), mean_u8 = uint8(rint(mean*255)).
 *   Stack form (all F frames resident): exact integer accumulation of sum(d), sum(d^2) with
 *   warp-shuffle reduction across frame slices, and an exact replay of the reference recurrence
 *   for the samples whose mean*255 is a rounding tie -- uint8 mean stays bit-exact, float64
 *   mean/sem agree to ~1e-13.  lut != NULL selects float64 accumulation of the LUT values.
 * ------------------------------------------------------------------------------------------- */
int cl_welford_update(const uint8_t* frames, int n_frames, int64_t n_samples, int channels,
                      const double* lut, double max_dn, double* mean, double* m2,
                      int64_t count0, void* stream);
int cl_welford_finalize(const double* mean, const double* m2, int64_t count, int64_t n_samples,
                        double max_dn, double* sem, uint8_t* mean_u8, void* stream);
size_t cl_welford_stack_workspace_bytes(int n_frames, int64_t n_samples);
int cl_welford_stack(const uint8_t* frames, int n_frames, int64_t n_samples, int channels,
                     const double* lut, double max_dn, double* mean, double* sem,
                     uint8_t* mean_u8, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K4  ICRF calibration objective for a whole differential-evolution population -- replaces
 *     _inverse_camera_response_function (modules/ICRF_calibration_exposure.py:20-44),
 *     _energy_function (:148-201), analyze_linearity (:66-145) and gf.nanaverage
 *     (general_functions.py:149-176).
 *
 *   cl_icrf_curves         : per candidate s: curve = mean (+) pca @ params[s]; curve += 1 -
 *                            curve[D-1]; curve[0] = 0; gates (:174-180) -> valid[s]; writes the
 *                            masked value table and its reciprocal used by the partial kernel.
 *   cl_icrf_energy_partial : pair_acc[s][pair][0..1] = per-(candidate, exposure pair) numerator
 *                            and denominator summed over this call's pixels (no std: sum |d| and
 *                            the valid count; std: sum |d|/sigma and sum 1/sigma).  Multi-GPU:
 *                            each rank calls it on its pixel shard, then all-reduces pair_acc.
 *   cl_icrf_energy_finalize: energy[s] = nanmean over pairs of num/den, NaN or gated -> +inf.
 *   Candidates are padded by the caller to a multiple of 32 (one lane per candidate).
 * ------------------------------------------------------------------------------------------- */
typedef struct cl_icrf_problem {
    int32_t n_candidates;   /* S, multiple of 32                                            */
    int32_t n_params;       /* 5 (use_mean_icrf) or 6 (exponent + 5), any >= 1              */
    int32_t datapoints;     /* D = curve length = LUT rows (<= 256 for uint8 samples,        */
                            /* <= 65536 for uint16 samples: the _u16 entry points)           */
    int32_t use_mean_icrf;  /* 1: mean + pca @ p ; 0: linspace(0,1,D)**p[0] + pca @ p[1:]   */
    int32_t lower, upper;   /* data limits as DN indices (ICRF_calibration_exposure.py:182) */
    int32_t n_exposures;    /* N, 2..CL_MAX_PAIR_EXPOSURES                                  */
    int32_t use_std;
} cl_icrf_problem;

/* cl_icrf_tables_bytes, cl_icrf_curves, cl_icrf_energy_workspace_bytes, cl_icrf_energy_finalize, cl_icrf_exchange_bytes
 * and cl_de_trial_curves accept 2 <= D <= 65536 (D > 256: one thread-block cluster per candidate builds the curve);
 * the uint8 partial / population calls accept D <= 256, their _u16 forms D <= 65536. */
size_t cl_icrf_tables_bytes(const cl_icrf_problem* p);   /* size of the `tables` scratch: 2 * S * D * 8 bytes */
int cl_icrf_curves(const cl_icrf_problem* p, const double* mean_icrf, const double* pca,
                   const double* params /* device [S][n_params] */, double* curves /* [S][D] */,
                   int32_t* valid /* [S] */, void* tables, void* stream);
size_t cl_icrf_energy_workspace_bytes(const cl_icrf_problem* p, int64_t n_pixels);
int cl_icrf_energy_partial(const cl_icrf_problem* p, const void* tables,
                           const uint8_t* dn /* device [n_pixels][N] */,
                           const double* std /* device [n_pixels][N] or NULL */,
                           const double* exposure_s /* HOST [N] */, int64_t n_pixels,
                           double* pair_acc /* device [S][pairs][2] */, void* workspace,
                           size_t workspace_bytes, void* stream);
/* The same for 16-bit (or 12-bit) cameras: dn is device [n_pixels][N] uint16, every dn < D <= 65536.  For D > 256 the
 * tables are gathered from global memory (L2) instead of being staged in shared memory. */
int cl_icrf_energy_partial_u16(const cl_icrf_problem* p, const void* tables,
                               const uint16_t* dn /* device [n_pixels][N] */,
                               const double* std /* device [n_pixels][N] or NULL */,
                               const double* exposure_s /* HOST [N] */, int64_t n_pixels,
                               double* pair_acc /* device [S][pairs][2] */, void* workspace,
                               size_t workspace_bytes, void* stream);
int cl_icrf_energy_finalize(const cl_icrf_problem* p, const double* pair_acc,
                            const int32_t* valid, double* energy /* device [S] */, void* stream);

/* The whole objective for one population on this rank's pixel shard in two launches -- the partial kernel and
 * a fused tail: CTA reduction -> exchange of the (S x pairs x 2) sums with the other ranks through PEER MEMORY
 * (plain stores into every peer's exchange buffer over NVLink + a flag; no NCCL launch) -> identical finalize
 * on every rank.  Replaces the loop body of solve_channel (ICRF_calibration_exposure.py:357-370 calling
 * _energy_function :148-201) for a population sharded over the GPUs of one node.
 *   peers->buffers[r]: device pointer, valid on THIS device, to rank r's exchange buffer of
 *   cl_icrf_exchange_bytes(p, world) bytes, zero-initialised once (cl_peer_alloc does that; buffers[rank] is
 *   this rank's own).  world == 1: any zeroed device buffer of that size; nothing is exchanged.
 *   Every rank must make the same sequence of calls (the buffers carry a generation counter).
 *   pair_acc receives the sums over ALL ranks, energy the finalised energies. */
#define CL_MAX_PEERS 16
typedef struct cl_peer_group {
    int32_t world, rank;
    void* buffers[CL_MAX_PEERS];
} cl_peer_group;
/* select != NULL: the differential-evolution selection of this generation (what cl_de_select does, see below) runs in
 * the same launch right after the finalize, with the energies just computed as the trial energies. */
typedef struct cl_de_select_args {
    double* pop;              /* device [n_members][n_params], unit cube */
    double* energies;         /* device [n_members] */
    const double* trial;      /* device [n_members][n_params] */
    int32_t n_members, n_params;
    double tol, atol;
    int64_t* generation;      /* device counter, incremented */
    int32_t* status;          /* device [4] */
    double* best;             /* device [3] */
} cl_de_select_args;
size_t cl_icrf_exchange_bytes(const cl_icrf_problem* p, int world);
int cl_icrf_energy_population(const cl_icrf_problem* p, const void* tables, const uint8_t* dn, const double* std,
                              const double* exposure_s /* HOST [N] */, int64_t n_pixels, const int32_t* valid,
                              double* pair_acc, double* energy, void* workspace, size_t workspace_bytes,
                              const cl_peer_group* peers, const cl_de_select_args* select /* nullable */,
                              void* stream);
/* cl_icrf_energy_population for uint16 samples (dn < D <= 65536); the exchange buffers and the peer route are the
 * same as for uint8 (cl_icrf_exchange_bytes depends on neither D nor the sample type). */
int cl_icrf_energy_population_u16(const cl_icrf_problem* p, const void* tables, const uint16_t* dn,
                                  const double* std, const double* exposure_s /* HOST [N] */, int64_t n_pixels,
                                  const int32_t* valid, double* pair_acc, double* energy, void* workspace,
                                  size_t workspace_bytes, const cl_peer_group* peers,
                                  const cl_de_select_args* select /* nullable */, void* stream);

/* Peer-visible device buffers (CUDA IPC) for the exchange above: cl_peer_alloc on the owning rank (cudaMalloc,
 * zero-filled, synchronous), the 64-byte handle travels to the other processes by any means
 * (torch.distributed.all_gather_object in parallel.py), cl_peer_open maps it there.  These four calls are the
 * only ones of the library that allocate or synchronise; they are set-up, not data path. */
typedef struct cl_ipc_handle { unsigned char bytes[64]; } cl_ipc_handle;
int cl_peer_alloc(size_t bytes, void** dev_ptr, cl_ipc_handle* handle);
int cl_peer_open(const cl_ipc_handle* handle, void** dev_ptr);
int cl_peer_close(void* dev_ptr);
int cl_peer_free(void* dev_ptr);

/* ---------------------------------------------------------------------------------------------
 * Linearity analysis of one exposure pair (SURVEY.md 8f, first "next" row) -- replaces
 * AbstractMeasurand.apply_thresholds (modules/measurand.py:375-428), compute_difference
 * (:620-655) and compute_dimension_statistics(axis=(0,1)) (:318-350) as
 * ExposureSeries.process_linearity chains them (modules/exposure_series.py:421-446).
 *
 *   a = x - m*y,  r = a / (m*y)  (+ first-order uncertainties when a std is given);
 *   stats[which][k][c], which: 0 = absolute, 1 = relative; k: 0 = mean, 1 = std, 2 = error
 *   (NaN-skipping; inverse-sigma weighted when any std is given, error = mean sigma, else NaN).
 *   lower / upper: HOST arrays [C] of per-channel limits applied to x and y first (values outside
 *   become NaN), or both NULL when the inputs are already thresholded.
 * ------------------------------------------------------------------------------------------- */
size_t cl_pair_statistics_workspace_bytes(int channels);
int cl_pair_statistics(const double* x_val, const double* x_std, const double* y_val, const double* y_std,
                       double multiplier, const double* lower, const double* upper, int64_t n_samples,
                       int channels, double* stats /* device [2][3][C] */, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ---- Egress: 8-bit export ---------------------------------------------------------------------
 * Replaces the array part of ImageSet.save_8bit (modules/image_set.py:321-358):
 *   max_float = np.amax(val); if max_float > 1: val /= max_float
 *   out = np.around(val * max_dn).astype(uint8)
 * val: n float64 samples (device); out: n bytes (device); out_max: optional device double receiving
 * np.amax(val) (NaN if any sample is NaN -- then, like the reference, nothing is normalised).
 * Bytes are identical to NumPy's (IEEE divide / multiply, round-half-even, C cast through int32).
 * Two launches; workspace holds the per-block maxima. */
size_t cl_quantize_8bit_workspace_bytes(void);
int cl_quantize_8bit(const double* val, int64_t n_samples, double max_dn, uint8_t* out, double* out_max,
                     void* workspace, size_t workspace_bytes, void* stream);

/* ---- Differential evolution on the device (calibration driver) -----------------------------------
 * Replaces the host loop of scipy's DifferentialEvolutionSolver as the reference configures it
 * (modules/ICRF_calibration_exposure.py:357-361: 'currenttobest1bin', mutation (0, 1.95) = dither,
 * recombination 0.4, tol 0.01), in its vectorized 'deferred' form.  One generation =
 *   cl_de_trial -> cl_icrf_curves / cl_icrf_energy_partial / [all-reduce] / cl_icrf_energy_finalize -> cl_de_select
 * All pointers are device pointers.  pop: [S][P] in the unit cube, row 0 = best member; energies [S];
 * generation: one int64 counter (read by cl_de_trial, incremented by cl_de_select); lower / upper [P];
 * trial [S][P] (unit cube) and params [S][P] (scaled, the input of cl_icrf_curves) are outputs.
 * Random draws are counter based (splitmix64 keyed by seed, generation, member, slot): see oracle/de.py.
 * status [4] int32 = {converged, generations done, members replaced, previous index of the best};
 * best [3] = {lowest energy, std(E), mean(E)}.  Converged <=> no +inf energy and
 * std(E) <= atol + tol * |mean(E)|  (scipy's rule). */
int cl_de_trial(const double* pop, int n_members, int n_params, double dither_lo, double dither_hi,
                double crossover, uint64_t seed, const int64_t* generation, const double* lower,
                const double* upper, double* trial, double* params, void* stream);
/* cl_de_trial fused with cl_icrf_curves (one launch: CTA s draws member s's trial vector and builds its curve
 * and tables; D > 256: every CTA of candidate s's cluster draws it, one writes trial / params).
 * n_members <= p->n_candidates; the padding candidates evaluate the zero parameter vector. */
int cl_de_trial_curves(const cl_icrf_problem* p, const double* pop, int n_members, double dither_lo,
                       double dither_hi, double crossover, uint64_t seed, const int64_t* generation,
                       const double* lower, const double* upper, double* trial, double* params,
                       const double* mean_icrf, const double* pca, double* curves, int32_t* valid, void* tables,
                       void* stream);
int cl_de_select(double* pop, double* energies, const double* trial, const double* trial_energies,
                 int n_members, int n_params, double tol, double atol, int64_t* generation, int32_t* status,
                 double* best, void* stream);

/* ---- Measurand operators with uncertainty propagation (SURVEY.md 8f, rank 4) --------------------------------
 * One fused streaming pass per operator instead of the reference's chain of NumPy ufuncs
 * (modules/measurand.py:106-241 operators, :243-279 logarithms, :620-655 compute_difference).
 *   cl_measurand_binary: op 0 add, 1 sub, 2 mul, 3 div, 4 pow;  out = x (op) y with std per the reference formulae.
 *     y_period == n: same shape; otherwise y is a "suffix" operand (per-channel vector, scalar): element i of x
 *     pairs with element i % y_period of y.  x_std / y_std may be NULL (taken as zeros); out_std == NULL: values only.
 *   cl_measurand_log: base10 == 0: log(x), std / log(x) (the reference's literal formula); 1: log10(x),
 *     std / (x (log 5 + log 2)).
 *   cl_measurand_difference: abs = x - m y, rel = abs / (m y), and their uncertainties when any std is given. */
int cl_measurand_binary(int op, const double* x_val, const double* x_std, const double* y_val, const double* y_std,
                        int64_t n, int64_t y_period, double* out_val, double* out_std, void* stream);
int cl_measurand_log(int base10, const double* val, const double* std, int64_t n, double* out_val, double* out_std,
                     void* stream);
int cl_measurand_difference(const double* x_val, const double* x_std, const double* y_val, const double* y_std,
                            double multiplier, int64_t n, double* abs_val, double* abs_std, double* rel_val,
                            double* rel_std, void* stream);

/* ---- Camera noise profiles ---------------------------------------------------------------------------------
 * Replaces the scatter loop of compute_noise_profiles (modules/video_processing.py:92-104): for every sample of
 * every frame, hist[mean_u8[sample]][frame[sample]][channel] += 1.  frames: device [n_frames][n_samples] uint8
 * (channel-interleaved images), mean_u8: device [n_samples] (the uint8 mean frame of welford_algorithm), hist: device
 * int64 [256][256][channels], ACCUMULATED into (the caller clears it once and may feed the video in chunks). */
int cl_noise_profiles(const uint8_t* frames, int n_frames, int64_t n_samples, int channels, const uint8_t* mean_u8,
                      int64_t* hist, void* stream);

/* ---- Per-channel histogram -------------------------------------------------------------------------
 * Replaces the array part of compute_channel_histogram (modules/measurand.py:430-469): np.histogram of
 * the finite values of channel `channel` of an interleaved (n_pixels, channels) float64 array with `bins`
 * uniform bins on [first_edge, last_edge]; std != NULL: samples with sigma == 0 are dropped and the rest
 * weigh 1/sigma.  edges: device [bins + 1] = np.linspace(first_edge, last_edge, bins + 1) (NumPy's edge
 * corrections compare against them).  hist: device [bins] float64 (exact counts when unweighted); it is
 * cleared by the call. */
int cl_channel_histogram(const double* val, const double* std, int64_t n_pixels, int channels, int channel,
                         int bins, double first_edge, double last_edge, const double* edges, double* hist,
                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CAMERA_LINEARITY_B200_H */
