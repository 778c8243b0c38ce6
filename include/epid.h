/* libepid -- B200-native (sm_100a) EPID image-analysis hot path.  C-ABI boundary.
 *
 * The reference (jrkerns/pylinac v3.46.0) is pure Python and has NO FFI of its own: its numerical
 * work goes through numpy / scipy.ndimage / scipy.signal call sites inside pylinac/core/image.py,
 * pylinac/core/array_utils.py, pylinac/core/profile.py and the module-level analyze() methods.
 * Each entry point below replaces one of those call sites (cited as file:line of the reference);
 * pylinac_b200/_native.py is the ctypes binding a maintainer would add (see INTEGRATION.md).
 *
 * Conventions
 *  - plain C, no exceptions; every function returns an int32 status (EPID_OK == 0, negative = error).
 *  - images are row-major [row=y][col=x]; a "batch" is n equal-sized frames, contiguous.
 *  - host pointers are owned by the caller; device memory is owned by ctx / batch handles.
 *  - calls are synchronous unless stated otherwise (they return after the result is in host memory).
 *  - there is NO CPU fallback: without a CUDA device every compute entry point returns EPID_ERR_NO_DEVICE.
 */
#ifndef EPID_H
#define EPID_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ----------------------------------------------------------------------------------------- status */
enum {
    EPID_OK = 0,
    EPID_ERR_NO_DEVICE = -1,      /* no CUDA device / driver */
    EPID_ERR_CUDA = -2,           /* CUDA runtime error, see epid_last_error() */
    EPID_ERR_INVALID = -3,        /* bad argument (maps to ValueError) */
    EPID_ERR_UNSUPPORTED = -4,    /* size / dtype outside what the kernels support */
    EPID_ERR_NOMEM = -5,
    EPID_ERR_NCCL = -6,
    EPID_ERR_INDEX = -7           /* an index outside the array, as numpy's IndexError (disk ROIs over the bottom / right edge) */
};

/* element types of image batches (numpy dtypes the reference's operators preserve, core/array_utils.py) */
enum { EPID_U8 = 0, EPID_U16 = 1, EPID_I32 = 2, EPID_F32 = 3, EPID_F64 = 4, EPID_I16 = 5, EPID_I64 = 6 };

typedef struct epid_ctx epid_ctx;     /* one per device: stream(s), scratch, optional NCCL communicator */
typedef struct epid_batch epid_batch; /* n frames resident in HBM */

/* ----------------------------------------------------------------------------------------- context */
int32_t epid_device_count(int32_t* count);                    /* EPID_OK with *count == 0 if no GPU */
int32_t epid_ctx_create(int32_t device, epid_ctx** out);
int32_t epid_ctx_destroy(epid_ctx* ctx);
const char* epid_last_error(void);                             /* thread-local message of the last failure */
int32_t epid_sync(epid_ctx* ctx);
int32_t epid_device_info(epid_ctx* ctx, int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, size_t* hbm_bytes);
/* PCI bus id ("0000:1b:00.0") of CUDA device `device`: lets a rank bind its host threads / pinned allocations to the GPU's NUMA node */
int32_t epid_device_pci_bus_id(int32_t device, char* out, int32_t cap);
int32_t epid_launch_count(epid_ctx* ctx, int64_t* launches);   /* kernels launched by this ctx so far */
int32_t epid_version(void);
/* options / diagnostic counters (no reference counterpart: the reference has a single CPU code path).
 * EPID_OPT_PF_EXACT_ONLY: 1 = always use the exact-histogram PicketFence pipeline (default 0: fused sample-guided front
 * kernel with automatic per-batch fallback to the exact pipeline).  EPID_CTR_PF_FALLBACKS: batches / chunks re-run exactly. */
/* Keys 2, 4 and 6 are retired and not reused: epid_set_option rejects them as unknown. */
enum { EPID_OPT_PF_EXACT_ONLY = 1,
       EPID_OPT_PF_WIN2 = 3 /* 1 (default) = two-kernel window path (medians + per-window analysis); 0 = single per-window kernel (bit-identical) */,
       EPID_OPT_PF_FAST_REDO = 5 /* 1 (default): a deferred frame whose _has_noise() == True can be certified by one exact count is median-filtered
                                    and re-run by the certified fast pipeline; 0 = every deferred frame goes to the exact-histogram pipeline */,
       EPID_OPT_STATS_EXACT = 7 /* 1: FieldAnalysis / Starshot compute check_inversion_by_histogram from the exact histogram for every frame
                                   (default 0: decision certified from exact counts at pilot thresholds, exact histogram only where that fails) */ };
enum { EPID_CTR_PF_FALLBACKS = 1, EPID_CTR_PF_REDONE_FRAMES = 2 /* frames re-run individually (fast re-run or exact pipeline) */,
       EPID_CTR_PF_EXACT_FRAMES = 3 /* of those: frames that went through the exact-histogram pipeline */,
       EPID_CTR_STATS_UNCERTIFIED = 4 /* FieldAnalysis / Starshot frames whose check_inversion_by_histogram decision needed exact percentiles */ };
int32_t epid_set_option(epid_ctx* ctx, int32_t key, int64_t value);
int32_t epid_get_counter(epid_ctx* ctx, int32_t key, int64_t* value);

/* pinned host memory (for the H2D legs of the batched entry points) */
int32_t epid_host_alloc(size_t bytes, void** out);
int32_t epid_host_free(void* p);

/* ----------------------------------------------------------------------------------------- batches */
/* replaces: ArrayImage(array) / DicomImage pixel_array  (core/image.py:1818-1848, 1431-1444) */
int32_t epid_batch_upload(epid_ctx* ctx, const void* host, int32_t dtype, int32_t n, int32_t h, int32_t w, epid_batch** out);
int32_t epid_batch_alloc(epid_ctx* ctx, int32_t dtype, int32_t n, int32_t h, int32_t w, epid_batch** out);
int32_t epid_batch_download(epid_batch* b, void* host);        /* whole batch, native dtype */
int32_t epid_batch_write(epid_batch* b, const void* host);     /* overwrite an existing batch from host memory (same shape / dtype) */
int32_t epid_batch_free(epid_batch* b);
int32_t epid_batch_shape(const epid_batch* b, int32_t* dtype, int32_t* n, int32_t* h, int32_t* w);
int32_t epid_batch_device_ptr(const epid_batch* b, void** dptr);

/* ----------------------------------------------------------------------------------------- frame statistics
 * One streaming read of every frame: min, max, sum, row sums, column sums, exact order statistics.
 * replaces: array.min()/max()/mean() (core/image.py:851,896; picketfence.py:231-232), np.percentile / np.median
 * of a full frame (picketfence.py:233,1510; core/image.py:918-920; winston_lutz.py:709,775; starshot.py:227,286),
 * np.sum/np.mean(image, axis) (picketfence.py:748-750,1513-1514; field_analysis.py:488-506).
 * The view [r0:r0+vh, c0:c0+vw] of each frame is analysed (crop is a view: core/image.py:714-745).
 * Integer dtypes U8/U16 only (exact integer histogram); q in percent, numpy 'linear' method.
 * Outputs (host, may be NULL): min,max: double[n]; sum: double[n] (exact integer sums < 2^53);
 * rowsum: double[n*vh] (sum over columns of each row); colsum: double[n*vw]; pct: double[n*nq]. */
int32_t epid_frame_stats(epid_ctx* ctx, const epid_batch* b, int32_t r0, int32_t c0, int32_t vh, int32_t vw,
                         const double* q_percent, int32_t nq,
                         double* mn, double* mx, double* sum, double* rowsum, double* colsum, double* pct);
/* full 65536-bin histogram of the view (uint32 counts [n][65536]); U8/U16 only */
int32_t epid_frame_histogram(epid_ctx* ctx, const epid_batch* b, int32_t r0, int32_t c0, int32_t vh, int32_t vw, uint32_t* hist);

/* ----------------------------------------------------------------------------------------- element-wise operators
 * All write a NEW batch (the reference rebinds self.array to a fresh ndarray, core/image.py:712,757,798,852,866). */
/* array_utils.invert  (core/array_utils.py:75-77): -a + max + min in the array's own dtype (modular for uints) */
int32_t epid_invert(epid_ctx* ctx, const epid_batch* in, epid_batch** out);
/* array_utils.bit_invert (core/array_utils.py:81-89): integer dtypes only, else EPID_ERR_INVALID */
int32_t epid_bit_invert(epid_ctx* ctx, const epid_batch* in, epid_batch** out);
/* array_utils.ground (core/array_utils.py:93-102): a - min + value, same dtype; mins: double[n] (may be NULL) */
int32_t epid_ground(epid_ctx* ctx, const epid_batch* in, double value, epid_batch** out, double* mins);
/* array_utils.normalize (core/array_utils.py:64-71): a / (value or max) -> F64; use_max != 0 ignores value */
int32_t epid_normalize(epid_ctx* ctx, const epid_batch* in, int32_t use_max, double value, epid_batch** out);
/* BaseImage.threshold (core/image.py:785-800): keep a >= t (kind 0, 'high') or a <= t (kind 1), else 0; same dtype */
int32_t epid_threshold(epid_ctx* ctx, const epid_batch* in, double t, int32_t kind, epid_batch** out);
/* BaseImage.as_binary (core/image.py:802-815): (a >= t) -> I64 0/1 */
int32_t epid_binarize(epid_ctx* ctx, const epid_batch* in, double t, epid_batch** out);

/* ----------------------------------------------------------------------------------------- stencils */
/* scipy.ndimage.median_filter(a, size=k) as called by array_utils.filter (core/array_utils.py:131):
 * full k x k footprint, mode='reflect', rank k*k/2, dtype preserved. */
int32_t epid_median_filter(epid_ctx* ctx, const epid_batch* in, int32_t size, epid_batch** out);
/* scipy.ndimage.gaussian_filter(a, sigma) as called by array_utils.filter (core/array_utils.py:133):
 * separable, axis 0 then axis 1, radius int(4*sigma+0.5), mode='reflect', float64 accumulate,
 * result of EACH pass cast to the input dtype (truncation for integers). */
int32_t epid_gaussian_filter(epid_ctx* ctx, const epid_batch* in, double sigma, epid_batch** out);
/* Same passes with caller-supplied correlate1d weights (2*radius+1 doubles).  The python binding passes the weights
 * scipy itself computes (scipy/ndimage/_filters.py:_gaussian_kernel1d) so integer results are bit-exact.
 * axes: 3 = axis 0 then axis 1 (2-D image), 1 = axis 0 only, 2 = axis 1 only (1-D profile stored as one row). */
int32_t epid_correlate1d_passes(epid_ctx* ctx, const epid_batch* in, const double* weights, int32_t radius, int32_t axes, epid_batch** out);
/* scipy.ndimage.sobel(a, axis) (core/image.py:1006-1007, BaseImage.gamma): reflect, same dtype semantics; out F32/F64 */
int32_t epid_sobel(epid_ctx* ctx, const epid_batch* in, int32_t axis, epid_batch** out);

/* ----------------------------------------------------------------------------------------- 1-D profiles
 * pylinac.core.profile.find_peaks (core/profile.py:2545-2649) == scipy.signal.find_peaks(height, distance,
 * prominence, width=min_width, rel_height = 1 - fwxm_height) + search-region trimming + top-max_number selection.
 * values: host double[n].  Arguments follow the reference's python signature after _parse_peak_args has NOT yet
 * been applied (threshold in [0,1] is a ratio of the range, separation in [0,1] a ratio of len, region <= 1 ratios).
 * peak_sort: 0 = 'prominences', 1 = 'peak_heights'.  max_number <= 0: all.  required_prominence < 0: none.
 * Outputs (capacity cap each): idx int64; heights, prominences, left_bases(int64), right_bases(int64), widths,
 * width_heights, left_ips, right_ips double.  *count = number of peaks returned. */
typedef struct {
    double threshold;           /* -inf allowed */
    double peak_separation;
    int32_t max_number;
    double fwxm_height;         /* 0..1 */
    double min_width;
    double search_lo, search_hi;
    int32_t peak_sort;
    double required_prominence; /* < 0: None */
} epid_peak_params;

int32_t epid_find_peaks(epid_ctx* ctx, const double* values, int32_t n, const epid_peak_params* p, int32_t cap,
                        int64_t* idx, double* heights, double* prominences, int64_t* left_bases, int64_t* right_bases,
                        double* widths, double* width_heights, double* left_ips, double* right_ips, int32_t* count);

/* ----------------------------------------------------------------------------------------- Picket Fence
 * PicketFence(image).analyze(**params) + the scalar set of results_data()  (picketfence.py:209-219, 280-329,
 * 636-912, 1313-1363, 1501-1743, 1857-1923) for a batch of frames, one result per frame. */
#define EPID_PF_MAX_PICKETS 32
#define EPID_PF_MAX_LEAVES 160

enum { /* per-frame status (maps to the reference's exceptions) */
    EPID_PF_OK = 0,
    EPID_PF_NO_PICKETS = 1,        /* ValueError "No pickets were found" (picketfence.py:760-764) */
    EPID_PF_NO_MEASUREMENTS = 2,   /* ValueError "No MLC measurements were found" (picketfence.py:804-807) */
    EPID_PF_TOO_MANY_PICKETS = 3,  /* more than EPID_PF_MAX_PICKETS peaks (unsupported) */
    EPID_PF_WINDOW_NO_PEAK = 4,    /* reference would raise IndexError inside FWXMProfile.field_edge_idx */
    EPID_PF_CAPACITY = 5,          /* measurement table capacity exceeded */
    EPID_PF_FLAT_IMAGE = 6         /* max == min: the reference divides by zero */
};

typedef struct {
    /* constructor (picketfence.py:280-329; PFDicomImage :209-219) */
    double dpmm;                 /* image.dpmm (core/image.py:1534-1547) */
    int32_t crop_px;             /* int(round(crop_mm * dpmm)) */
    int32_t filter_size;         /* median filter size, 0 = None */
    /* analyze() (picketfence.py:636-654) */
    double tolerance;
    double action_tolerance;     /* < 0: None */
    int32_t num_pickets;         /* 0: None */
    int32_t sag_px;              /* int(round(sag_adjustment * dpmm)) */
    int32_t orientation;         /* -1 auto, 0 Up-Down, 1 Left-Right */
    int32_t invert;
    double leaf_analysis_width_ratio;
    double picket_spacing;       /* < 0: None (auto) */
    double height_threshold;
    double edge_threshold;
    int32_t peak_sort;           /* 0 'prominences', 1 'peak_heights' */
    double required_prominence;
    int32_t separate_leaves;
    double nominal_gap_mm;
    int32_t has_cax_override;    /* PFDicomImage.center override (picketfence.py:246-260) */
    double cax_x_px, cax_y_px;   /* final centre in pixels when has_cax_override */
    /* MLC arrangement (picketfence.py:68-135): centres (mm), widths (mm), leaf numbers, in the reference's order */
    int32_t n_leaves;
    double leaf_center_mm[EPID_PF_MAX_LEAVES];
    double leaf_width_mm[EPID_PF_MAX_LEAVES];
    int32_t leaf_num[EPID_PF_MAX_LEAVES];
} epid_pf_params;

typedef struct { /* one per frame */
    int32_t status;
    int32_t orientation;                 /* 0 Up-Down, 1 Left-Right */
    int32_t noise_median_passes;         /* how often _check_for_noise filtered (picketfence.py:221-227) */
    int32_t corner_inverted;             /* check_inversion fired (core/image.py:868-897) */
    int32_t height, width;               /* analysed (cropped) shape */
    int32_t n_pickets;
    int32_t n_meas;                      /* rows of the measurement table that belong to this frame (after pruning) */
    int32_t n_leaves_removed;            /* leaf rows dropped by the median-count rule (picketfence.py:810-828) */
    int32_t passed;
    int32_t max_error_picket;
    int32_t max_error_leaf;              /* leaf number; for separate_leaves bank in max_error_bank (0 = A, 1 = B) */
    int32_t max_error_bank;
    int32_t n_failed;                    /* number of failing measurements (see table 'passed' flags) */
    double picket_spacing_px;
    double percent_passing;
    double max_error_mm;
    double abs_median_error_mm;
    double mean_picket_spacing_mm;
    double mlc_skew;
    double cax_px;                       /* image.center component along leaf travel */
    int32_t picket_idx[EPID_PF_MAX_PICKETS];      /* find_fwxm_peaks indices (bit-exact target) */
    double picket_val[EPID_PF_MAX_PICKETS];
    double fit_slope[EPID_PF_MAX_PICKETS];        /* np.polyfit(deg 1) of each picket */
    double fit_intercept[EPID_PF_MAX_PICKETS];
    double offsets_from_cax_mm[EPID_PF_MAX_PICKETS];
    double picket_width_max[EPID_PF_MAX_PICKETS]; /* picket_width_stat (picketfence.py:471-491) */
    double picket_width_mean[EPID_PF_MAX_PICKETS];
    double picket_width_median[EPID_PF_MAX_PICKETS];
    double picket_width_min[EPID_PF_MAX_PICKETS];
} epid_pf_summary;

typedef struct { /* one per kept MLCValue, leaf-major / picket-minor like PicketFence.mlc_meas */
    int32_t leaf_num;
    int32_t picket;
    int32_t passed[2];
    double position[2];      /* px along leaf travel; [1] only for separate_leaves */
    double error[2];         /* mm */
    double width_mm;         /* profile.field_width_mm */
} epid_pf_meas;

/* device-resident batch (uint16): results to host.  meas: [n][meas_cap].  Synchronous. */
int32_t epid_pf_analyze(epid_ctx* ctx, const epid_batch* frames, const epid_pf_params* p,
                        epid_pf_summary* summary, epid_pf_meas* meas, int32_t meas_cap);
/* end-to-end: host frames [n][h][w] uint16 (pinned or pageable) -> chunked H2D overlapped with compute -> results. */
int32_t epid_pf_analyze_host(epid_ctx* ctx, const uint16_t* frames, int32_t n, int32_t h, int32_t w,
                             const epid_pf_params* p, epid_pf_summary* summary, epid_pf_meas* meas, int32_t meas_cap);
/* timing hooks for bench.py: run the device-resident pipeline `iters` times back to back (results stay on the
 * device except the last), return the CUDA-event time of the whole region and of the frame-statistics kernel. */
int32_t epid_pf_bench(epid_ctx* ctx, const epid_batch* frames, const epid_pf_params* p, int32_t iters,
                      float* total_ms, float* stats_kernel_ms, int64_t* launches);
/* the same timed region with CUDA-event marks between the kernels: total_ms of `iters` back-to-back passes, stage_ms[k] summed over
 * the passes, kernel launches and the number of frames the per-frame exact fallback re-ran (when the batch contains deferred frames
 * the passes are timed with the host round trip of the fallback included).  stage_ms[0..8] (bench.py's per-kernel roofline table) =
 * init + pilot, stream, tail, windows (per-window kernel), windows (generic), finalize, exact front end (fallback only), windows
 * (two-kernel path: medians), windows (two-kernel path: per-window analysis) */
int32_t epid_pf_bench_timed(epid_ctx* ctx, const epid_batch* frames, const epid_pf_params* p, int32_t iters, float* total_ms,
                            float* stage_ms, int32_t nstages, int64_t* launches, int64_t* redone_frames);


/* ----------------------------------------------------------------------------------------- Starshot
 * Starshot(image).analyze(**params)  (starshot.py:105-125, 197-401, 701-834; CollapsedCircleProfile core/profile.py:
 * 2244-2283, 2405-2483) for a batch of uint16 frames, one result per frame. */
#define EPID_STAR_MAX_PEAKS 64

enum { /* per-frame status (maps to the reference's exceptions) */
    EPID_STAR_OK = 0,
    EPID_STAR_NO_WOBBLE = 1,       /* RuntimeError "unable to determine a reasonable wobble" (starshot.py:372-376) */
    EPID_STAR_NO_LINES = 2,        /* RuntimeError "unable to properly detect the radiation lines" (starshot.py:339-342) */
    EPID_STAR_NO_START_POINT = 3,  /* no FW80M peak in the central third (reference: IndexError) */
    EPID_STAR_CAPACITY = 4,        /* profile / peak capacity exceeded */
    EPID_STAR_FLAT_IMAGE = 5
};

typedef struct {
    double dpmm;                  /* image.dpmm */
    double radius;                /* analyze() arguments (starshot.py:230-240) */
    double min_peak_height;
    double max_wobble_diameter;
    double tolerance;
    int32_t has_start_point;
    double start_x, start_y;
    int32_t fwhm;
    int32_t recursive;
    int32_t invert;
} epid_star_params;

typedef struct { /* one per frame */
    int32_t status;
    int32_t hist_inverted;        /* check_inversion_by_histogram([4, 50, 96]) fired */
    int32_t start_x, start_y;     /* _get_reasonable_start_point (bit-exact target) */
    double local_max;             /* np.percentile(central third, 90) */
    int32_t iterations;           /* StarProfile constructions of _get_reasonable_wobble */
    int32_t profile_len;
    double radius_px;             /* circle_profile.radius */
    int32_t n_peaks, n_lines;
    int32_t peak_idx[EPID_STAR_MAX_PEAKS];   /* find_fwxm_peaks indices on the rolled profile (bit-exact target) */
    double peak_x[EPID_STAR_MAX_PEAKS], peak_y[EPID_STAR_MAX_PEAKS];
    double wobble_x, wobble_y;    /* wobble.center (px) */
    double wobble_radius_px, wobble_radius_mm;
    double angles[EPID_STAR_MAX_PEAKS / 2];
    int32_t passed;
    int32_t pad;
} epid_star_result;

/* gauss_weights / gauss_offsets: scipy _gaussian_kernel1d tables for sigma = 1 .. max_sigma (host; weights of sigma s start at
 * gauss_offsets[s], 2 * int(4 s + 0.5) + 1 doubles each), computed by the binding exactly like scipy does. */
int32_t epid_starshot_analyze(epid_ctx* ctx, const epid_batch* frames, const epid_star_params* p, const double* gauss_weights,
                              const int32_t* gauss_offsets, int32_t max_sigma, epid_star_result* results);


/* CircleProfile / CollapsedCircleProfile._profile + x / y locations (core/profile.py:2179-2283, 2405-2483) of ONE image
 * (batch of 1; U8 / U16 / F32 / F64): nearest-neighbour samples (scipy.ndimage.map_coordinates order=0, 0 outside) on
 * radians = arange(start_angle, 2 pi + start_angle - interval, interval)[::-1 if ccw], interval = 2 pi / (pi * r_max * 2 *
 * sampling_ratio); collapsed != 0: mean over num_profiles radii linspace(r (1 - width_ratio), r (1 + width_ratio)).
 * cap: capacity of the three output arrays; *count = number of samples. */
int32_t epid_circle_profile(epid_ctx* ctx, const epid_batch* image, double cx, double cy, double radius, double start_angle,
                            int32_t ccw, double sampling_ratio, int32_t collapsed, double width_ratio, int32_t num_profiles,
                            int32_t cap, double* profile, double* x_locations, double* y_locations, int32_t* count);

/* ----------------------------------------------------------------------------------------- Field analysis
 * FieldAnalysis(image).analyze(**params)  (field_analysis.py:445-864, 1069-1117; protocol functions :37-231; SingleProfile
 * core/profile.py:1125-1937) for a batch of uint16 frames, one result per frame.  Interpolation NONE / LINEAR, edge
 * detection FWHM / INFLECTION_DERIVATIVE, every normalisation, protocols NONE / VARIAN / SIEMENS / ELEKTA. */
enum { /* per-frame status */
    EPID_FIELD_OK = 0,
    EPID_FIELD_NO_EDGES = 1,     /* a profile without a usable peak / inflection (reference: IndexError in find_peaks output) */
    EPID_FIELD_FLAT_IMAGE = 2
};

typedef struct {
    double dpmm;                       /* image.dpmm */
    int32_t protocol;                  /* 0 NONE, 1 VARIAN, 2 SIEMENS, 3 ELEKTA (field_analysis.py:233-289) */
    int32_t centering;                 /* 0 MANUAL, 1 BEAM_CENTER, 2 GEOMETRIC_CENTER (core/profile.py:187-192) */
    double vert_position, horiz_position, vert_width, horiz_width;
    double in_field_ratio, slope_exclusion_ratio;
    int32_t invert;
    double penumbra_lower, penumbra_upper;
    int32_t interpolation;             /* 0 NONE, 1 LINEAR */
    double interpolation_resolution_mm;
    int32_t ground;
    int32_t normalization;             /* 0 NONE, 1 GEOMETRIC_CENTER, 2 BEAM_CENTER, 3 MAX */
    int32_t edge;                      /* 0 FWHM, 1 INFLECTION_DERIVATIVE */
    double edge_smoothing_ratio;
} epid_field_params;

typedef struct { /* one per frame: FieldAnalysis._results + protocol results (field_analysis.py:755-863) */
    int32_t status;
    int32_t hist_inverted;             /* check_inversion_by_histogram() fired (field_analysis.py:472) */
    int32_t strip_rows[2];             /* rows [bottom, top) averaged into the horizontal profile */
    int32_t strip_cols[2];             /* columns [left, right) averaged into the vertical profile */
    int32_t profile_len[2];            /* samples of the horizontal / vertical SingleProfile */
    double top_penumbra_mm, bottom_penumbra_mm, left_penumbra_mm, right_penumbra_mm;
    double geometric_center_index_x_y[2], beam_center_index_x_y[2];
    double field_size_vertical_mm, field_size_horizontal_mm;
    double beam_center_to_top_mm, beam_center_to_bottom_mm, beam_center_to_left_mm, beam_center_to_right_mm;
    double cax_to_top_mm, cax_to_bottom_mm, cax_to_left_mm, cax_to_right_mm;
    double top_position_index_x_y[2];
    double top_horizontal_distance_from_cax_mm, top_vertical_distance_from_cax_mm;
    double top_horizontal_distance_from_beam_center_mm, top_vertical_distance_from_beam_center_mm;
    double left_slope_percent_mm, right_slope_percent_mm, top_slope_percent_mm, bottom_slope_percent_mm;
    double symmetry_horizontal, symmetry_vertical, flatness_horizontal, flatness_vertical;
} epid_field_result;

/* samples of SingleProfile(values of length n0, dpmm, interpolation, resolution) (core/profile.py:1306-1322) */
int32_t epid_field_profile_len(int32_t n0, double dpmm, int32_t interpolation, double resolution_mm);
/* gauss_h / gauss_v: scipy gaussian_filter1d weights (2 * lw + 1 doubles, already reversed for correlate1d) for
 * sigma = edge_smoothing_ratio * profile length of the horizontal / vertical profile; may be NULL when edge == 0. */
int32_t epid_field_analyze(epid_ctx* ctx, const epid_batch* frames, const epid_field_params* p, const double* gauss_h, int32_t lw_h,
                           const double* gauss_v, int32_t lw_v, epid_field_result* results);

/* SingleProfile(values, dpmm, interpolation, ground, ..., edge_detection_method, ...) and its query methods for ONE host
 * profile (core/profile.py:1125-1937): fwxm_data(x), beam_center(), geometric_center(), inflection_data(), penumbra(lower,
 * upper), field_data(in_field_ratio, slope_exclusion_ratio), all evaluated in one launch.  Indices are in the units of the
 * original samples (x_values = range(len(values))); the interpolated abscissae are linspace(x_start, x_stop, n). */
typedef struct {
    double dpmm;                       /* <= 0: None (interpolation_factor is used) */
    int32_t interpolation;             /* 0 NONE, 1 LINEAR, 2 = values are already sampled on linspace(x_start, x_stop, n0): cubic
                                          (Interpolation.SPLINE) interpolation or custom uniform x_values, prepared by the caller */
    double interpolation_resolution_mm, interpolation_factor;
    int32_t ground, normalization, edge, centering;   /* codes as in epid_field_params; centering 2 = GEOMETRIC_CENTER; edge 2 = the
                                          field edges are supplied (edge_left / edge_right: Hill-function inflection points) */
    double edge_smoothing_ratio;
    double x_start, x_stop;            /* interpolation == 2 */
    double edge_left, edge_right;      /* edge == 2 */
} epid_sp_params;

typedef struct {
    int32_t status;                    /* 0 ok, 1: no usable peak while normalising */
    int32_t n;                         /* samples after interpolation */
    double x_start, x_stop;
    double values_max;
    double geometric_center_index, geometric_center_value;
    int32_t beam_ok, fwxm_ok, infl_ok, pen_ok, fd_ok, fd_field_values_n;
    double beam_center_index, beam_center_value_at_rounded;
    double fwxm_left, fwxm_right, fwxm_center_value_at_rounded, fwxm_left_value_at_rounded, fwxm_right_value_at_rounded;
    double infl_left, infl_right, infl_left_value_exact, infl_right_value_exact, infl_left_value_rounded, infl_right_value_rounded;
    double pen_left_lower, pen_left_upper, pen_right_lower, pen_right_upper;
    double fd_width, fd_beam_center, fd_cax, fd_left, fd_right, fd_inner_left, fd_inner_right;
    double fd_left_slope, fd_left_intercept, fd_right_slope, fd_right_intercept;
    double fd_top_index, fd_top_value, fd_top_params[3];
    double fd_beam_center_value, fd_cax_value, fd_left_value, fd_right_value;
} epid_sp_result;

/* x_values: NULL, or with interpolation == 2 the n0 increasing (possibly unevenly spaced) abscissae of `values` (x_start / x_stop are
 * then x_values[0] / x_values[n0 - 1]).  gauss: gaussian_filter1d weights for sigma = edge_smoothing_ratio * n_expect (NULL when edge == 0).  values_out (cap):
 * the interpolated / grounded / normalised values; field_values_out (cap): field_data()["field values"]. */
int32_t epid_single_profile(epid_ctx* ctx, const double* values, const double* x_values, int32_t n0, const epid_sp_params* p, const double* gauss, int32_t lw,
                            int32_t n_expect, double fwxm_x, double pen_lower, double pen_upper, double in_field_ratio,
                            double slope_exclusion_ratio, epid_sp_result* result, double* values_out, double* field_values_out,
                            int32_t cap);

/* ----------------------------------------------------------------------------------------- Winston-Lutz (per image)
 * WinstonLutz2D(image).analyze(bb_size_mm, low_density_bb, open_field, bb_proximity_mm) (winston_lutz.py:668-829, 1109-1231;
 * SizedDiskLocator / find_features metrics/image.py:564-612, metrics/utils.py:66-190; predicates metrics/features.py:7-68) for a
 * batch of uint16 frames, one result per frame.  BB arrangement ISO (nominal BB position = EPID centre), no shift vector. */
enum { /* per-frame status (maps to the reference's exceptions) */
    EPID_WL_OK = 0,
    EPID_WL_NO_BB = 1,        /* ValueError "Couldn't find the minimum number of disks" / BB_ERROR_MESSAGE */
    EPID_WL_MISMATCH = 2,     /* ValueError "The number of detected fields and BBs do not match" */
    EPID_WL_NO_FIELD = 3,     /* ValueError "No fields were detected" */
    EPID_WL_CAPACITY = 4,     /* search window / field / region larger than the kernels' shared-memory tiles */
    EPID_WL_FLAT_IMAGE = 5
};

typedef struct {
    double dpmm;
    double bb_size_mm;
    int32_t low_density_bb;
    int32_t open_field;
    double bb_proximity_mm;
} epid_wl_params;

typedef struct { /* one per frame */
    int32_t status;
    int32_t inverted;             /* check_inversion_by_histogram((0.01, 50, 99.99)) fired */
    int32_t crop_px;              /* pixels _clean_edges removed from every edge */
    int32_t height, width;        /* analysed (cropped) shape */
    int32_t n_bbs;                /* BB candidates accepted at the first successful threshold */
    int32_t threshold_passes;     /* thresholds visited by find_features */
    int32_t pad;
    double bb_x, bb_y;            /* matched BB (weighted centroid), pixels of the cropped image */
    double field_x, field_y;      /* field CAX (centre of mass of the filled field mask) */
    double epid_x, epid_y;        /* image centre */
    double cax2bb_x, cax2bb_y, cax2bb_distance;         /* mm */
    double cax2epid_x, cax2epid_y, cax2epid_distance;   /* mm */
} epid_wl_result;

int32_t epid_wl2d_analyze(epid_ctx* ctx, const epid_batch* frames, const epid_wl_params* p, epid_wl_result* results);

/* ----------------------------------------------------------------------------------------- SizedDiskRegion / SizedDiskLocator
 * img.compute(SizedDiskLocator(...)) (metrics/image.py:402-667): sample = image[window] around the expected position, inverted,
 * stretched to [0, 1]; find_features (metrics/utils.py:66-190): <= 50 thresholds { label (4-connectivity), clear_border, regionprops,
 * is_right_size_bb / is_round / is_right_circumference / is_symmetric / is_solid } -> weighted centroids, de-duplicated by the
 * minimum separation, until max_number points are found.  One result per uint16 frame; status values are EPID_WL_*. */
#define EPID_DISK_MAX 8
typedef struct {
    double dpmm;
    double expected_x, expected_y;     /* pixels, image coordinates (the caller has applied from_center / the physical-units quirks) */
    double window_w, window_h;         /* search window, pixels */
    double radius_mm, tolerance_mm;
    double min_separation_px;
    int32_t invert;
    int32_t max_number;
    int32_t conditions;                /* bit mask of the detection conditions: 1 is_right_size_bb, 2 is_round, 4 is_right_circumference,
                                          8 is_symmetric, 16 is_solid (metrics/features.py:7-68), 32 is_modest_size (winston_lutz.py:598-606) */
    int32_t pad;
} epid_disk_params;

typedef struct {
    int32_t status;
    int32_t n_points;                  /* detected disks (image coordinates x[], y[]) */
    int32_t n_regions;                 /* regions that passed every condition at the LAST threshold visited (what find_features returns) */
    int32_t passes;
    int32_t left, top;                 /* offsets of the sample window */
    double x[EPID_DISK_MAX], y[EPID_DISK_MAX];
    /* regionprops of those regions, sample (window) coordinates */
    double r_area[EPID_DISK_MAX], r_filled_area[EPID_DISK_MAX], r_perimeter[EPID_DISK_MAX], r_convex_area[EPID_DISK_MAX];
    double r_centroid_y[EPID_DISK_MAX], r_centroid_x[EPID_DISK_MAX], r_wcentroid_y[EPID_DISK_MAX], r_wcentroid_x[EPID_DISK_MAX];
    int32_t r_bbox[EPID_DISK_MAX][4];  /* min_row, min_col, max_row, max_col (half-open) */
} epid_disk_result;

int32_t epid_disk_locate(epid_ctx* ctx, const epid_batch* frames, const epid_disk_params* p, epid_disk_result* results);

/* ----------------------------------------------------------------------------------------- spline zoom
 * scipy.ndimage.zoom(a, zoom, order, mode) for 2-D frames (both axes) or 1-D profiles (h == 1: the sample axis) ->
 * float64 batch of shape round(shape * zoom).  order 1 or 3; mode 0 = 'constant' (equate_images, core/image.py:217), 1 = 'nearest'
 * (ProfileBase.as_resampled, core/profile.py:384-390), 3 = 'nearest' with grid_mode=True (PhysicalProfileMixin.as_resampled,
 * core/profile.py:951-1013). */
int32_t epid_zoom(epid_ctx* ctx, const epid_batch* in, double zoom, int32_t order, int32_t mode, epid_batch** out);

/* BaseImage.rotate(angle, mode) (core/image.py:780-783): skimage.transform.rotate(order 1) semantics -- img_as_float conversion
 * (uint8 / 255, uint16 / 65535), counter-clockwise rotation by angle_deg about (cols / 2 - 0.5, rows / 2 - 0.5), bilinear sampling;
 * mode 0 = 'constant' (0 outside), 1 = 'edge'.  float64 output of the input shape. */
int32_t epid_rotate(epid_ctx* ctx, const epid_batch* in, double angle_deg, int32_t mode, epid_batch** out);

/* ----------------------------------------------------------------------------------------- gamma map
 * BaseImage.gamma (core/image.py:928-1017), Bakai eq. 6: ref / comp are the float64 images AFTER the reference's inversion check,
 * ground() and normalize(); threshold_abs = threshold * max(ref); dose_frac = doseTA / 100; dist_px = distTA * dpmm.  The Sobel
 * gradient (scipy.ndimage.sobel on the float32 reference with nan below the threshold, mode reflect), hypot and the division are
 * one fused kernel; out: a new float64 batch (nan where the reference is below the threshold). */
int32_t epid_gamma(epid_ctx* ctx, const epid_batch* ref, const epid_batch* comp, double threshold_abs, double dose_frac, double dist_px,
                   epid_batch** out);

/* ----------------------------------------------------------------------------------------- ROI statistics / weighted centroid
 * RectangleROI.mean / std / min / max (core/roi.py:533-706): pixels of a rectangle given by its corners verts_xy[nroi][4][(x, y)]
 * (any rotation), selected like skimage.draw.polygon (pixel centres inside or on the boundary, clipped to the image).  Every ROI is
 * evaluated on every frame of the batch: outputs [n][nroi] (may be NULL).  std is the population standard deviation (np.std). */
int32_t epid_roi_stats(epid_ctx* ctx, const epid_batch* b, int32_t nroi, const double* verts_xy, double* count, double* mean,
                       double* std, double* mn, double* mx);
/* DiskROI.pixel_value / mean / std / min / max (core/roi.py:103-132) and LowContrastDiskROI.percentile (core/roi.py:406-408) of ndisk
 * disks (centers_xy[ndisk][(x, y)], radii[ndisk]) on every frame: outputs [n][ndisk] (may be NULL), pct [n][ndisk][npct] (may be NULL).
 * Pixel set: skimage.draw.disk(center=(y, x), radius) WITHOUT shape, as DiskROI.circle_mask (core/roi.py:134-138) calls it -- box
 * ceil(c - r) .. floor(c + r), ((i - r_org) / r)**2 + ((j - c_org) / r)**2 < 1 in fp64, and numpy's negative-index wrap-around for rows /
 * columns in [-dim, -1].  A selected index outside [-dim, dim - 1] returns EPID_ERR_INDEX.  8 / 16-bit frames: exact integer moments
 * (mean, min, max bit-exact, std from the exact N * S2 - S1^2); other dtypes: fp64 moments, std from the centred second moment.
 * median (np.median) and the percentiles (np.percentile, linear; 0 <= p <= 100 else EPID_ERR_INVALID; at most EPID_DISK_MAX_PCT) are
 * exact order statistics (radix select) combined with numpy's arithmetic (float32 frames in float32).  A disk with no pixels gives
 * count 0 and NaN statistics; a disk containing a NaN pixel gives NaN statistics. */
#define EPID_DISK_MAX_PCT 16
int32_t epid_disk_roi_stats(epid_ctx* ctx, const epid_batch* b, int32_t ndisk, const double* centers_xy, const double* radii,
                            int32_t npct, const double* percentiles, double* count, double* mean, double* std, double* mn,
                            double* mx, double* median, double* pct);
/* DiskROI.circle_mask / pixel_values (clip = 0, core/roi.py:103-105, 134-138) and the pixel set of masked_array (clip = 1:
 * draw.disk(..., shape=shape), core/roi.py:140-150) of one disk on frame `frame`: *count = number of pixels; when values != NULL
 * (capacity >= count, element type = the batch dtype) the values in np.nonzero (row-major) order, and when rows / cols != NULL the row /
 * column indices skimage returns (unwrapped: negative for the wrapped rows / columns of clip = 0).  Call once with values == NULL for
 * the count, then with a buffer.  clip = 0 and a selected index outside [-dim, dim - 1]: EPID_ERR_INDEX. */
int32_t epid_disk_roi_pixels(epid_ctx* ctx, const epid_batch* b, int32_t frame, const double* center_xy, double radius, int32_t clip,
                             int64_t capacity, void* values, int32_t* rows, int32_t* cols, int64_t* count);
/* WeightedCentroid.calculate (metrics/image.py:959-983): cx = sum(x * a) / sum(a), cy likewise; total = sum(a) (may be NULL). */
int32_t epid_weighted_centroid(epid_ctx* ctx, const epid_batch* b, double* cx, double* cy, double* total);

/* ----------------------------------------------------------------------------------------- VMAT (DRGS / DRMLC) and DLG
 * VMATBase.__init__ / analyze, VMATLinearBase._identify_images / _roi_profiles / _calculate_segments, Segment.r_corr / stdev,
 * _update_r_corrs (vmat.py:249-275, 309-346, 408-436, 739-841): n independent (image 1, image 2) pairs, img1->n == img2->n, uint16.
 * Per pair on the device: ground() + check_inversion() of both images (folded into an affine map of the raw pixels, nothing is
 * rewritten), column-mean FWXM profiles (ground, beam-centre normalisation, stretch, 90th-percentile normalisation, in-field
 * length / std) -> which image is the open field, field centre (image centre + warning flag when it lies outside the central
 * third), then per segment the mean / std of DMLC / open over the pixels of the segment rectangle (never materialising the ratio
 * image) -> R_corr, R_dev, pass / fail and the aggregates. */
#define EPID_VMAT_MAX_SEG 16
typedef struct {
    int32_t ground;              /* VMATBase(ground=True) */
    int32_t check_inversion;     /* VMATBase(check_inversion=True) */
    int32_t invert_image_order;  /* analyze(invert_image_order=False) */
    int32_t nseg;                /* len(roi_config) <= EPID_VMAT_MAX_SEG */
    double dpmm;
    double tolerance_percent;    /* analyze(tolerance=1.5) */
    double seg_w_mm, seg_h_mm;   /* segment_size_mm: (5, 100) */
    double offset_mm[EPID_VMAT_MAX_SEG];
} epid_vmat_params;

typedef struct {
    int32_t status;              /* 0 ok; 2: a column-mean profile has no peak (the reference raises IndexError) */
    int32_t open_is_first;       /* 1: image 1 is the open field (after invert_image_order) */
    int32_t inverted[2];         /* check_inversion() flipped image 1 / 2 */
    int32_t center_warning;      /* field centre outside the central third: image centre used (the reference warns) */
    int32_t passed;
    int32_t nseg;
    int32_t pad_;
    double x_field_center;
    double profile_center_idx[2];                 /* FWXM centre of the column-mean profile of image 1 / 2 */
    double field_len[2], field_std[2];            /* len / np.std of field_values() of image 1 / 2 */
    double r_corr[EPID_VMAT_MAX_SEG], r_dev[EPID_VMAT_MAX_SEG], stdev[EPID_VMAT_MAX_SEG];
    double center_x[EPID_VMAT_MAX_SEG], center_y[EPID_VMAT_MAX_SEG], npix[EPID_VMAT_MAX_SEG];
    int32_t seg_passed[EPID_VMAT_MAX_SEG];
    double max_r_deviation, avg_abs_r_deviation, avg_r_deviation;
} epid_vmat_row;
int32_t epid_vmat_analyze(epid_ctx* ctx, const epid_batch* img1, const epid_batch* img2, const epid_vmat_params* p,
                          epid_vmat_row* rows /* [n] host */);

/* element-wise true division num / den -> a new float64 batch (`dmlc_image.array / open_image.array`, vmat.py:339; x / 0 = inf,
 * 0 / 0 = nan like numpy); both uint16 or both float64, same shape.  Each frame is first mapped by v -> sign * v + offset
 * (sign_off[2 * (2 * i + which)] = sign, [.. + 1] = offset, which = 0 num / 1 den; NULL = identity): the ground() / invert() the
 * reference applied to the images before dividing. */
int32_t epid_divide(epid_ctx* ctx, const epid_batch* num, const epid_batch* den, const double* sign_off, epid_batch** out);

/* DLG.analyze (dlg.py:32-86, 112-127): per frame and per leaf window [bottom[l]:top[l], c0:c1] the column-mean profile, the
 * inversion rule of _determine_measured_gap and the prominence of its largest peak (signed) -> measured[n][nleaf]; then
 * scipy.stats.linregress(planned, measured) per frame -> slope, intercept, dlg = intercept / slope.  uint16 frames. */
int32_t epid_dlg_analyze(epid_ctx* ctx, const epid_batch* b, int32_t nleaf, const int32_t* bottom, const int32_t* top, int32_t c0,
                         int32_t c1, const double* planned, double* measured, double* slope, double* intercept, double* dlg);

/* ----------------------------------------------------------------------------------------- whole-frame feature finders
 * GlobalSizedDiskLocator.calculate (metrics/image.py:329-354 -> find_features, metrics/utils.py:66-190) and GlobalSizedFieldLocator /
 * GlobalFieldLocator.calculate (metrics/image.py:817-897): the whole frame is binarised at the reference's rising thresholds,
 * labelled (4-connectivity for disks, 8 for fields), cleared at the border and every region is put through the detection conditions.
 * The device returns every region that passed, for every threshold, ordered like the reference visits them (threshold, then label);
 * the reference's point de-duplication / stop rule (which depends on what was found so far) is scalar work on these records in the
 * binding.  uint16 frames. */
typedef struct {
    int32_t mode;            /* 0: find_features (stretch(invert?(array)), cutoffs imin + k * step, k = 1..), 1: field locator (array as is,
                                cutoffs imin + (5 + k) * step) */
    int32_t invert;          /* mode 0: GlobalSizedDiskLocator(invert=True) */
    int32_t sample_kind;     /* 0: image.array is the integer frame; 1: image.array is the ground()-ed + normalize()-d float image of the
                                frame (Winston-Lutz images after analyze()) */
    int32_t conditions;      /* bit mask: 1 is_right_size_bb, 2 is_round, 4 is_right_circumference, 8 is_symmetric, 32 is_modest_size,
                                64 is_square, 128 is_right_square_size, 256 is_right_square_perimeter, 512 is_right_area_square
                                (metrics/features.py, winston_lutz.py:598-621) */
    double dpmm;
    double radius_mm, tolerance_mm;                              /* bb_size / tolerance of the disk conditions */
    double field_width_mm, field_height_mm, field_tolerance_mm;  /* field conditions */
    double bb_size_mm, rad_size_mm;                              /* is_modest_size / is_right_square_size */
} epid_locate_params;

typedef struct {
    int32_t threshold_index;     /* 0-based position of the threshold in the reference's sweep */
    int32_t label_root;          /* raster index of the region's first pixel (= order of skimage's labels) */
    int32_t bbox[4];             /* min_row, min_col, max_row, max_col (half-open) */
    double area, area_filled, perimeter, equivalent_diameter;
    double centroid_y, centroid_x, wcentroid_y, wcentroid_x;
} epid_region;

/* regions: [n][region_cap]; counts[n]: accepted regions per frame; flags[n]: 1 = more candidates than the device list holds at some
 * threshold, 2 = more accepted regions than region_cap */
int32_t epid_global_locate(epid_ctx* ctx, const epid_batch* frames, const epid_locate_params* p, epid_region* regions, int32_t region_cap,
                           int32_t* counts, int32_t* flags);

/* ----------------------------------------------------------------------------------------- Canny / Hough (JawOrthogonality)
 * contrib/orthogonality.py:29-50: skimage.feature.canny(stretch(image)) -> skimage.transform.hough_line -> hough_line_peaks.
 * scikit-image is absent from the build container: restated from the published algorithms, parity unpinned (oracle/edges_oracle.py).
 * epid_canny: float64 frames; weights = scipy's gaussian kernel (2 * radius + 1 doubles) for the smoothing sigma; thresholds are
 * absolute (skimage defaults for float images: 0.1 / 0.2) -> uint8 edge maps (a new batch).
 * epid_hough_line: one uint8 edge map, ntheta angles (radians) -> int32 accumulator batch [1][2 * offset + 1][ntheta], offset =
 * ceil(hypot(rows, cols)); the distance bins are linspace(-offset, offset, 2 * offset + 1).
 * epid_hough_candidates: the device half of hough_line_peaks / _prominent_peaks: maximum filter (2 d + 1 per axis, mode 'constant'),
 * pixels equal to their local maximum and > threshold (threshold < 0: 0.5 * max) as (row, col, value) triples; `filtered` keeps the
 * max-filtered accumulator on the device for epid_gather_i32 (values at arbitrary (row, col) pairs). */
int32_t epid_canny(epid_ctx* ctx, const epid_batch* in, const double* weights, int32_t radius, double low_threshold, double high_threshold,
                   epid_batch** out);
int32_t epid_hough_line(epid_ctx* ctx, const epid_batch* edges, int32_t ntheta, const double* theta, epid_batch** accum, int32_t* offset_out);
int32_t epid_hough_candidates(epid_ctx* ctx, const epid_batch* accum, int32_t min_xdistance, int32_t min_ydistance, double threshold,
                              int32_t cap, int32_t* cand_yxv, int32_t* count, int32_t* global_max, epid_batch** filtered);
int32_t epid_gather_i32(epid_ctx* ctx, const epid_batch* img, int32_t npts, const int32_t* yx, int32_t* values);

/* ----------------------------------------------------------------------------------------- multi-GPU (NCCL)
 * The batch shards by frame index with no data-path collective; the only exchange is the final gather of the
 * fixed-size per-frame result structs (SURVEY.md 8e).  id: 128-byte ncclUniqueId created by rank 0. */
int32_t epid_comm_unique_id(void* id128);
int32_t epid_comm_init(epid_ctx* ctx, int32_t nranks, int32_t rank, const void* id128);
int32_t epid_comm_destroy(epid_ctx* ctx);
/* size and rank of ctx's communicator (1, 0 until epid_comm_init succeeded): lets the host side check that the gather it is about
 * to post matches the job's world size instead of silently taking the single-rank path */
int32_t epid_comm_info(const epid_ctx* ctx, int32_t* nranks, int32_t* rank);
/* all ranks contribute bytes_per_rank bytes (host); `all` (host, nranks*bytes_per_rank) is filled on every rank */
int32_t epid_gather_results(epid_ctx* ctx, const void* local, size_t bytes_per_rank, void* all);
int32_t epid_barrier(epid_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* EPID_H */
