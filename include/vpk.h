/* vpk.h -- C ABI of the B200-native vanishing-point hot path (libvpk.so).
 *
 * Drop-in boundary for the lines -> sphere image -> CNN -> EM -> VPs path of
 * fkluger/vanishing_points_2017.  Each entry point names the reference
 * interface it replaces (file:line in the reference repository).  Plain
 * pointers and sizes only; every function returns an int status (VPK_OK == 0)
 * and never throws.  Unless a parameter is documented as a device pointer,
 * buffers are HOST memory owned by the caller; the library stages them through
 * device workspaces owned by the context.
 *
 * Ragged batches: image b owns rows offsets[b] .. offsets[b+1]-1 of the flat
 * (sumN, 4) segment / (sumN, 3) line arrays (row-major float64, the dtype the
 * reference's numpy arrays carry).
 */
#ifndef VPK_H
#define VPK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VPK_API __attribute__((visibility("default")))
#else
#define VPK_API
#endif

#define VPK_ABI_VERSION 1
#define VPK_MAX_VP 64   /* capacity of the per-image VP arrays in vpk_em_result   */
#define VPK_GRID 20     /* CNN response grid, cnn/deploy.prototxt:283-296         */
#define VPK_CNN_SIZE 500 /* CNN input side, cnn/deploy.prototxt:7                 */

/* function status */
enum { VPK_OK = 0, VPK_ERR_ARG = 1, VPK_ERR_CUDA = 2, VPK_ERR_STATE = 3, VPK_ERR_NOMEM = 4 };

/* per-image EM status (the reference returns a dict of None instead,
 * vp_localisation.py:205-206, 258-260, 402-404; no initial VP is an unhandled
 * np.vstack([]) ValueError at :165) */
enum { VPK_EM_OK = 0, VPK_EM_NO_INITIAL_VPS = 1, VPK_EM_NO_VPS_LEFT = 2, VPK_EM_CAPACITY = 3 };

/* sphere-mapping formulation (SURVEY.md section 8(a) row S1) */
enum { VPK_SPHERE_VOTES = 0,   /* pairwise-intersection vote histogram (north_star) */
       VPK_SPHERE_CURVES = 1   /* reference geometry: great-circle coverage raster   */ };

typedef struct vpk_ctx vpk_ctx;

/* ---- context ------------------------------------------------------------ */
/* replaces caffe.set_mode_gpu()/set_device(gpu_id), evaluation.py:20-21 */
VPK_API int vpk_create(int device, vpk_ctx** out);
VPK_API int vpk_destroy(vpk_ctx* ctx);
VPK_API int vpk_abi_version(void);
/* message of the last failing call on this thread ("" if none) */
VPK_API const char* vpk_last_error(void);
/* block until all work queued by this context has finished */
VPK_API int vpk_synchronize(vpk_ctx* ctx);
/* number of kernels this context has launched so far */
VPK_API int64_t vpk_launch_count(const vpk_ctx* ctx);

/* Device timestamps: vpk_mark records mark `slot` (0..3) on the context's stream; vpk_mark_elapsed returns the device
 * time from one recorded mark to another, which may belong to another context of the same device (several contexts,
 * each driven by its own host thread, keep several batches in flight; see pipeline.StreamedPipeline). */
VPK_API int vpk_mark(vpk_ctx* ctx, int32_t slot);
VPK_API int vpk_mark_elapsed(vpk_ctx* from, int32_t slot_from, vpk_ctx* to, int32_t slot_to, float* ms);

/* per-kernel device timing (CUDA events on the context's stream). */
VPK_API int vpk_profile_enable(vpk_ctx* ctx, int enable);
VPK_API int vpk_profile_reset(vpk_ctx* ctx);
/* Returns the number of distinct kernels seen; fills up to `cap` entries. */
VPK_API int vpk_profile_read(vpk_ctx* ctx, int cap, const char** names, double* total_ms, int64_t* launches);

/* ---- S0: line construction ---------------------------------------------- */
/* replaces the per-segment loop of evaluation.py:158-168 (and :199-209):
 * lines[n] = [x1,y1,1] x [x2,y2,1]. */
VPK_API int vpk_lines_from_segments(vpk_ctx* ctx, const double* segments, int64_t n, double* lines_out);

/* ---- S1: sphere mapping ------------------------------------------------- */
/* replaces sphere_mapping.sphere_line_plot (sphere_mapping.py:36-72) as
 * reached through evaluation.get_sphere_image (evaluation.py:12-14).
 *  mode VOTES : hist_out[b] (S*S uint32) = number of pairwise intersections
 *               per cell, or, with `weights` (sumN float64, nullable),
 *               whist_out[b] (S*S float32) = sum of Q.16-quantised w_i*w_j;
 *               image_out[b] = floor(255*h/max h).
 *  mode CURVES: hist_out[b] = number of lines whose sampled great circle covers
 *               the pixel; image_out[b] = floor(255*(1-(1-alpha)^k)).
 * Row 0 of every S*S plane is beta = +pi/2 (image orientation of the
 * reference canvas); column 0 is alpha = -pi/2.  Any output may be NULL. */
VPK_API int vpk_sphere_map(vpk_ctx* ctx, const double* lines, const int32_t* offsets, int32_t n_images,
                   int32_t size, int32_t mode, double alpha, const double* weights,
                   uint32_t* hist_out, float* whist_out, uint8_t* image_out);

/* ---- C0/C1: CNN --------------------------------------------------------- */
/* replaces evaluation.init_caffe (evaluation.py:17-22) + read_mean_blob
 * (:25-31).  weights[k]/biases[k], k = 0..7, are float32 host arrays in Caffe
 * blob layout for conv1..conv5, fc6, fc7, fc8_20x20 of cnn/deploy.prototxt
 * ((out, in/group, kh, kw) resp. (out, in) row-major); mean is 500*500
 * float32 or NULL (zeros). */
VPK_API int vpk_cnn_load(vpk_ctx* ctx, const float* const* weights, const float* const* biases, const float* mean);
/* replaces evaluation.caffe_forward (evaluation.py:34-38) for a batch:
 * images (n, 500, 500) uint8 -> sigout (n, 20, 20) float32; logits_out
 * (fc8 before the sigmoid) may be NULL. */
VPK_API int vpk_cnn_forward(vpk_ctx* ctx, const uint8_t* images, int32_t n_images, float* sigout, float* logits_out);

/* Diagnostics: raw copy of activation buffer `which` (VPK_CNN_BUF_*) of the last chunk (up to 1024 images) the last
 * vpk_cnn_forward ran, for its first n_images images (<= that chunk's size), in the device layout: padding rings and
 * group padding included.  Per image, row-major, NHWC:
 *   A1     bf16 (125, 125, 64)  conv1 operand: [Y, X, kwb*16 + dy*4 + dx] = image[4Y+dy, 4(X+kwb)+dx] - mean,
 *                               0 where X + kwb > 124
 *   C1     bf16 (123, 123, 96)  conv1 + ReLU + norm1
 *   A2     bf16 (65, 65, 128)   pool1, zero ring of 2; channel c of group c / 48 at (c / 48) * 64 + c % 48
 *   C2     bf16 (61, 61, 256)   conv2 + ReLU + norm2
 *   A3     bf16 (32, 32, 256)   pool2, zero ring of 1
 *   A4     bf16 (32, 32, 384)   conv3 + ReLU, zero ring of 1
 *   A5     bf16 (32, 32, 384)   conv4 + ReLU, zero ring of 1
 *   C5     bf16 (30, 30, 256)   conv5 + ReLU
 *   A6     bf16 (15, 15, 256)   pool5 = fc6 input (fc6's K runs over (y, x, c), Caffe's over (c, y, x))
 *   F6, F7 bf16 (4096)          fc6 / fc7 + ReLU
 *   LOGITS float32 (400)        fc8
 *   SIG    float32 (400)        sigmoid of fc8
 * Fails with VPK_ERR_STATE if no vpk_cnn_forward ran since the context's CNN was created or a pipeline run reused
 * the buffers, and with VPK_ERR_ARG for a bad `which` or too many images. */
enum { VPK_CNN_BUF_A1 = 0, VPK_CNN_BUF_C1, VPK_CNN_BUF_A2, VPK_CNN_BUF_C2, VPK_CNN_BUF_A3, VPK_CNN_BUF_A4, VPK_CNN_BUF_A5,
       VPK_CNN_BUF_C5, VPK_CNN_BUF_A6, VPK_CNN_BUF_F6, VPK_CNN_BUF_F7, VPK_CNN_BUF_LOGITS, VPK_CNN_BUF_SIG, VPK_CNN_NBUF };
VPK_API int vpk_cnn_debug_fetch(vpk_ctx* ctx, int32_t which, int32_t n_images, void* out);

/* Diagnostics: one plain GEMM out = act(a * b^T + bias) through the tcgen05 kernel every
 * CNN layer uses.  a (m,k) and b (n,k) are bf16 bit patterns, out (m,n) float32;
 * k % 64 == 0, bn % 16 == 0, 16 <= bn <= 256, n % bn == 0.  ksplit > 1: the K range is dealt to
 * ksplit CTAs per output tile and a finishing pass adds the partial tiles in order (how the fully
 * connected layers run for batches of up to 256 images); ksplit = 1: one CTA per tile. */
VPK_API int vpk_debug_gemm(vpk_ctx* ctx, int32_t m, int32_t n, int32_t k, const uint16_t* a, const uint16_t* b,
                           const float* bias, int32_t relu, int32_t bn, int32_t ksplit, float* out);

/* ---- E0..E12: EM --------------------------------------------------------- */
/* keyword arguments of vp_localisation.expectation_maximisation
 * (vp_localisation.py:168-172), same names and defaults */
typedef struct vpk_em_config {
    int32_t num_iter;           /* 100  */
    int32_t num_init_vp;        /* 25   */
    int32_t split_merge_freq;   /* 10   */
    int32_t num_min_lines;      /* 3    */
    int32_t do_merge;           /* 1    */
    int32_t do_split;           /* 1    */
    int32_t do_iterations;      /* 1    */
    int32_t use_weights;        /* 1    */
    double wbias;               /* 1    */
    double merge_thresh;        /* 1e-3 */
    double outlier_thresh;      /* 1.96^2 */
    double final_convergence;   /* 5e-3 */
    double s_thresh;            /* 1e-200 */
} vpk_em_config;
VPK_API void vpk_em_default_config(vpk_em_config* cfg);

/* the reference's result dict (vp_localisation.py:441-442), flattened.
 * All pointers are caller-owned host arrays; decision_metric may be NULL. */
typedef struct vpk_em_result {
    int32_t* status;          /* (B)               VPK_EM_*                         */
    int32_t* n_vp;            /* (B)               rows of 'vp'                     */
    int32_t* iterations;      /* (B)               'iterations'                     */
    double* vp;               /* (B, VPK_MAX_VP, 3) 'vp'                            */
    double* sigma;            /* (B, VPK_MAX_VP)    'sigma'                         */
    int32_t* counts;          /* (B, VPK_MAX_VP)    'counts'                        */
    double* counts_weighted;  /* (B, VPK_MAX_VP)    'counts_weighted'               */
    int32_t* vp_assoc;        /* (sumN)             'vp_assoc' (-1 = outlier)       */
    double* decision_metric;  /* (VPK_MAX_VP*sumN) or NULL: image b's (n_vp, N_b)
                                 row-major block starts at VPK_MAX_VP*offsets[b]   */
} vpk_em_result;

/* replaces vp_localisation.expectation_maximisation (vp_localisation.py:
 * 168-450) called per image by evaluation.run_em_single (evaluation.py:
 * 344-347), for a ragged batch.  lines: (sumN,3) (normalised internally, the
 * caller's array is not mutated); segments: (sumN,4); responses: (B,20,20)
 * float64; sphere_images: (B,S,S) uint8; init_vp/init_vp_offsets: optional
 * per-image initial VPs (the reference's init_vp kwarg) or NULL. */
VPK_API int vpk_em(vpk_ctx* ctx, const double* lines, const double* segments, const int32_t* offsets,
           int32_t n_images, const double* responses, const uint8_t* sphere_images, int32_t size,
           const double* init_vp, const int32_t* init_vp_offsets,
           const vpk_em_config* cfg, vpk_em_result* out);

/* 'distribution' of the reference's result dict (vp_localisation.py:441-442): the PDF namedtuple of
 * probability_functions.py:5 that calc_probabilities (:99-120) returns for the LAST E-step, for image `image` of the
 * last vpk_em / vpk_pipeline_run call of this context.  Evaluated on the device from the planes that superstep left
 * in the EM workspace, so it must be asked for before the next EM call and only for batches that ran in one
 * workspace wave.  n_vp / n_lines: the image's 'vp' rows and lines (checked).  Caller-allocated float64 arrays:
 * p_v (n_vp), p_lv (n_lines, n_vp), p_vl (n_vp, n_lines), p_l (n_lines), lvsq (n_lines, n_vp), angles (n_vp, 2). */
VPK_API int vpk_em_distribution(vpk_ctx* ctx, int32_t image, int32_t n_vp, int32_t n_lines, double* p_v, double* p_lv,
                                double* p_vl, double* p_l, double* lvsq, double* angles);

/* Diagnostics: raw copy of buffer `which` (VPK_EM_BUF_*) of image `image`'s EM workspace as the last vpk_em /
 * vpk_pipeline_run call of this context left it, in the device layout (float64).  N = the image's lines, M = its
 * 'vp' rows (n_vp); kMP = 32, kMPS = 36 and the layouts are those of csrc/em_core.cuh:
 *   LSIM     ceil(N/64)*64*N   similarity matrix of em_pair: 64-column slabs of N x 64 doubles, element (j, k) at
 *                              ((k/64)*N + j)*64 + ((k%64) ^ ((j&3)<<2))   (lsim_index)
 *   COLSUM   N                 column sums of lsim (em_pair; 0 with use_weights = 0, set by em_init)
 *   LWEIGHT  N                 kNN line weights (em_pair; 1 with use_weights = 0, set by em_init)
 *   LVSQ     M*N               (M, N) row-major planes of the last superstep's em_estep: lvsq, p(v|l)
 *   PVL      M*N
 *   W        M*N               (M, N) weight matrix of the last superstep's em_wmat (= the decision metric)
 *   WT       ceil(M/32)*N*36   em_wmat's operand p(v|l)*lweight: pass p (rows 32p..32p+31) at p*N*36, line n of the
 *                              pass at n*s, s = 8*t+4, t = ceil(min(M-32p, 32)/8); rows M..8t-1 of the last pass are
 *                              zeros, the last 4 doubles of a line are never written   (wt_index)
 *   ESTEP    5*M               the E-step constants of those planes, rows pv | vx | vy | inv2s | coef
 * The planes (LVSQ .. ESTEP) belong to the image's final hypotheses: an image that finished with VPK_EM_OK ends in
 * the final-count phase (vp_localisation.py:415-437), which asks for a new E-step and weight matrix on the
 * remaining 'vp' rows each time it drops one and finishes without another, so M is n_vp, and pv .. coef are
 * evaluated on 'vp' and 'sigma' (vx = vp0/vp2, vy = vp1/vp2, inv2s = 1/(2 sigma), coef = 1/sqrt(2 pi sigma)).
 * count (may be NULL) receives the buffer's size in doubles; out = NULL only asks for it.
 * Fails with VPK_ERR_STATE before any EM call, after a batch that ran in more than one workspace wave, for LSIM
 * of a batch run with use_weights = 0 (no pair pass), and for the planes of an image whose status is not
 * VPK_EM_OK; with VPK_ERR_ARG for a bad `which`, an image not in the last batch or capacity < the size. */
enum { VPK_EM_BUF_LSIM = 0, VPK_EM_BUF_COLSUM, VPK_EM_BUF_LWEIGHT, VPK_EM_BUF_LVSQ, VPK_EM_BUF_PVL, VPK_EM_BUF_W,
       VPK_EM_BUF_WT, VPK_EM_BUF_ESTEP, VPK_EM_NBUF };
VPK_API int vpk_em_debug_fetch(vpk_ctx* ctx, int32_t image, int32_t which, double* out, int64_t capacity, int64_t* count);

/* Profiling runs only (vpk_profile_enable): accumulated algorithmic work of the weight-matrix
 * products (vp_localisation.py:515-524) since the last reset: out[0] = bytes of similarity
 * matrix consumed (8 N^2 per product), out[1] = flops (2 M N^2 per product), out[2] = number
 * of per-image products, out[3] = supersteps, out[4] = algorithmic bytes of the POST kernel
 * (the planes w, lvsq, pvl of every active image once per superstep: 8 (3 M N + 5 N)),
 * out[5] = of the E-step kernel (same figure: three planes written). */
VPK_API int vpk_em_stats(vpk_ctx* ctx, uint64_t out[6], int reset);
/* Profiling runs only: SM cycles the leading CTA of every image's cluster spent per phase of the fused
 * EM kernel since the last reset: out[0] E-step, [1] barrier after E, [2] weight-matrix product, [3] barrier
 * after W, [4] M-step sums spread over the cluster, [5] POST (state machine), [6] barrier + state mirror. */
VPK_API int vpk_em_phase_cycles(vpk_ctx* ctx, uint64_t out[8], int reset);

/* ---- whole path ---------------------------------------------------------- */
/* example.py:37-39 / benchmark.py:59-66 for a ragged batch, without the
 * per-image pickles: segments -> lines -> sphere image -> CNN -> EM, all
 * intermediates staying in HBM.
 *   vpk_pipeline_upload : host segments -> device-resident batch (H2D).
 *   vpk_pipeline_run    : run the path on the resident batch (no H2D).
 *   vpk_pipeline_fetch  : copy the results to host arrays (D2H).
 *   vpk_pipeline_host   : the three in sequence (the end-to-end call).      */
VPK_API int vpk_pipeline_upload(vpk_ctx* ctx, const double* segments, const int32_t* offsets, int32_t n_images);
VPK_API int vpk_pipeline_run(vpk_ctx* ctx, int32_t size, int32_t sphere_mode, double alpha, const vpk_em_config* cfg);
VPK_API int vpk_pipeline_fetch(vpk_ctx* ctx, vpk_em_result* out, float* sigout /* (B,20,20) or NULL */,
                       uint8_t* sphere_images /* (B,S,S) or NULL */);
VPK_API int vpk_pipeline_host(vpk_ctx* ctx, const double* segments, const int32_t* offsets, int32_t n_images,
                      int32_t size, int32_t sphere_mode, double alpha, const vpk_em_config* cfg,
                      vpk_em_result* out, float* sigout, uint8_t* sphere_images);
/* ---- N2: raw LSD output -> normalised segments (+ lines) ---------------------- */
/* The normalisation evaluation.detect_lsd_lines applies to lsd.detect_line_segments' rows (reference
 * evaluation.py:227-251) and the line construction of evaluation.py:158-168, for a ragged batch on the
 * device.  lsd: (sum N, ncols) float64 rows x1, y1, x2, y2, [width, p, -log10 NFA] in pixels
 * (ncols >= 4; 7 for LSD's own output); widths / heights: image sizes in pixels.  segments_out (sum N, 4):
 * origin at the image centre, divided by max(w, h) / 2, y up -- bit-identical to the numpy expressions;
 * lines_out (sum N, 3) = [x1,y1,1] x [x2,y2,1] or NULL; nfa_out (sum N) = column 6 or NULL. */
VPK_API int vpk_segments_from_lsd(vpk_ctx* ctx, const double* lsd, int32_t ncols, const int32_t* offsets, const int32_t* widths,
                                  const int32_t* heights, int32_t n_images, double* segments_out, double* lines_out,
                                  double* nfa_out);
/* vpk_pipeline_upload for raw LSD rows: they are normalised on the device into the resident batch. */
VPK_API int vpk_pipeline_upload_lsd(vpk_ctx* ctx, const double* lsd, int32_t ncols, const int32_t* offsets,
                                    const int32_t* widths, const int32_t* heights, int32_t n_images);

/* ---- N4: the LSD line segment detector ----------------------------------------- */
/* lsd.detect_line_segments (lsdpython/lsd.pyx:17-18, LSD 1.6's LineSegmentDetection) as evaluation.detect_lsd_lines
 * calls it (reference evaluation.py:227-251), on the device for a ragged batch of grayscale images. */
typedef struct vpk_lsd_config {
    double scale;        /* 0.8  */
    double sigma_scale;  /* 0.6  */
    double quant;        /* 2.0  */
    double ang_th;       /* 22.5 */
    double log_eps;      /* 0.0  */
    double density_th;   /* 0.7  */
    int32_t n_bins;      /* 1024 */
} vpk_lsd_config;
VPK_API void vpk_lsd_default_config(vpk_lsd_config* cfg);
/* pixel types of vpk_lsd's images */
enum { VPK_PIX_U8 = 0, VPK_PIX_F64 = 1 };
/* images: host array of gray values of type `dtype`; image b is the row-major heights[b] x widths[b] block that
 * starts at element pixel_offsets[b] (pixel_offsets has B+1 entries, pixel_offsets[b+1] - pixel_offsets[b] =
 * widths[b] * heights[b]).  Runs the detector, keeps the rows on the device and writes the number of segments
 * of every image to counts_out (B).  A sampled side (ceil(side * scale)) must be below 65536. */
VPK_API int vpk_lsd(vpk_ctx* ctx, const void* images, int32_t dtype, const int64_t* pixel_offsets, const int32_t* widths,
                    const int32_t* heights, int32_t n_images, const vpk_lsd_config* cfg, int32_t* counts_out);
/* rows of the last vpk_lsd call: (sum counts, 7) float64 x1, y1, x2, y2, width, p, -log10(NFA) in pixels of the
 * input images, image after image, each image's rows in LSD's own output order. */
VPK_API int vpk_lsd_fetch(vpk_ctx* ctx, double* rows_out);
/* vpk_lsd followed by vpk_pipeline_upload_lsd's normalisation, on the device: the rows never leave it; only the
 * per-image counts come back (counts_out (B), may be NULL). */
VPK_API int vpk_pipeline_upload_images(vpk_ctx* ctx, const void* images, int32_t dtype, const int64_t* pixel_offsets,
                                       const int32_t* widths, const int32_t* heights, int32_t n_images,
                                       const vpk_lsd_config* cfg, int32_t* counts_out);

/* ---- N5: photo preparation in front of LSD ------------------------------------ */
/* The head of evaluation.create_data_pickles (reference evaluation.py:139-154): `convert ... -resize TxT` (here
 * OpenCV 4.13's INTER_AREA rule in float64), the 8-bit RGB read back, skimage.color.rgb2gray; DESIGN.md section 4.7.
 * Photos: host array of uint8 RGB, photo b the row-major heights[b] x widths[b] x 3 block starting at byte
 * byte_offsets[b] (B+1 entries, byte_offsets[b+1] - byte_offsets[b] = 3 * widths[b] * heights[b]).  target_size <= 0:
 * no resize; otherwise s = target_size / max(w, h) and, if s < 1, W' = max(1, rint(w s)), H' = max(1, rint(h s)).
 * Photos are never enlarged. */
/* the prepared size (W', H') of one w x h photo; host only, needs no device or context */
VPK_API int vpk_prepared_size(int32_t w, int32_t h, int32_t target_size, int32_t* out_w, int32_t* out_h);
/* gray_out: the reference's datum['image'], rgb2gray's float64 output in [0, 1], photo after photo, each a row-major
 * out_heights[b] x out_widths[b] plane (sum W' H' doubles, see vpk_prepared_size); out_widths / out_heights (B). */
VPK_API int vpk_prepare_images(vpk_ctx* ctx, const uint8_t* rgb, const int64_t* byte_offsets, const int32_t* widths,
                               const int32_t* heights, int32_t n_images, int32_t target_size, int32_t* out_widths,
                               int32_t* out_heights, double* gray_out);
/* vpk_prepare_images followed by vpk_pipeline_upload_images on the prepared planes times 255 (detect_lsd_lines' scaling,
 * evaluation.py:229-231), on the device: the planes are written where the detector reads them, and the detector's
 * frames are the prepared sizes.  Only the per-image counts and prepared sizes come back (each may be NULL);
 * vpk_lsd_fetch returns the rows.  A sampled prepared side (ceil(side * scale)) must be below 65536. */
VPK_API int vpk_pipeline_upload_photos(vpk_ctx* ctx, const uint8_t* rgb, const int64_t* byte_offsets, const int32_t* widths,
                                       const int32_t* heights, int32_t n_images, int32_t target_size,
                                       const vpk_lsd_config* cfg, int32_t* counts_out, int32_t* out_widths,
                                       int32_t* out_heights);

/* ---- N6: JPEG decoding in front of photo preparation ---------------------------- */
/* The read of the dataset's JPEG files by `convert` (reference evaluation.py:142-143), on the device and bit for bit
 * with libjpeg-turbo 3.1's default decode (islow IDCT, fancy upsampling, jdcolor.c's YCbCr -> RGB); DESIGN.md
 * section 4.8.  Decoded: baseline and extended sequential Huffman JPEG (SOF0 / SOF1), 8-bit, one interleaved scan,
 * 3 components in YCbCr or 1 component (gray), sampling factors up to 4 with integer ratios, restart intervals.
 * EXIF orientation is ignored (the stored orientation, as `convert` without -auto-orient sees it).
 * Files: host array `data`, file b the byte_offsets[b] .. byte_offsets[b+1] bytes (B+1 non-decreasing entries). */
enum {
    VPK_JPEG_OK = 0,
    VPK_JPEG_PROGRESSIVE = 1,   /* SOF2 */
    VPK_JPEG_ARITHMETIC = 2,    /* SOF9..SOF15, DAC */
    VPK_JPEG_PRECISION = 3,     /* not 8-bit samples */
    VPK_JPEG_COLOR = 4,         /* CMYK / YCCK (4 components), or RGB (Adobe transform 0, or component IDs 'R','G','B') */
    VPK_JPEG_LAYOUT = 5,        /* 2 components, a scan without every component (multi-scan), fractional sampling, DNL */
    VPK_JPEG_MALFORMED = 6,     /* markers the parser cannot follow: truncated or overrunning segments, missing tables */
    VPK_JPEG_LOSSLESS = 7,      /* lossless or hierarchical process (SOF3, SOF5..SOF7, DHP, EXP) */
    VPK_JPEG_CORRUPT = 8        /* status after decoding: the entropy-coded data is inconsistent (ends before the last
                                 * block, a code not in its table, a run past coefficient 63, data left over, RSTn out
                                 * of sequence); the photo's pixels are unspecified but deterministic */
};
/* Reads the markers of every file up to its SOS segment, never the entropy-coded data; host only, needs no device or
 * context.  widths / heights / components (B, each may be NULL) receive the frame's size and component count (0
 * unless the parser read a SOF0 / SOF1 frame header); support (B, may be NULL) VPK_JPEG_OK or the reason a file is refused. */
VPK_API int vpk_jpeg_info(const uint8_t* data, const int64_t* byte_offsets, int32_t n, int32_t* widths, int32_t* heights,
                          int32_t* components, int32_t* support);
/* Decodes every file on the device.  pixels_out: photo after photo, row-major height x width x components bytes (RGB,
 * or gray for 1 component); status_out (B): VPK_JPEG_OK or VPK_JPEG_CORRUPT.  Fails with VPK_ERR_ARG before any
 * device work, naming the first refused file and its reason. */
VPK_API int vpk_decode_jpegs(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n, uint8_t* pixels_out,
                             int32_t* status_out);
/* vpk_decode_jpegs followed by vpk_pipeline_upload_photos on the decoded photos, on the device: only the files cross
 * PCIe, the decoder writes the RGB photos where the preparation kernel reads them.  counts_out / out_widths /
 * out_heights as vpk_pipeline_upload_photos, status_out (B) as vpk_decode_jpegs (each may be NULL; a CORRUPT photo's
 * rows come from its unspecified pixels).  A refused file or a 1-component file (gray photos cannot be prepared)
 * fails the call with VPK_ERR_ARG, naming its index and reason. */
VPK_API int vpk_pipeline_upload_jpegs(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n,
                                      int32_t target_size, const vpk_lsd_config* cfg, int32_t* counts_out,
                                      int32_t* out_widths, int32_t* out_heights, int32_t* status_out);
/* Decoder statistics of the last decode on this context: out[0] subsequences, out[1] subsequences re-decoded after
 * their first decode (the synchronisation work), out[2] the most synchronisation rounds inside one CTA, out[3] extra
 * launches across CTAs.  out[1] and out[2] are counted only while profiling is enabled (vpk_profile_enable), 0
 * otherwise.  Fails with VPK_ERR_STATE before any decode. */
VPK_API int vpk_jpeg_stats(vpk_ctx* ctx, int64_t* out);

/* ---- N7: PNG decoding in front of photo preparation ----------------------------- */
/* The read of PNG files (reference evaluation.py:142-143: the dataset's *.png files, and the 8-bit PNG every photo
 * is written to and read back), on the device and bit for bit with libpng's decode; DESIGN.md section 4.9.
 * Decoded: 8-bit and lower files, non-interlaced or Adam7, any split of the zlib stream over IDAT chunks: gray (colour
 * type 0; 1, 2, 4 or 8 bits, scaled to 0..255 as libpng's expand does) and gray + alpha (4) to gray; RGB (2), palette
 * (3; 1 to 8 bits, an index beyond PLTE gives black) and RGBA (6) to RGB.  Alpha is dropped, not composited; tRNS,
 * gAMA, iCCP, sRGB and eXIf are ignored (no colour management, no EXIF orientation); an APNG decodes as its default
 * image.  Files: host array `data`, file b the byte_offsets[b] .. byte_offsets[b+1] bytes (B+1 non-decreasing entries). */
enum {
    VPK_PNG_OK = 0,
    VPK_PNG_NOT_PNG = 1,        /* no PNG signature (a JPEG passed by mistake, ...) */
    VPK_PNG_DEPTH = 2,          /* 16-bit samples */
    VPK_PNG_MALFORMED = 3,      /* a truncated or overrunning chunk, IHDR values PNG forbids, chunks out of order or
                                 * IDAT chunks that are not consecutive, no PLTE for colour type 3, an unknown critical
                                 * chunk, a bad length or CRC on IHDR or on the PLTE of a palette file (elsewhere PLTE is
                                 * ignored), no IDAT or IEND, an invalid zlib header (a method other than deflate, a
                                 * window above 32 K, a preset dictionary, a bad check) */
    VPK_PNG_CORRUPT = 4         /* status after decoding: an IDAT CRC mismatch, an Adler-32 mismatch, a stream that ends
                                 * before the last row, a filter byte above 4, an invalid deflate stream (zlib's
                                 * verdicts, up to the last row and the end of the stream right after it), running out of
                                 * IDAT data; the file's pixels are unspecified but deterministic.  Data after the last
                                 * row is not an error, nor are zlib's errors past it (libpng warns and decodes the
                                 * image) */
};
/* Walks the chunks of every file (chunk headers, IHDR and PLTE; never the IDAT payloads); host only, needs no device
 * or context.  widths / heights / color_types (B, each may be NULL) receive IHDR's values (0 unless IHDR was read);
 * support (B, may be NULL) VPK_PNG_OK or the reason a file is refused. */
VPK_API int vpk_png_info(const uint8_t* data, const int64_t* byte_offsets, int32_t n, int32_t* widths, int32_t* heights,
                         int32_t* color_types, int32_t* support);
/* Decodes every file on the device.  pixels_out: file after file, row-major height x width x channels bytes (RGB for
 * colour types 2, 3 and 6, gray for 0 and 4); status_out (B): VPK_PNG_OK or VPK_PNG_CORRUPT.  Fails with VPK_ERR_ARG
 * before any device work, naming the first refused file and its reason. */
VPK_API int vpk_decode_pngs(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n, uint8_t* pixels_out,
                            int32_t* status_out);
/* vpk_decode_pngs followed by vpk_pipeline_upload_photos on the decoded photos, on the device: only the files cross
 * PCIe, the decoder writes the RGB photos where the preparation kernel reads them.  counts_out / out_widths /
 * out_heights as vpk_pipeline_upload_photos, status_out (B) as vpk_decode_pngs (each may be NULL; a CORRUPT file's
 * rows come from its unspecified pixels).  A refused file or a gray one (colour type 0 or 4: gray photos cannot be
 * prepared) fails the call with VPK_ERR_ARG, naming its index and reason. */
VPK_API int vpk_pipeline_upload_pngs(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n,
                                     int32_t target_size, const vpk_lsd_config* cfg, int32_t* counts_out,
                                     int32_t* out_widths, int32_t* out_heights, int32_t* status_out);

/* ---- N8: mixed batches of files in front of photo preparation -------------------- */
/* The dataset listing of the reference's evaluation.get_data_list (*.jpg, *.png and *.pgm in one dataset) in one
 * call; DESIGN.md section 4.10.  Each file's format comes from its leading bytes: JPEG (FF D8 FF), PNG (the PNG
 * signature) or netpbm ("P1" .. "P7"), of which binary PGM (P5) with maxval 255 is taken; its payload is the photo.
 * JPEG and PNG files are decoded as vpk_decode_jpegs / vpk_decode_pngs do.  A file is gray when its decoded photo has
 * one channel (a 1-component JPEG, PNG colour type 0 or 4, a PGM), else RGB.  Gray photos are prepared as the
 * reference prepares them: skimage 0.12's rgb2gray returns a 2-D input unchanged, so datum['image'] is the resized
 * uint8 plane, and detect_lsd_lines multiplies it by 255 only if its maximum is at most 1.
 * Files: host array `data`, file b the byte_offsets[b] .. byte_offsets[b+1] bytes (B+1 non-decreasing entries). */
enum { VPK_FILE_UNKNOWN = 0, VPK_FILE_JPEG = 1, VPK_FILE_PNG = 2, VPK_FILE_PGM = 3 };
enum {
    VPK_PGM_OK = 0,
    VPK_PGM_ASCII = 1,          /* ASCII PGM (P2) */
    VPK_PGM_BITMAP = 2,         /* PBM bitmaps (P1, P4) */
    VPK_PGM_PAM = 3,            /* PAM (P7) */
    VPK_PGM_PPM = 4,            /* colour netpbm (P3, P6): not a format the reference lists */
    VPK_PGM_MAXVAL = 5,         /* maxval below 255 (the reference's rescale by ImageMagick is not pinned) */
    VPK_PGM_DEPTH = 6,          /* maxval above 255: 16-bit samples */
    VPK_PGM_MALFORMED = 7       /* a header that is not magic, width, height, maxval separated by whitespace and '#'
                                 * comments with exactly one whitespace byte before the payload, or a truncated
                                 * payload (bytes after the payload are allowed) */
};
/* Sniffs and parses every file (headers only); host only, needs no device or context.  formats (B) VPK_FILE_*;
 * widths / heights (B) the photo's size (0 where the header does not give it); channels (B) 3 for RGB, 1 for gray, 0
 * where unknown; support (B) the format's own reason code (VPK_JPEG_*, VPK_PNG_*, VPK_PGM_*; 0: taken), 1 for a file
 * of unknown format.  Each may be NULL. */
VPK_API int vpk_file_info(const uint8_t* data, const int64_t* byte_offsets, int32_t n, int32_t* formats, int32_t* widths,
                          int32_t* heights, int32_t* channels, int32_t* support);
/* Decodes every file on the device, each format's files by its decoder.  pixels_out: photo after photo, row-major
 * height x width x channels bytes (RGB or gray); status_out (B): the format's own OK / CORRUPT code (VPK_JPEG_*,
 * VPK_PNG_*; a PGM is always VPK_PGM_OK).  A refused or unknown file fails the call with VPK_ERR_ARG before any device
 * work, naming its index, its format and the reason. */
VPK_API int vpk_decode_files(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n, uint8_t* pixels_out,
                             int32_t* status_out);
/* The reference's datum['image'] of every file as float64, photo after photo, each a row-major out_heights[b] x
 * out_widths[b] plane (see vpk_prepared_size): rgb2gray in [0, 1] for RGB photos (vpk_prepare_images), the resized
 * uint8 values for gray ones.  Refused files as vpk_decode_files. */
VPK_API int vpk_prepare_files(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n, int32_t target_size,
                              int32_t* out_widths, int32_t* out_heights, double* planes_out);
/* vpk_prepare_files followed by vpk_pipeline_upload_images on detect_lsd_lines' input (the plane times 255 when its
 * maximum is at most 1, decided on the device), in input order: only the files cross PCIe, each once.  counts_out /
 * out_widths / out_heights as vpk_pipeline_upload_photos, status_out (B) as vpk_decode_files (each may be NULL).
 * Refused files as vpk_decode_files. */
VPK_API int vpk_pipeline_upload_files(vpk_ctx* ctx, const uint8_t* data, const int64_t* byte_offsets, int32_t n,
                                      int32_t target_size, const vpk_lsd_config* cfg, int32_t* counts_out,
                                      int32_t* out_widths, int32_t* out_heights, int32_t* status_out);

/* ---- N1: horizon line and orthogonal VP triplet --------------------------- */
/* calc_horizon.calculate_horizon_and_ortho_vp(em_result, maxbest=10, theta_vmin=pi/10, theta_z=pi/4)
 * (reference calc_horizon.py:19-225; callers example.py:65, benchmark.py:233) for a batch of EM
 * results.  vp (B, VPK_MAX_VP, 3) float64, counts (B, VPK_MAX_VP) int32 and n_vp (B) int32 are laid
 * out as vpk_em writes them (an image without VPs has n_vp = 0 and gets the reference's default
 * horizon, calc_horizon.py:207-212).  points (B, 5, 3) float64 receives the reference's return
 * values hP1, hP2, zVP, hVP1, hVP2 in that order; best_combo (B, 3) int32 the indices of the chosen
 * VPs (two entries and -1 when fewer than three VPs take part).
 * Optional (row N4, the evaluation of benchmark.py:247-253): with true_horizons (B,3) homogeneous
 * ground-truth horizon lines, scales (B) and heights (B) (benchmark.py's `scale` and `imageHeight`),
 * errors (B) receives max(|hP1.y - thP1.y|, |hP2.y - thP2.y|) / 2 * scale / imageHeight; all four NULL
 * otherwise. */
VPK_API int vpk_horizon(vpk_ctx* ctx, const double* vp, const int32_t* counts, const int32_t* n_vp, int32_t n_images,
                        int32_t maxbest, double theta_vmin, double theta_z, const double* true_horizons,
                        const double* scales, const double* heights, double* points, int32_t* best_combo, double* errors);
/* The same on the device-resident EM result of the last vpk_pipeline_run (no host round trip of the
 * EM result; only the 5 points + 3 indices per image come back). */
VPK_API int vpk_pipeline_horizon(vpk_ctx* ctx, int32_t maxbest, double theta_vmin, double theta_z,
                                 const double* true_horizons, const double* scales, const double* heights, double* points,
                                 int32_t* best_combo, double* errors);

/* ---- N9: pipeline input and output in CUDA memory ------------------------------- */
/* The entry points above in a form for data that is already on the device (photos decoded by another GPU decoder,
 * gray planes, segments from a model) and for results consumed there; DESIGN.md section 4.11.  The data pointers
 * below are caller-owned DEVICE (or managed) memory of the context's device; every other pointer is host memory.
 * Interop: the library links the CUDA runtime statically and runs on the device's primary context (cudaSetDevice),
 * the one PyTorch and the CUDA runtime of other libraries use, so their device pointers and stream handles are valid
 * here.  Strides are in ELEMENTS, non-negative (0 repeats an element), so views (crops, column slices, a CHW tensor
 * permuted to HWC) need no copy; no element outside ptr + sum (extent - 1) * stride is read.
 * Ordering: `stream` is the caller's stream (a cudaStream_t; 0: the legacy default stream).  Each call's device work
 * runs after the work queued on `stream` before the call (an event recorded there, waited for on the context's
 * stream), and device outputs are ordered before the work queued on `stream` after the call (the reverse event).
 * The upload calls still synchronise the host with the context's stream before they return (they return the
 * per-image counts and plan the ragged batch on the host), so their inputs may be reused once they return;
 * vpk_pipeline_fetch_device and vpk_pipeline_horizon_device never block the host.
 * Validation happens before any device work: a pointer that is host memory, memory of another device or not a CUDA
 * pointer, a negative stride, a zero size or a channel count other than 1 or 3 fails with VPK_ERR_ARG, naming the
 * image. */
/* vpk_pipeline_upload from device segments: (sum N, 4) float64, element (n, k) at segments[n * row_stride + k * col_stride];
 * offsets (B+1) are host memory. */
VPK_API int vpk_pipeline_upload_device(vpk_ctx* ctx, const double* segments, int64_t row_stride, int64_t col_stride,
                                       const int32_t* offsets, int32_t n_images, void* stream);
/* vpk_pipeline_upload_images from device gray images of one dtype (VPK_PIX_U8 or VPK_PIX_F64): images (B) device
 * pointers, image b's pixel (y, x) at images[b][y * strides[2b] + x * strides[2b+1]], widths[b] x heights[b]. */
VPK_API int vpk_pipeline_upload_images_device(vpk_ctx* ctx, const void* const* images, const int64_t* strides,
                                              const int32_t* widths, const int32_t* heights, int32_t n_images, int32_t dtype,
                                              const vpk_lsd_config* cfg, void* stream, int32_t* counts_out);
/* vpk_pipeline_upload_photos from device uint8 photos: photo b's sample (y, x, c) at photos[b][y * strides[3b] +
 * x * strides[3b+1] + c * strides[3b+2]], widths[b] x heights[b] x channels[b].  A 3-channel photo is prepared as by
 * vpk_pipeline_upload_photos, a 1-channel photo as a gray file by vpk_pipeline_upload_files (the resized uint8 plane,
 * times 255 only if its maximum is at most 1).  counts_out / out_widths / out_heights as vpk_pipeline_upload_photos. */
VPK_API int vpk_pipeline_upload_photos_device(vpk_ctx* ctx, const uint8_t* const* photos, const int64_t* strides,
                                              const int32_t* widths, const int32_t* heights, const int32_t* channels,
                                              int32_t n_images, int32_t target_size, const vpk_lsd_config* cfg, void* stream,
                                              int32_t* counts_out, int32_t* out_widths, int32_t* out_heights);
/* vpk_pipeline_fetch into device buffers of exactly its layout: the vpk_em_result fields (decision_metric ignored),
 * sigout (B,20,20) float32 and sphere_images (B,S,S) uint8 are device pointers; out, sigout and sphere_images may be
 * NULL.  Asynchronous. */
VPK_API int vpk_pipeline_fetch_device(vpk_ctx* ctx, vpk_em_result* out, float* sigout, uint8_t* sphere_images, void* stream);
/* vpk_pipeline_horizon into device arrays points (B,5,3), best_combo (B,3), errors (B) or NULL; with errors, the
 * contiguous true_horizons (B,3), scales (B) and heights (B) are device arrays too.  Asynchronous. */
VPK_API int vpk_pipeline_horizon_device(vpk_ctx* ctx, int32_t maxbest, double theta_vmin, double theta_z,
                                        const double* true_horizons, const double* scales, const double* heights,
                                        double* points, int32_t* best_combo, double* errors, void* stream);

/* device time of the last vpk_pipeline_run per stage: [lines+sphere, cnn, em, total] ms */
VPK_API int vpk_pipeline_stage_ms(vpk_ctx* ctx, float ms[4]);

#ifdef __cplusplus
}
#endif
#endif /* VPK_H */
