/*
 * slowflow_gpu.h -- C ABI of libslowflow_gpu.so: the B200 (sm_100a) implementation of Slow Flow's
 * variational energy-minimisation hot path.
 *
 * The library is a drop-in for ONE path of JJanai/slowflow and nothing else.  Every entry point
 * cites the reference interface it replaces (paths relative to the reference root).  All
 * signatures are plain C: pointers, sizes, PODs -- no CUDA, torch or C++ types.
 *
 *   1. Legacy drop-in:  variational() / variational_params_default() with the reference's exact
 *      signatures (epic_flow_extended/variational.h:27,30), callers adaptiveFR.cpp:574 and
 *      epicflow.cpp:127.  Host buffers in, host buffers out, abort-on-error like the reference.
 *   2. Handle API (sfgpu_*): re-entrant, one context per host thread / device / stream, int status
 *      codes + sfgpu_last_error().  Adds the multi-frame entry (Variational_MT::variational,
 *      epic_flow_extended/variational_mt.h:37, callers slow_flow.cpp:888,1023), device-resident
 *      and pipelined-sequence variants for the sharded driver, and operator-level twins of
 *      variational_aux.h:12-29 / solver.h:11 for parity tests.
 *
 * There is NO CPU fallback: every compute entry fails (status != 0, or abort for the legacy entry)
 * when no CUDA device is usable.
 */
#ifndef SLOWFLOW_GPU_H_
#define SLOWFLOW_GPU_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- containers: identical layout to epic_flow_extended/image.h:17-34.  If the reference's
 * image.h was included first its definitions are used (same names, same fields).  Every sfgpu_* entry that takes them
 * returns SFGPU_ERR_ARG, before it touches the device or any buffer, when an argument has NULL data, width or height
 * < 1, a stride other than ceil4(width), colour planes that are not contiguous, or another geometry than the call's. ---- */
#ifndef __IMAGE_H_
typedef struct image_s {
    int width;   /* valid columns */
    int height;  /* rows */
    int stride;  /* floats per row = ceil4(width) (image.c:25) */
    float *data; /* 16-byte aligned, row-major */
} image_t;

typedef struct color_image_s {
    int width, height, stride;
    float *c1, *c2, *c3; /* planar; c2 = c1 + stride*height, c3 = c2 + stride*height (image.c:80-87) */
} color_image_t;
#endif

/* ---- two-frame parameters: identical to epic_flow_extended/variational.h:15-24 ---- */
#ifndef __VARIATIONAL_H_
typedef struct variational_params_s {
    float alpha;      /* smoothness weight */
    float gamma;      /* gradient constancy weight */
    float delta;      /* colour constancy weight */
    float sigma;      /* presmoothing (unused: disabled in the reference, variational.c:124-136) */
    int niter_outer;  /* warping fixed-point iterations */
    int niter_inner;  /* lagged-nonlinearity iterations */
    int niter_solver; /* SOR sweeps */
    float sor_omega;  /* SOR relaxation */
} variational_params_t;

/* replaces variational.c:85-98 */
void variational_params_default(variational_params_t *params);
/* replaces variational.c:101-143.  wx, wy: in/out flow planes (host); im1, im2: host colour images.
 * params == NULL -> defaults.  Uses a thread-local default context on the current CUDA device.
 * Errors print to stderr and exit(1) (the reference's convention, image.c:19-30). */
void variational(image_t *wx, image_t *wy, const color_image_t *im1, const color_image_t *im2,
                 variational_params_t *params);
#endif

/* ---- multi-frame parameters: POD of the ParameterList keys Variational_MT reads
 * (variational_mt.cpp:173-192, 250-251, 533-568; key names in comments) ---- */
#define SF_MT_MAX_REF 8
enum { SF_ROBUST_QUADRATIC = 0, SF_ROBUST_MODL1 = 1, SF_ROBUST_LORENTZIAN = 2, SF_ROBUST_TRUNC_MODL1 = 3,
       SF_ROBUST_GEMAN_MCCLURE = 4 }; /* select_robust_function, variational_aux_mt.cpp:906-925 */

typedef struct sf_mt_params_s {
    int S;                       /* slow_flow_S: ref = S-1, F = 2*ref+1 frames */
    int layers;                  /* slow_flow_layers */
    float p_scale;               /* slow_flow_p_scale */
    float alpha, gamma, delta;   /* slow_flow_alpha / gamma / delta */
    int dataterm;                /* slow_flow_dataterm (1 = normalised data term) */
    int smoothing;               /* slow_flow_smoothing (0 or 1) */
    int one_direction;           /* slow_flow_method == "forward" (or Variational_MT::one_direction) */
    float rho[SF_MT_MAX_REF];    /* slow_flow_rho_a */
    float omega[SF_MT_MAX_REF];  /* slow_flow_omega_a */
    int robust_color;  float robust_color_eps, robust_color_truncation;
    int robust_grad;   float robust_grad_eps, robust_grad_truncation;  /* robust_grad < 0: reuse colour settings (Q8) */
    int robust_reg;    float robust_reg_eps, robust_reg_truncation;
    int niter_alter, niter_outer, niter_inner, niter_solver, niter_graphc;
    float thres_outer, thres_inner, sor_omega;
    int occlusion_reasoning;     /* slow_flow_occlusion_reasoning */
    float occlusion_penalty, occlusion_alpha;
    int graphcut_int_terms;      /* 1: emulate gco's integer EnergyTermType (costs truncate to 0) */
    int hbit;                    /* 16bit */
    float img_norm_avg[3], img_norm_std[3]; /* slow_flow_img_norm_{avg,std}_{1,2,3} (written by normalize) */
} sf_mt_params_t;

/* defaults of slow_flow.cpp:64-128 (setDefault) */
void sf_mt_params_default(sf_mt_params_t *params);

/* ---- handle API ---- */
typedef struct sfgpu_ctx sfgpu_ctx;

enum { SFGPU_OK = 0, SFGPU_ERR_CUDA = 1, SFGPU_ERR_ARG = 2, SFGPU_ERR_NOMEM = 3, SFGPU_ERR_UNSUPPORTED = 4 };

/* Create a context on `device`.  `stream` is a cudaStream_t passed as void* (NULL: the context
 * creates its own non-blocking stream).  One context must only be used by one host thread at a time. */
int sfgpu_create(int device, void *stream, sfgpu_ctx **out);
void sfgpu_destroy(sfgpu_ctx *ctx);
/* last error message of the calling thread ("" if none) */
const char *sfgpu_last_error(void);
/* number of usable CUDA devices (0 if none / driver missing) */
int sfgpu_device_count(void);
/* block until all work queued on the context's stream is done */
int sfgpu_synchronize(sfgpu_ctx *ctx);

/* solver selection: 0 = temporally blocked red-black SOR (default), 1 = one launch per half sweep
 * (validation / tiny images).  Both are red-black and produce identical iterates. */
int sfgpu_set_sor_variant(sfgpu_ctx *ctx, int variant);
/* sweeps fused per HBM round trip of the blocked solver (1..8; default chosen per image size) */
int sfgpu_set_sor_fuse(sfgpu_ctx *ctx, int sweeps_per_launch);

/* two-frame refinement, host buffers (replaces variational.c:101; synchronous) */
int sfgpu_variational(sfgpu_ctx *ctx, image_t *wx, image_t *wy, const color_image_t *im1,
                      const color_image_t *im2, const variational_params_t *params);

/* two-frame refinement on device-resident planes (asynchronous on the context's stream).
 * d_wx, d_wy: stride*height floats, in/out.  d_im1, d_im2: 3*stride*height floats, planar. */
int sfgpu_variational_dev(sfgpu_ctx *ctx, float *d_wx, float *d_wy, const float *d_im1, const float *d_im2,
                          int width, int height, int stride, const variational_params_t *params);

/* Pipelined sequence refinement (config 5; the shard loop of slow_flow.cpp:706 / adaptiveFR.cpp:496):
 * n_pairs consecutive frame pairs (pair j = frames[j], frames[j+1]); wx[j], wy[j] in/out.
 * Host buffers; uploads of pair j+1 and downloads of pair j-1 overlap the solve of pair j, and a
 * frame shared by two pairs is uploaded once.  Page-locked host memory (cudaMallocHost / sfgpu_host_register) is
 * pipelined as given; ordinary pageable memory (the reference's image_new) is staged pair by pair through the context's
 * page-locked slots by a few host threads (fast, but without overlap between pairs). */
int sfgpu_variational_sequence(sfgpu_ctx *ctx, int n_pairs, const color_image_t *const *frames,
                               image_t *const *wx, image_t *const *wy, const variational_params_t *params);

/* The same pipeline fed with the INTEGER images the reference holds before its float conversion: 8-bit frames as
 * adaptiveFR.cpp:450-464 has them (cv::Mat CV_8UC1 / CV_8UC3 -> mat2colorImg<uchar> / colorMat2colorImg<Vec3b>,
 * utils/utils.h:122-160) and 16-bit frames as slow_flow.cpp:470-477 loads them (CV_16UC1/3 -> convertTo(CV_32F)).
 * The fields are the cv::Mat fields those converters read.  channels == 1: the grey value goes to all three planes;
 * channels == 3: interleaved sample c of a pixel goes to plane c.  The conversion runs on the device and is exact
 * (every 8-/16-bit integer is a float), so results are identical to converting on the host and calling
 * sfgpu_variational_sequence -- but a 2560x1440 frame crosses PCIe as 11 (22) MB instead of 44 MB.
 * continue_from_previous != 0: frames[0] is the last frame of the previous sequence call on this context (same
 * geometry, no other call in between); it is still resident in the device ring and is not uploaded again. */
typedef struct sf_frame_int_s {
    int width, height;
    int channels;       /* 1 or 3 */
    size_t step;        /* bytes per row (cv::Mat::step) */
    const void *data;   /* unsigned char (u8 entry) or unsigned short (u16 entry) samples */
} sf_frame_int_t;
int sfgpu_variational_sequence_u8(sfgpu_ctx *ctx, int n_pairs, const sf_frame_int_t *frames, image_t *const *wx,
                                  image_t *const *wy, const variational_params_t *params, int continue_from_previous);
int sfgpu_variational_sequence_u16(sfgpu_ctx *ctx, int n_pairs, const sf_frame_int_t *frames, image_t *const *wx,
                                   image_t *const *wy, const variational_params_t *params, int continue_from_previous);

/* page-lock / unlock a host range so transfers are asynchronous (cudaHostRegister) */
int sfgpu_host_register(void *ptr, unsigned long long bytes);
int sfgpu_host_unregister(void *ptr);

/* multi-frame refinement (replaces Variational_MT::variational, variational_mt.cpp:526-784).
 * im: F = 2*(S-1)+1 host colour images, reference frame at index S-1.  channel_w may be NULL (all
 * ones, variational_mt.cpp:535-538).  occlusions_out may be NULL (or have NULL data); otherwise receives the -1/0/+1
 * labels of the finest level (Variational_MT::getOcclusions).  channel_w and occlusions_out, when given, have the
 * flow's geometry.  avg_change_out: the returned Point2f. */
int sfgpu_variational_mt(sfgpu_ctx *ctx, image_t *wx, image_t *wy, const color_image_t *const *im,
                         const sf_mt_params_t *params, const color_image_t *channel_w,
                         image_t *occlusions_out, float avg_change_out[2]);

/* Frame cache of the multi-frame entry for callers that solve many windows over ONE sequence, like the jet loop of
 * slow_flow.cpp:706-1030: consecutive windows share frames and the backward window of a jet reads the frames of its
 * forward window, so with the cache a frame crosses PCIe once instead of once per window that contains it.
 * max_frames > 0: sfgpu_variational_mt keeps device copies of up to max_frames level-0 frames, keyed by the host pointer
 * im[f]->c1 and the geometry, least recently used first out.  CONTRACT: while the cache is enabled the caller must not
 * change the contents of a frame it has passed (normalize() first, then enable).  max_frames == 0 disables the cache and
 * frees it; every call empties it.  A window with more than max_frames frames is solved without the cache.  Off by
 * default: an unmodified call site keeps the reference's semantics.  SLOWFLOW_GPU_TRACE=1 prints the hit / miss counts
 * when the context is destroyed. */
int sfgpu_mt_frame_cache(sfgpu_ctx *ctx, int max_frames);

/* normalize() of variational_mt.cpp:17-85: in place on F host frames; fills params->img_norm_* */
int sfgpu_normalize(sfgpu_ctx *ctx, color_image_t *const *seq, int F, sf_mt_params_t *params);

/* The jet loop of slow_flow.cpp:706-1030 (deep_matching = 0) over ONE sequence of integer frames, on the device.
 * frames[0 .. n_frames-1]: the loaded sequence as cv::Mat fields (sf_frame_int_t, like sfgpu_variational_sequence_u8/u16),
 * bits = 8 or 16, all of one width x height.  scale != 1: every frame is pre-scaled first, exactly as sfgpu_prescale
 * does (slow_flow.cpp:538-542).  The sequence is then normalised as ONE sequence over all n_frames (normalize(),
 * variational_mt.cpp:17-85); params->img_norm_avg / img_norm_std receive the values normalize() publishes (6 significant
 * digits), and those published values are the ones the windows use.
 * With steps = params->S - 1, jet j in [first_jet, first_jet + n_jets) writes, at index k = j - first_jet:
 *   fwd_x[k], fwd_y[k]   forward window frames[j*steps .. j*steps + 2*steps]: zero initial flow, channel_w
 *                        (NULL: all ones), one_direction = params->one_direction; result x steps (:865-911)
 *   back_x[k], back_y[k] backward window, the reversed frames j*steps + 3*steps down to j*steps + steps:
 *                        no channel weights (Q10), one_direction = params->one_direction || backward_one_direction;
 *                        result x steps (:1018-1030)
 *   occlusions[k]        (the array may be NULL) the forward window's -1/0/+1 labels (Variational_MT::getOcclusions)
 * Every output, bit for bit and on whole planes, equals this sequence of calls:
 *   unpack the frame to float (exact) -> sfgpu_prescale -> sfgpu_normalize over all n_frames
 *   -> sfgpu_variational_mt per window -> multiply by steps in fp32.
 * Output planes (and channel_w) have the (scaled) frame geometry.  n_frames >= 1 + (first_jet + n_jets + 2) * steps: a
 * multi-GPU caller shards the jets with first_jet / n_jets, and every shard normalises over the whole sequence.
 * Each jet's new frames are uploaded while the previous jet solves, and with page-locked memory every window's results
 * are downloaded while the next window computes (pageable memory is staged as in sfgpu_variational_sequence).
 * sfgpu_get_mt_stats afterwards sums the windows of the call; its setup_ms is the time of the statistics pass and
 * total_ms that of the call.  Every argument check runs before anything is written.  SFGPU_ERR_UNSUPPORTED for
 * smoothing >= 2, like sfgpu_variational_mt.  Uses the context's io area, so a following sfgpu_variational_sequence_u8/u16
 * cannot use continue_from_previous.  sfgpu_slow_flow_jets_epic (with the EPIC entries below) is the same loop with EPIC
 * initial flows. */
int sfgpu_slow_flow_jets(sfgpu_ctx *ctx, int n_frames, const sf_frame_int_t *frames, int bits, float scale,
                         int first_jet, int n_jets, sf_mt_params_t *params, int backward_one_direction,
                         const color_image_t *channel_w, image_t *const *fwd_x, image_t *const *fwd_y,
                         image_t *const *back_x, image_t *const *back_y, image_t *const *occlusions);

/* iteration statistics of the last sfgpu_variational_mt (or sfgpu_slow_flow_jets) call on this context */
typedef struct sfgpu_mt_stats_s {
    int levels;            /* pyramid levels actually run */
    int outer_iterations;  /* total outer iterations executed over all levels / alternations */
    int sor_calls;         /* sor_coupled invocations */
    int graphcut_calls;    /* optimizeOcc invocations */
    /* host wall-clock split of the call (milliseconds) */
    double setup_ms;       /* workspace, uploads, pyramid (until the coarsest level starts) */
    double graphcut_ms;    /* optimizeOcc, host wall clock of all calls (device labelling: the time to queue it) */
    double total_ms;
    long long pixel_outer_iterations; /* sum over the executed outer iterations of width*height of their level */
} sfgpu_mt_stats_t;
int sfgpu_get_mt_stats(sfgpu_ctx *ctx, sfgpu_mt_stats_t *out);

/* Output side of a window: the files dense_tracking consumes (dense_tracking.cpp:1119-1162).  Host only.
 *  - .flo: writeFlowFile / readFlowFile of epic_flow_extended/io.c:50-96 (tag 202021.25, width, height, interleaved u,v)
 *  - occlusion .pbm: slow_flow.cpp:893-905 (labels -1/0/+1 -> 0/128/255 -> binary PBM as cv::imwrite stores it) */
int sfgpu_write_flo(const char *filename, const image_t *flowx, const image_t *flowy);
int sfgpu_read_flo_size(const char *filename, int *width, int *height);
int sfgpu_read_flo(const char *filename, image_t *flowx, image_t *flowy);
int sfgpu_write_occlusion_pbm(const char *filename, const image_t *occlusions);
/* device selection for "one host thread per device" drivers that do not link the CUDA runtime themselves;
 * sfgpu_create(-1, ...) creates the context on the calling thread's current device */
int sfgpu_set_device(int device);
int sfgpu_get_device(void);

/* Input side of a window (what slow_flow.cpp does to each frame before the solver):
 *  - sfgpu_prescale: GaussianBlur(sigma = 1/sqrt(2*scale), replicate border) + resize(fx = fy = scale, INTER_LINEAR) of a
 *    float colour image (slow_flow.cpp:538-542).  dst must have the geometry sfgpu_prescale_size reports
 *    (cvRound(width*scale) x cvRound(height*scale), stride = ceil4).
 *  - sfgpu_raw_weighting: rawWeighting (utils/utils.cpp:1336-1374, slow_flow.cpp:596-600): channel weights of a Bayer
 *    mosaic with its red site at (red_x, red_y); weight is clamped to [0, 3].  Only valid columns are written. */
int sfgpu_prescale_size(int width, int height, float scale, int *out_width, int *out_height);
int sfgpu_prescale(sfgpu_ctx *ctx, color_image_t *dst, const color_image_t *src, float scale);
int sfgpu_raw_weighting(sfgpu_ctx *ctx, color_image_t *weights, int red_x, int red_y, float weight);

/* Labelling step of optimizeOcc (variational_aux_mt.cpp:851-881: gco expansion on a grid graph with data costs
 * d0/d1 per site and Potts weight alpha) as the exact binary min-cut the GPU path uses.  Host-only operator twin for
 * tests: costs are dense w*h arrays, labels[p] in {0, 1}; int_terms selects gco's stock integer EnergyTermType. */
int sfgpu_grid_mincut(int w, int h, const float *d0, const float *d1, float alpha, int int_terms, int *labels);
/* The same labelling by the DEVICE solver the multi-frame path uses (sf_mincut.cu: layered push scheme on exact
 * distances inside one cooperative kernel).  The canonical labelling is unique, so labels equal sfgpu_grid_mincut's.
 * stats (nullable): {phases, grid-wide passes}. */
int sfgpu_grid_mincut_dev(sfgpu_ctx *ctx, int w, int h, const float *d0, const float *d1, float alpha, int int_terms,
                          int *labels, int stats[2]);

/* ---- per-kernel timing (CUDA events on the context's stream) for bench.py's roofline ---- */
typedef struct sfgpu_profile_s {
    double sor_ms;        /* sum of device time of all SOR launches since reset */
    long long sor_launches;
    long long sor_calls;   /* sor_coupled invocations */
    long long sor_pixel_sweeps; /* sum over calls of width*height*niter_solver */
    double data_ms;       /* fused derivative + data-term kernel */
    long long data_launches;
    long long data_pixels;
    long long kernel_launches; /* every kernel launched by this context since reset */
    double graphcut_ms;   /* occlusion labelling on the device: data costs + min-cut kernel (multi-frame path) */
} sfgpu_profile_t;
int sfgpu_profile_enable(sfgpu_ctx *ctx, int on);   /* on=1 brackets SOR / data-term launches with events */
int sfgpu_profile_reset(sfgpu_ctx *ctx);
int sfgpu_profile_get(sfgpu_ctx *ctx, sfgpu_profile_t *out); /* synchronises the stream */

/* ---- operator-level twins (host buffers; test path).  Same argument meaning as the reference. ---- */
/* variational_aux.c:18 / variational_aux_mt.cpp:722 (factor) ; mask may be NULL */
int sfgpu_image_warp(sfgpu_ctx *ctx, color_image_t *dst, image_t *mask, const color_image_t *src,
                     const image_t *wx, const image_t *wy, int factor);
/* The multi-frame path's per-frame pass as an operator: image_warp with its time factor (variational_aux_mt.cpp:722)
 * followed by the five spatial derivative images of the WARPED frame (the filters and border rules of get_derivatives,
 * variational_mt.cpp:111-166, image.c:400-526).  variant 0 = the production kernel (one fused marching pass,
 * sf_wderivs.cu), variant 1 = the two-kernel path it replaced (A/B reference). */
int sfgpu_warp_frame_derivs(sfgpu_ctx *ctx, const color_image_t *src, const image_t *wx, const image_t *wy, int factor,
                            int variant, color_image_t *warped, image_t *mask, color_image_t *dx, color_image_t *dy,
                            color_image_t *dxx, color_image_t *dxy, color_image_t *dyy);
/* variational_aux.c:183 (coef = 5, deriv = 5-tap); result written into dst.
 * MT variant (variational_aux_mt.cpp:673): avg/std/hbit de-normalisation; pass NULL for two-frame. */
int sfgpu_compute_dpsis_weight(sfgpu_ctx *ctx, image_t *dst, const color_image_t *im, float coef,
                               const float *avg3, const float *std3, int hbit);
/* variational_aux.c:84 (robust_reg < 0) or variational_aux_mt.cpp:18 modes 0/1 with a penalty */
int sfgpu_compute_smoothness(sfgpu_ctx *ctx, image_t *dst_horiz, image_t *dst_vert, const image_t *uu,
                             const image_t *vv, const image_t *dpsis_weight, float alpha_factor,
                             int robust_reg, float reg_eps, float reg_trunc, int mode);
/* get_derivatives + compute_data_and_match (variational_aux.c:55,215) in one fused pass:
 * im2w is the already warped second image. */
int sfgpu_compute_data_and_match(sfgpu_ctx *ctx, image_t *a11, image_t *a12, image_t *a22, image_t *b1,
                                 image_t *b2, const image_t *mask, const image_t *du, const image_t *dv,
                                 const color_image_t *im1, const color_image_t *im2w,
                                 float half_delta_over3, float half_gamma_over3);
/* The PRODUCTION kernel of the default two-frame path (k_prep_two_frame) as an operator: one outer iteration's
 * image_warp -> get_derivatives -> compute_data_and_match -> sub_laplacian x2 (variational_aux.c:18-78, 153-180, 215-302)
 * followed by the in-place block inverse of sor_coupled's first sweep (solver.c:101-106).  im2 is the UNWARPED second
 * image; wx, wy warp it and are the argument of the Laplacian; du, dv may be NULL (zero increment).  Whole planes are
 * written, stride padding included (zeros). */
int sfgpu_prep_two_frame(sfgpu_ctx *ctx, image_t *a11, image_t *a12, image_t *a22, image_t *b1, image_t *b2,
                         const color_image_t *im1, const color_image_t *im2, const image_t *wx, const image_t *wy,
                         const image_t *du, const image_t *dv, const image_t *dpsis_horiz, const image_t *dpsis_vert,
                         float half_delta_over3, float half_gamma_over3);
/* The multi-frame path's linear system as an operator: one linearisation of compute_one_level (variational_mt.cpp:289-365)
 * on the frames im[0 .. 2(S-1)] of one level -- warps, derivatives, the occlusion factor of occ (-1 / 0 / +1), smoothness
 * on uu = wx + du, every data term and the Laplacian -- through the production kernels the context's switches select,
 * followed by the block inverse of the SOR's first sweep.  du, dv may be NULL (first inner iteration); channel_w may be
 * NULL.  Whole planes are written, stride padding included. */
int sfgpu_mt_system(sfgpu_ctx *ctx, image_t *a11, image_t *a12, image_t *a22, image_t *b1, image_t *b2, image_t *psi_h,
                    image_t *psi_v, const color_image_t *const *im, const image_t *wx, const image_t *wy, const image_t *du,
                    const image_t *dv, const image_t *occ, const color_image_t *channel_w, const sf_mt_params_t *params);
/* The data costs of the occlusion labelling (variational_aux_mt.cpp:786-848) at (wx, wy): d0 / d1 of the W x H pixels. */
int sfgpu_mt_occ_costs(sfgpu_ctx *ctx, image_t *d0, image_t *d1, const color_image_t *const *im, const image_t *wx,
                       const image_t *wy, const sf_mt_params_t *params);
/* variational_aux.c:153 */
int sfgpu_sub_laplacian(sfgpu_ctx *ctx, image_t *dst, const image_t *src, const image_t *weight_horiz,
                        const image_t *weight_vert);
/* solver.c:63 with red-black ordering.  Like the reference, a11/a12/a22 are overwritten with the
 * inverted blocks. */
int sfgpu_sor_coupled(sfgpu_ctx *ctx, image_t *du, image_t *dv, image_t *a11, image_t *a12, image_t *a22,
                      const image_t *b1, const image_t *b2, const image_t *dpsis_horiz,
                      const image_t *dpsis_vert, int iterations, float omega);

/* image.c:400-645, 658-688 and variational_aux.c:55-78 -- the separable filters and the derivative set the hot path
 * computes on the fly, as stand-alone operators for tests.  order 1 = 3 taps, order 2 = 5 taps (coeffs[2*order+1]);
 * color_image_convolve_hv: pass NULL coefficients for the direction that is skipped (like a NULL convolution_t*).
 * get_derivatives uses the [1,-8,0,8,-1]/12 filter of variational.c:118-119. */
int sfgpu_convolve_horiz(sfgpu_ctx *ctx, image_t *dst, const image_t *src, int order, const float *coeffs);
int sfgpu_convolve_vert(sfgpu_ctx *ctx, image_t *dst, const image_t *src, int order, const float *coeffs);
int sfgpu_color_image_convolve_hv(sfgpu_ctx *ctx, color_image_t *dst, const color_image_t *src, int horiz_order,
                                  const float *horiz_coeffs, int vert_order, const float *vert_coeffs);
int sfgpu_get_derivatives(sfgpu_ctx *ctx, const color_image_t *im1, const color_image_t *im2, color_image_t *dx,
                          color_image_t *dy, color_image_t *dt, color_image_t *dxx, color_image_t *dxy, color_image_t *dyy,
                          color_image_t *dxt, color_image_t *dyt);

/* ---- EPIC sparse-to-dense interpolation (SURVEY 8f rank 4): the step that produces the flow variational() refines.
 * Types are those of epic_flow_extended/epic.h:5-14 and array_types.h:70-77; if the reference headers were included first
 * (array_types.h defines ___ARRAY_TYPES_H___; define SLOWFLOW_GPU_HAVE_EPIC_H after including the guard-less epic.h) their
 * definitions are used. */
#ifndef ___ARRAY_TYPES_H___
typedef struct { float *pixels; int tx, ty; } float_image; /* row-major tx columns x ty rows */
#endif
#ifndef SLOWFLOW_GPU_HAVE_EPIC_H
typedef struct epic_params_s {
    char method[20];     /* "LA" locally-weighted affine or "NW" Nadaraya-Watson */
    float saliency_th;   /* matches from pixels with a saliency below this are removed (0: off) */
    int pref_nn;         /* neighbours of the consistency filter (0: off) */
    float pref_th;       /* its threshold, pixels */
    int nn;              /* neighbours of the interpolation */
    float coef_kernel;   /* kernel exp(-coef * geodesic distance) */
    float euc;           /* constant added to the edge cost */
    int verbose;
} epic_params_t;
/* replaces epic.cpp:131-140 */
void epic_params_default(epic_params_t *params);
#endif
typedef struct sfgpu_epic_stats_s {
    int matches_in, matches_after_saliency, matches_after_consistency;
    int sweeps_prefilter, sweeps_interpolation; /* distance-transform sweeps executed (epic_aux.cpp:170-178) */
} sfgpu_epic_stats_t;
/* replaces epic() (epic.cpp:147-234; callers epicflow.cpp:125, adaptiveFR.cpp:568, slow_flow.cpp:819,979,
 * dense_tracking.cpp:1294).  flowx, flowy: output planes (host); im: first image in Lab (only the saliency filter reads
 * it); input_matches: ty rows of tx >= 4 floats x1 y1 x2 y2; edges: width x height costs, and like in the reference
 * params->euc is ADDED TO THE CALLER'S ARRAY.  stats may be NULL.  The reference's n_thread argument has no meaning here. */
int sfgpu_epic(sfgpu_ctx *ctx, image_t *flowx, image_t *flowy, const color_image_t *im, const float_image *input_matches,
               float_image *edges, const epic_params_t *params, sfgpu_epic_stats_t *stats);
/* epic() on n images of ONE geometry in one call: item k is exactly sfgpu_epic(ctx, flowx[k], flowy[k], im[k],
 * input_matches[k], edges[k], params, &stats[k]).  params is shared; match counts may differ per item.  euc is added to
 * every caller's edges[k] once, like sfgpu_epic (so the edges[k] must be distinct arrays).  stats: n entries or NULL.
 * The items' distance transforms, neighbour searches and fits run side by side on the device, which is what makes a batch
 * faster than n calls.  On error nothing is written to any flow plane and the message names the first failing item;
 * SFGPU_ERR_ARG for n < 1, a null pointer, items of different width / height / stride, any check sfgpu_epic makes, and an
 * item with no match left after the filters. */
int sfgpu_epic_batch(sfgpu_ctx *ctx, int n, image_t *const *flowx, image_t *const *flowy, const color_image_t *const *im,
                     const float_image *const *input_matches, float_image *const *edges, const epic_params_t *params,
                     sfgpu_epic_stats_t *stats);
/* replaces rgb_to_lab (image.c:694; callers epicflow.cpp:124, adaptiveFR.cpp:568, slow_flow.cpp:814): the first image of
 * epic() in Lab with the reference's attenuation of dark and light colours.  dst: same geometry as src (planar, stride =
 * ceil4(width)).  Whole stride rows are converted, padding columns included, like the reference's loop over stride*height.
 * Same arithmetic as the reference operation for operation (C's float / double promotions, no FMA); the device's double
 * pow / exp may, very rarely, round a result one float ulp away from glibc's. */
int sfgpu_rgb_to_lab(sfgpu_ctx *ctx, color_image_t *dst, const color_image_t *src);
/* The EpicFlow two-step (epicflow.cpp:124-129, adaptiveFR.cpp:568-574) over n_pairs consecutive pairs of ONE geometry:
 * pair k = frames[k], frames[k+1] (RGB in [0,255], as variational() takes them).  Pair k's wx[k], wy[k] are, bit for bit,
 *   lab = rgb_to_lab(frames[k]); sfgpu_epic(wx[k], wy[k], lab, matches[k], edges[k], epic_params, &stats[k]);
 *   sfgpu_variational(wx[k], wy[k], frames[k], frames[k+1], flow_params);
 * (the incoming contents of wx, wy are not read).  epic_params is required; flow_params == NULL -> defaults.  euc is added
 * once to every edges[k] (distinct arrays), like epic().  stats: n_pairs entries or NULL.
 * Each frame is uploaded once for both steps, the Lab planes are made on the device and the interpolated flows stay there
 * until they are refined.  Pairs run in chunks of 8 EPIC items; with page-locked memory the next chunk's uploads and the
 * refined flows' downloads overlap the computation (pageable memory is staged as in sfgpu_variational_sequence).
 * Errors: every argument check (those of sfgpu_epic_batch and sfgpu_variational) runs first, and a failed check writes no
 * flow plane and no edge array.  A pair left with no match after the filters is found while running: the chunks before
 * its chunk are then complete (flows, stats, edges), its chunk and the later pairs' flows are not written, the later
 * chunks' edges are untouched, and the message names the pair.  A following sfgpu_variational_sequence_u8/u16 cannot use
 * continue_from_previous. */
int sfgpu_epicflow_sequence(sfgpu_ctx *ctx, int n_pairs, const color_image_t *const *frames, const float_image *const *matches,
                            float_image *const *edges, const epic_params_t *epic_params, const variational_params_t *flow_params,
                            image_t *const *wx, image_t *const *wy, sfgpu_epic_stats_t *stats);
/* The jet loop of slow_flow.cpp:706-1030 in its other mode (deep_matching != 0): every window starts from an EPIC
 * interpolation of sparse matches (forward window slow_flow.cpp:801-843, backward window :979) instead of a zero flow.
 * Frames, bits, scale, first_jet / n_jets, params (img_norm_* published), backward_one_direction, channel_w (forward
 * windows only), the outputs (x S-1), occlusions and SFGPU_ERR_UNSUPPORTED for smoothing >= 2 are as in
 * sfgpu_slow_flow_jets.  With s = S-1, nf[f] = frame f after unpack, sfgpu_prescale (scale != 1) and sfgpu_normalize over
 * all n_frames (what sfgpu_slow_flow_jets computes), and r = j*s + s the reference frame of jet j's forward window, the
 * outputs at k = j - first_jet are, bit for bit and on whole planes:
 *   forward:  lab = sfgpu_rgb_to_lab(nf[r])                       (only when saliency_th != 0)
 *             sfgpu_epic(fx, fy, lab, fwd_matches[k], edges[k], epic_params, &epic_stats[2k])
 *             fx, fy *= 1.0f / s                                  (fp32)
 *             sfgpu_variational_mt(fx, fy, nf[j*s .. j*s + 2s], params, channel_w, occlusions[k])
 *             fwd_x[k], fwd_y[k] = fx, fy * s
 *   backward: the same with Lab from nf[r + s], back_matches[k], edges[k + 1], &epic_stats[2k + 1], the frames
 *             nf[j*s + 3s - i] for i = 0 .. 2s, no channel weights, and one_direction = params->one_direction ||
 *             backward_one_direction.
 * Matches and edge maps are in the window geometry (after pre-scaling); edges[m] (n_jets + 1 distinct arrays) belongs to
 * reference frame (first_jet + m)*s + s and serves jet m - 1's backward and jet m's forward window.  euc is added once to
 * every edges[m] in the caller's array, as epic() adds it; since the reference reads the edge file afresh per window, both
 * windows see edges + euc, as here.  Lab is converted from the window's own normalised reference frame: normalize() runs
 * in place on the sequence (slow_flow.cpp:673) before the loop (:706) reads im = &seq[j*steps] (:721-724) and calls
 * rgb_to_lab (:814), which also puts 8- and 16-bit sequences on one scale for the saliency filter.  epic_params is required;
 * epic_stats: 2 * n_jets entries (forward, backward per jet) or NULL.
 * Jets run in chunks of 4 (8 EPIC items in one batch); with page-locked memory the next chunk's frames and edge maps go up
 * while this chunk's windows solve, and every window's results go down while the next one computes.  Device memory is
 * bounded by the chunk, not by n_jets.
 * Errors: every argument check (those of sfgpu_slow_flow_jets and of sfgpu_epic: match columns >= 4, method, edge
 * geometry; and distinct edge arrays) runs before anything is written.  A window left with no match after the filters
 * stops the call: the chunks before its chunk are complete (flows, occlusions, stats, edges), the later outputs are not
 * written, the later chunks' edge maps are untouched, and the message names the jet and the direction. */
int sfgpu_slow_flow_jets_epic(sfgpu_ctx *ctx, int n_frames, const sf_frame_int_t *frames, int bits, float scale,
                              int first_jet, int n_jets, sf_mt_params_t *params, int backward_one_direction,
                              const color_image_t *channel_w, const float_image *const *fwd_matches,
                              const float_image *const *back_matches, float_image *const *edges,
                              const epic_params_t *epic_params, image_t *const *fwd_x, image_t *const *fwd_y,
                              image_t *const *back_x, image_t *const *back_y, image_t *const *occlusions,
                              sfgpu_epic_stats_t *epic_stats);

/* operator twin of dist_trf_nnfield_subset (epic_aux.cpp:350-401) with the seeds as the query points: the label map
 * (w*h), and per seed the nn nearest seeds over the geodesic neighbourhood graph with their distances */
int sfgpu_epic_nnfield(sfgpu_ctx *ctx, int *best, float *dist, int *labels, const int *seeds, int ns, int nn,
                       const float *cost, int w, int h, int *sweeps);

/* library / build identification, e.g. "slowflow_gpu 0.1 sm_100a" */
const char *sfgpu_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SLOWFLOW_GPU_H_ */
