/*
 * loma_nerf_b200.h -- C ABI of libloma_nerf_b200.so
 *
 * A from-scratch sm_100a (B200) implementation of the one hot path loma-nerf runs through its
 * loma-compiled _code/nerf.so and _code/mlp_fit.so: positional encoding -> per-sample coordinate
 * MLP (forward + reverse-mode gradient) -> front-to-back alpha compositing (forward + backward)
 * -> SSE loss.  Two groups of entry points:
 *
 *  (1) COMPAT: the five symbols the reference hosts bind with ctypes
 *      (loma_public/compiler.py:262-276 sets their argtypes; train_nerf.py:212-213,
 *      fit_img.py:358-360 fetch them).  Same names, argument order, ragged float** and float***
 *      buffers, in-place outputs and accumulate-into-d_ semantics as the loma-generated C.
 *      Host pointers in, host pointers out, synchronous.
 *  (2) FLAT: contiguous-buffer entry points (device pointers, or pinned/pageable host pointers
 *      for the *_host variants) used by benchmarks, the Python mirror and multi-GPU sharding.
 *      The compat symbols are thin gather/scatter wrappers over these.
 *
 * No torch types, no C++ types: plain pointers, ints, floats and POD structs.
 * There is NO CPU fallback: every entry point fails (status != 0 / NaN loss) without a CUDA
 * device.  All arithmetic is IEEE fp32 unless lnb_step_args.path selects the tensor cores
 * (LNB_PATH_TC: bf16 operands, fp32 accumulation).
 */
#ifndef LOMA_NERF_B200_H
#define LOMA_NERF_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LNB_API __attribute__((visibility("default")))
#else
#define LNB_API
#endif

#define LNB_ABI_VERSION 4
#define LNB_MAX_LAYERS 16

/* ------------------------------------------------------------------------------------------
 * (1) COMPAT symbols
 * ------------------------------------------------------------------------------------------ */

/* replaces: loma function nerf_evaluate_and_march, /root/reference/scripts/nerf.py:1-304
 * (call site train_nerf.py:325-366, eval call site train_nerf.py:616-657).
 * Writes in place: intermediate_outputs (accumulated onto entry contents, then activated),
 * img_sample_rgba_arr, alpha, cumprod_alpha, weights_samples (overwritten), accumulated_color
 * (accumulated onto entry contents).  Returns the SSE loss; NaN on any CUDA failure. */
LNB_API float nerf_evaluate_and_march(float **layer_input, int layer_input_h, int layer_input_w,
                              float ***ws, float **bs, float **target_image, int target_image_h,
                              int target_image_w, int num_weights, int **weight_shapes,
                              int **bias_shapes, int **intermediate_output_shapes,
                              float ***intermediate_outputs, float ***img_sample_rgba_arr,
                              int num_samples, float **dists, float **alpha, float **cumprod_alpha,
                              float **weights_samples, float **accumulated_color);

/* replaces: grad_nerf_evaluate_and_march = rev_diff(nerf_evaluate_and_march),
 * scripts/nerf.py:306; signature rule loma_public/reverse_diff.py:504-517 (each In argument is
 * followed by its adjoint; int -> int*; trailing float _dreturn); call site train_nerf.py:395-478.
 * Accumulates into d_layer_input, d_ws, d_bs, d_target_image, d_dists, d_accumulated_color,
 * d_intermediate_outputs (pre-activation adjoints dZ_l); leaves the primal scratch arrays and all
 * int adjoints untouched; d_img_sample_rgba_arr, d_alpha, d_cumprod_alpha, d_weights_samples are
 * left as they were (the reference ends them at zero).  On CUDA failure d_ws is NaN-filled so the
 * host's NaN guard (train_nerf.py:486-489) trips. */
LNB_API void grad_nerf_evaluate_and_march(
    float **layer_input, float **d_layer_input, int layer_input_h, int *d_layer_input_h,
    int layer_input_w, int *d_layer_input_w, float ***ws, float ***d_ws, float **bs, float **d_bs,
    float **target_image, float **d_target_image, int target_image_h, int *d_target_image_h,
    int target_image_w, int *d_target_image_w, int num_weights, int *d_num_weights,
    int **weight_shapes, int **d_weight_shapes, int **bias_shapes, int **d_bias_shapes,
    int **intermediate_output_shapes, int **d_intermediate_output_shapes,
    float ***intermediate_outputs, float ***d_intermediate_outputs, float ***img_sample_rgba_arr,
    float ***d_img_sample_rgba_arr, int num_samples, int *d_num_samples, float **dists,
    float **d_dists, float **alpha, float **d_alpha, float **cumprod_alpha,
    float **d_cumprod_alpha, float **weights_samples, float **d_weights_samples,
    float **accumulated_color, float **d_accumulated_color, float _dreturn);

/* replaces: loma function mlp_fit, scripts/mlp_fit.py:1-147 (call site fit_img.py:515-530).
 * layer_output is unused by the reference and by us. */
LNB_API float mlp_fit(float **layer_input, int layer_input_h, int layer_input_w, float **layer_output,
              float ***ws, float **bs, float **target_image, int target_image_h,
              int target_image_w, int num_weights, int **weight_shapes, int **bias_shapes,
              int **intermediate_output_shapes, float ***intermediate_outputs);

/* replaces: grad_mlp_fit = rev_diff(mlp_fit), scripts/mlp_fit.py:174 (call site
 * fit_img.py:468-498). */
LNB_API void grad_mlp_fit(float **layer_input, float **d_layer_input, int layer_input_h,
                  int *d_layer_input_h, int layer_input_w, int *d_layer_input_w,
                  float **layer_output, float **d_layer_output, float ***ws, float ***d_ws,
                  float **bs, float **d_bs, float **target_image, float **d_target_image,
                  int target_image_h, int *d_target_image_h, int target_image_w,
                  int *d_target_image_w, int num_weights, int *d_num_weights, int **weight_shapes,
                  int **d_weight_shapes, int **bias_shapes, int **d_bias_shapes,
                  int **intermediate_output_shapes, int **d_intermediate_output_shapes,
                  float ***intermediate_outputs, float ***d_intermediate_outputs, float _dreturn);

/* replaces: loma function mult_a_b, scripts/mlp_fit.py:150-172 (required by fit_img.py:360-374).
 * c[i][j] += sum_k a[i][k] * b[k][j]. */
LNB_API void mult_a_b(float **a, int a_h, int a_w, float **b, int b_h, int b_w, float **c);

/* replaces: the forward-mode pair constructor the loma compiler emits into every library (autodiff.py:199-208;
 * `_dfloat make__dfloat(float val, float dval)` in the generated C).  Neither host script calls it; it is exported
 * so that the symbol table of the drop-in matches the generated one. */
typedef struct { float val; float dval; } _dfloat;
LNB_API _dfloat make__dfloat(float val, float dval);

/* ------------------------------------------------------------------------------------------
 * (2) FLAT API
 * ------------------------------------------------------------------------------------------ */

typedef struct lnb_ctx lnb_ctx; /* device, stream, workspace; one per (thread, GPU) */

enum { LNB_OK = 0, LNB_ERR_CUDA = 1, LNB_ERR_ARG = 2, LNB_ERR_UNSUPPORTED = 3 };
enum { LNB_HEAD_NERF = 0,     /* sigmoid on channels 0-2, ReLU on channel 3: nerf.py:147-167 */
       LNB_HEAD_SIGMOID = 1 };/* sigmoid on every channel:                  mlp_fit.py:121-132 */
enum { LNB_RAY_F64 = 0, LNB_RAY_F32 = 1 };
enum { LNB_SEED_VALUE = 0,    /* backward seed _dreturn = args->seed                        */
       LNB_SEED_LOSS = 1 };   /* backward seed = this step's loss (train_nerf.py:477)       */
enum { LNB_PATH_F32 = 0,      /* fp32 CUDA-core kernels, <=1e-5 of the reference: the fused  */
                              /* kernel when the problem fits it, else the layerwise kernels */
       LNB_PATH_TC = 1,       /* tcgen05 tensor-core kernels (bf16 operands, fp32 accumulate);*/
                              /* LNB_ERR_UNSUPPORTED when the problem does not fit them.      */
                              /* Weight gradients are summed in tensor memory in MMA          */
                              /* completion order: their last bits may differ between launches*/
                              /* (colours and losses are bit-stable; LNB_PATH_F32 is fully    */
                              /* reproducible)                                                */
       LNB_PATH_F32_LAYERWISE = 2 }; /* force the layerwise fp32 kernels (all intermediates)  */

/* The MLP: weights in the reference's padded layout (mlp_utils.py:272-313):
 * ws [n_layers][max_in][max_out] with ws[l][k][j] = weight from input k to output j
 * (mlp_utils.py:166-175), bs [n_layers][max_out]; dims[l] = in_l, dims[l+1] = out_l. */
typedef struct {
    int n_layers;
    int dims[LNB_MAX_LAYERS + 1];
    int max_in, max_out;
    int head; /* LNB_HEAD_* */
} lnb_mlp;

/* CAMERA MODE input (nerf only): rays AND sample depths are generated on the device from a pose, so nothing per ray or per
 * sample crosses the bus or sits in HBM -- the device-side form of get_rays (train_nerf.py:23-62) and of the sample
 * construction (train_nerf.py:289-311).  Ray r looks through pixel q = pixels ? pixels[r] : first_pixel + r of a
 * height x width grid, row = q / width, col = q % width, with normalised coordinates i = col / (width-1),
 * j = row / (width-1) (get_rays builds BOTH axes from linspace(0, 1, width), train_nerf.py:37-39);
 *   dir = ((i - cx) / fx, -(j - cy) / fy, -1) @ R^T  (not normalised),  origin = T,  [R | T] = c2w (3 x 4, row-major).
 * Sample depths: stratified == 0: t = linspace(near, far, S) (train_nerf.py:289, endpoint included);
 * stratified == 1: t_s = near + (s + u)(far - near) / S with u = lnb_uniform(seed, q, s) in [0, 1), the counter-based
 * generator documented at lnb_uniform below (SURVEY.md 8d's synthetic sampling; the reference has the jitter commented
 * out).  dists = t[s+1] - t[s], last 1e8.  The exact path forms every value in float64 like numpy does and rounds
 * once to float32; the tensor-core path computes in float32.
 * With VIEW DIRECTIONS (dims[0] even, see pe_bands in lnb_step_args) the direction of ray r is dir / |dir|, dir as above
 * (what lnb_camera_rays returns as rays_d). */
typedef struct {
    double c2w[12];
    double fx, fy, cx, cy;        /* normalized_K[0][0], [1][1], [0][2], [1][2] */
    int width, height;
    long long first_pixel;
    const int *pixels;            /* optional [R] pixel indices (device pointer; host pointer for the *_host calls) */
    double near, far;
    int stratified;
    unsigned long long seed;
} lnb_camera;
/* u = (z >> 40) * 2^-24 with z = mix(seed + 0x9E3779B97F4A7C15 * (q * 4096 + s + 1)), mix = the SplitMix64 finaliser
 * (z ^= z >> 30; z *= 0xBF58476D1CE4E5B9; z ^= z >> 27; z *= 0x94D049BB133111EB; z ^= z >> 31).  Host-callable. */
LNB_API double lnb_uniform(unsigned long long seed, long long pixel, int s);

/* HIERARCHICAL SAMPLING (the NeRF paper's sample_pdf): importance sampling of fine depths from a coarse pass's compositing
 * weights, device pointers, float64 arithmetic.  t [R][S] float64 (the coarse depths), w [R][S] float32 (the coarse pass's
 * weights_samples: lnb_step_args.weights, or lnb_trainer_step_weights), out [R][S + n_fine] float64.  Row r:
 *   bins      m_k = 0.5 * (t_k + t_{k+1}), k = 0 .. S-2;
 *   weights   v_j = (double)w_{j+1} + 1e-5, j = 0 .. S-3 (the first and last weights are dropped, as in the paper);
 *   cdf       c_0 = 0, c_{j+1} = c_j + v_j summed sequentially in j, cdf_k = c_k / c_{S-2} (cdf_0 = 0, cdf_{S-2} = 1
 *             exactly; the paper normalises before it sums, the same mathematically);
 *   positions u_i, i = 0 .. n_fine-1: stratified == 0: np.linspace(0.0, 1.0, n_fine) bit for bit (i * (1 / (n_fine-1)),
 *             the last value exactly 1; [0.0] for n_fine = 1); stratified != 0: u_i = (i + xi_i) / n_fine with
 *             xi_i = lnb_uniform(seed, ray0 + r, i);
 *   ind       = the number of k with cdf_k <= u_i (numpy's searchsorted(side="right")),
 *             below = max(ind-1, 0), above = min(ind, S-2);
 *   d         = cdf_above - cdf_below, d = 1 when d < 1e-5;  tau = (u_i - cdf_below) / d;
 *   x_i       = m_below + tau * (m_above - m_below);
 *   out row r = the S + n_fine values {t_k} U {x_i} in ascending order (np.sort of the concatenation; only the values are
 *             defined, so ties need no rule).
 * Every operation is float64 and rounded, with no FMA contraction: the rows are bit-equal to that numpy statement.  The
 * weights are constants (no gradient flows through the sampled depths, as in the paper) and are expected >= 0.  ray0 makes
 * a chunked or sharded call reproduce the whole-batch call bit for bit (for contiguous camera chunks: first_pixel).
 * LNB_ERR_ARG for null pointers, S < 3 (no interior weights), n_fine < 1 or S + n_fine > 4096; R = 0 is a no-op (the
 * pointers of an empty batch may be NULL).
 * Camera mode on the tensor-core path forms its depths in float32, while lnb_camera_rays returns the float64 ones this
 * sampler bins: the two differ by at most one float32 ulp, far below the bf16 error of those kernels. */
LNB_API int lnb_sample_pdf(lnb_ctx *ctx, const double *t, const float *w, int R, int S, int n_fine,
                           int stratified, unsigned long long seed, long long ray0, double *out);

/* One forward(+backward) problem in the reference's layout.  N = R*S samples.  Pointers are
 * DEVICE pointers for lnb_nerf_step / lnb_fit_step and HOST pointers for the *_host variants.
 * Any output pointer may be NULL (not produced).  Accumulating outputs (+=) are marked. */
typedef struct {
    int R, S;                 /* rays (target rows) and samples per ray; mlp_fit: S = 1        */
    int n_rows;               /* rows of X actually multiplied (layer_input_h); 0 -> R*S        */
    int rows;                 /* rows the reference host declares in intermediate_output_shapes */
                              /* (>= n_rows; bias/activation run over them, nerf.py:95);0->n_rows*/
    int target_w;             /* columns of target (3)                                          */
    const float *X;           /* [n_rows][c_in] pre-encoded features                            */
    const float *ws, *bs;     /* padded weights / biases                                        */
    const float *target;      /* [R][target_w] or NULL (render: no loss)                        */
    const float *dists;       /* [R][S] (nerf only)                                             */
    /* forward outputs */
    float *inter;             /* [n_layers][inter_rows][inter_ld] post-activation layer outputs */
    int inter_rows, inter_ld; /*   (+= onto entry contents when inter_accumulate != 0)          */
    int inter_accumulate;
    float *rgba;              /* [R][S][4]  overwritten                                         */
    float *alpha, *cumprod, *weights; /* [R][S] overwritten                                     */
    float *color;             /* [R][3]  += (nerf.py:284-286) when color_accumulate, else =     */
    int color_accumulate;
    float *loss;              /* [1] overwritten                                                */
    /* backward (performed when want_grad != 0) */
    int want_grad;
    int seed_mode;            /* LNB_SEED_*                                                     */
    float seed;
    float *d_ws, *d_bs;       /* += padded layout                                               */
    float *d_X;               /* += [n_rows][c_in] or NULL                                      */
    float *d_target;          /* += [R][target_w] or NULL                                       */
    float *d_dists;           /* += [R][S] or NULL                                              */
    float *d_color;           /* += [R][3] or NULL  (d_accumulated_color)                       */
    float *d_inter;           /* += [n_layers][inter_rows][inter_ld] dZ_l, or NULL              */
    int path;                 /* LNB_PATH_*                                                     */
    /* RAYS MODE (nerf only; selected when X == NULL): the features are computed on the device  */
    /* from rays and sample depths exactly as the reference host does it: pts = o + d*t          */
    /* (train_nerf.py:289-299), X = positional_encoding_3d(pts, pe_bands) (pos_encoding.py:38-70),*/
    /* dists = [t[s+1]-t[s] ..., 1e8] (train_nerf.py:306-311).  `dists` is then ignored.         */
    const void *rays_o, *rays_d; /* [R][3]                                                      */
    const void *t;            /* [R][S] sample depths along each ray                            */
    int ray_dtype;            /* LNB_RAY_F64 (the reference's get_rays/linspace dtype) or F32   */
    int pe_bands;             /* E.  dims[0] selects the input form (rays and camera mode alike): */
    /*   dims[0] == 3 + 6E (odd): X = PE(pts, E), positions only.                                 */
    /*   dims[0] == (3 + 6E) + (3 + 6 E_d), E_d >= 0 (even): X = [PE(pts, E) | PE(u, E_d)] with   */
    /*   the unit view direction u = d / |d|, d = rays_d[r] (camera mode: the generated direction),*/
    /*   the same for all S samples of a ray; E_d = (dims[0] - 6 - 6E) / 6.  PE is                 */
    /*   positional_encoding_3d (slot 0 identity, slots 2i+1 / 2i+2 sin / cos(2^i .), feature =    */
    /*   3 * slot + coord).  The exact path forms |d| = sqrt((d0^2 + d1^2) + d2^2) in float64 with */
    /*   every operation rounded (no FMA), divides, encodes in float64 and rounds once to float32. */
    /*   Any other width is LNB_ERR_ARG.                                                          */
    /* CAMERA MODE (selected when X == NULL, rays_o == NULL and cam != NULL): see lnb_camera.      */
    /* `cam` is always a HOST pointer (a few bytes, passed to the kernels by value).               */
    const lnb_camera *cam;
} lnb_step_args;

LNB_API int lnb_abi_version(void);
/* Fills out[0..n) with {sizeof(lnb_mlp), sizeof(lnb_step_args), offsetof(lnb_step_args, X),
 * inter, rgba, loss, want_grad, d_ws, path, rays_o, pe_bands, cam, sizeof(lnb_camera), offsetof(lnb_camera, pixels)};
 * returns how many values exist.  Lets a foreign-
 * language binding verify its struct mirror without a GPU. */
LNB_API int lnb_struct_layout(int *out, int n);
LNB_API int lnb_device_count(void);
/* device < 0: the current CUDA device. */
LNB_API int lnb_create(lnb_ctx **out, int device);
LNB_API void lnb_destroy(lnb_ctx *ctx);
/* stream is a cudaStream_t: NULL = CUDA's legacy default stream, (void*)-1 = the context's own
 * non-blocking stream (the initial setting). */
LNB_API int lnb_set_stream(lnb_ctx *ctx, void *stream);
LNB_API int lnb_synchronize(lnb_ctx *ctx);
LNB_API const char *lnb_last_error(lnb_ctx *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
LNB_API long long lnb_launch_count(lnb_ctx *ctx);
/* Kernel timing for roofline reports: while enabled, every launch of the dominant (fused)
 * kernel is bracketed by CUDA events on the context's stream.  lnb_profile_read synchronises and
 * returns the summed duration, the launch count and the kernel's name. */
LNB_API int lnb_profile(lnb_ctx *ctx, int enable);
LNB_API int lnb_profile_read(lnb_ctx *ctx, double *ms_total, long long *launches, char *name, int name_len);
/* page-locked host memory for the *_host entry points (they copy straight from / to such
 * buffers; pageable buffers bounce through the context's own pinned staging). */
LNB_API void *lnb_host_alloc(size_t bytes);
LNB_API void lnb_host_free(void *p);

/* nerf path: MLP -> compositing -> loss [-> backward].  Device pointers, asynchronous on the
 * context's stream.  Follows scripts/nerf.py:67-304 and its reverse (SURVEY.md 8 a3-a7). */
LNB_API int lnb_nerf_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args);
/* mlp_fit path: MLP -> loss [-> backward].  scripts/mlp_fit.py:39-147. */
LNB_API int lnb_fit_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args);
/* Same, HOST pointers (pinned or pageable): stages H2D, runs, stages D2H, synchronises. */
LNB_API int lnb_nerf_step_host(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args);
LNB_API int lnb_fit_step_host(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args);

/* COMPOSITING EXTRAS of a nerf step: opacity and depth maps, and compositing onto a background colour (the NeRF paper's
 * acc_map, depth_map and white-background renders).  With w_s the compositing weight of sample s (weights_samples,
 * nerf.py:270: w_s = alpha_s T_s, inclusive transmittance) and t_s its depth (lnb_step_args.t in rays mode, the depth
 * lnb_camera defines in camera mode):
 *   acc_r   = sum_s w_s                       (opacity)
 *   depth_r = sum_s w_s t_s                   (expected depth, NOT divided by acc_r, like the paper's depth_map; rays and
 *                                              camera mode only: features mode has no depths)
 *   color_r = sum_s w_s rgb_s + (1 - acc_r) bg   when background == 1 (overwritten, or added to the caller's colour under
 *                                              color_accumulate); the loss, d_color and d_target use this colour.
 * The reference's inclusive transmittance gives sum_s w_s <= 1 + O(1e-10) (the 1e-10 added to every 1 - alpha), so
 * 1 - acc_r is the light that reaches the background under the same model.
 * Backward: the one change is d_w_s = sum_c (rgb_{s,c} - bg_c) dcol_c; the transmittance scan, d_alpha, d_sigma, d_dists
 * and the MLP adjoint follow from d_w_s as without a background.  bg is a constant (no gradient); acc and depth are
 * forward outputs only (no gradient flows into them).
 * A NULL lnb_composite, or one that asks for nothing (background 0, acc and depth NULL), is exactly lnb_nerf_step: the
 * same kernels, the same bits.  Otherwise: LNB_PATH_TC runs the fused kernels' extras instantiations (or the wide path);
 * the exact path runs on the layerwise fp32 kernels (the fused exact kernel has no extras).  LNB_ERR_ARG for depth in
 * features mode, background not 0 or 1, or a non-finite bg.  The compat symbols keep the reference's compositing. */
typedef struct {
    int background;      /* 0: none (the reference's compositing); 1: composite onto bg */
    float bg[3];
    float *acc;          /* [R] overwritten, or NULL (device pointer; host pointer for the *_host call) */
    float *depth;        /* [R] overwritten, or NULL (rays / camera mode only)                           */
} lnb_composite;
LNB_API int lnb_nerf_step_composite(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args, const lnb_composite *comp);
LNB_API int lnb_nerf_step_composite_host(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args, const lnb_composite *comp);
/* Fills out[0..n) with {sizeof(lnb_composite), offsetof background, bg, acc, depth}; returns how many values exist. */
LNB_API int lnb_composite_layout(int *out, int n);

/* VIEWS MODE (nerf only): camera mode with a pose per ray, so that one batch can mix rays from every training view (the NeRF
 * paper's "random rays from all images" batching) and a step's whole batch can be drawn on the device (lnb_views_draw).
 * Ray r is camera mode's ray of pixel q = pixels[r] under the pose poses[view[r]]: direction, origin, linspace depths, dists
 * and the view direction follow the lnb_camera rule unchanged, with c2w = poses[view[r]].  The stratified jitter is
 * u = lnb_uniform(seed', g, s) with the 64-bit key g = view[r] * P + q (P = width * height) and seed' = *seed_dev when
 * seed_dev is set, else seed.  So:
 *   - with every ray on view 0, views mode is camera mode with that pose (pixels = the same list), bit for bit;
 *   - with linspace depths that holds for any single view v.
 * view[r] and pixels[r] are checked on the device: an index outside [0, n_views) or [0, P) makes that ray's colour, and so the
 * loss, NaN (nothing outside the pose table is read).  LNB_ERR_ARG for NULL pointers when R > 0, n_views < 1, width < 2,
 * height < 1, P >= 2^31, a zero focal length or S > 4096.  All pointers are device pointers; the struct itself is a host
 * pointer (passed to the kernels by value). */
typedef struct {
    const double *poses;                 /* [n_views][12] c2w rows, as lnb_camera.c2w                          */
    int n_views, width, height;          /* every view has the same pixel grid; P = width * height             */
    double fx, fy, cx, cy, near, far;    /* shared normalised intrinsics and depth range, as lnb_camera        */
    int stratified;
    unsigned long long seed;             /* jitter seed ...                                                    */
    const unsigned long long *seed_dev;  /* ... or, when non-NULL, read from device memory (lnb_views_draw's step_seed) */
    const int *view, *pixels;            /* [R] per ray                                                        */
} lnb_views;
/* Fills out[0..n) with {sizeof(lnb_views), offsetof poses, n_views, fx, near, stratified, seed, seed_dev, view, pixels};
 * returns how many values exist. */
LNB_API int lnb_views_layout(int *out, int n);
/* The step for a views batch: args has no X, rays or cam (LNB_ERR_ARG otherwise); comp is optional (lnb_composite, the depth
 * being views mode's).  Device pointers, asynchronous on the context's stream. */
LNB_API int lnb_nerf_step_views(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args, const lnb_views *views,
                                const lnb_composite *comp);
/* The rays and sample depths views mode generates (any output may be NULL): rays_o, rays_d [R][3], t [R][S] float64.  A ray
 * with an out-of-range index gets NaN.  Device pointers (views itself is a host pointer). */
LNB_API int lnb_views_rays(lnb_ctx *ctx, const lnb_views *views, int R, int S, double *rays_o, double *rays_d, double *t);
/* THE DRAW: one step's batch from a device-resident scene, images [n_views][P][3] float32.  It reads k = counter[0] and leaves
 * counter[0] = k + 1 (counter[1] is the draw's own block ticket: 0 before the first call, left at 0), so every replay of a
 * captured graph draws a new batch.  With z(k, i) = mix(seed + 0x9E3779B97F4A7C15 * (k * 2^32 + i + 1)) mod 2^64, mix the
 * SplitMix64 finaliser of lnb_uniform, and umulhi(z, n) the high 64 bits of the 128-bit product z * n:
 *   one_view == 0 (every view, the paper's batching): g_r = umulhi(z(k, r), n_views * P), view_r = g_r / P, pixels_r = g_r mod P;
 *   one_view != 0 (one view per step, the paper's Blender protocol): v = umulhi(z(k, 2^32 - 1), n_views), view_r = v,
 *                 pixels_r = umulhi(z(k, r), P);
 *   *step_seed = z(k, 2^32 - 2) (the step's jitter seed: lnb_views.seed_dev = step_seed);
 *   target_r   = images[view_r][pixels_r] (the bits copied).
 * R < 2^32 - 2.  The draw never lets a dependent launch start early (no programmatic trigger): the fused train kernel builds
 * its first tile's inputs before it waits for its predecessor, so a step launched right after the draw only starts once the
 * batch is complete.  Device pointers. */
LNB_API int lnb_views_draw(lnb_ctx *ctx, const float *images, int n_views, long long P, int R, int one_view,
                           unsigned long long seed, unsigned long long *counter, int *view, int *pixels, float *target,
                           unsigned long long *step_seed);
/* umulhi(z(k, i), n) of the draw, host-callable (like lnb_uniform): the draw's rule without a GPU. */
LNB_API unsigned long long lnb_views_pick(unsigned long long seed, unsigned long long k, unsigned long long i,
                                          unsigned long long n);

/* Positional encoding, pos_encoding.py:4-70: x [n][F] float64 -> out [n][F*(1+2E)] float32,
 * feature = slot*F + coord, slot 0 identity, 2i+1 sin(2^i x), 2i+2 cos(2^i x); float64 range
 * reduction so the result matches the reference's float64-then-cast values. Device pointers. */
LNB_API int lnb_pos_encoding(lnb_ctx *ctx, const double *x, long long n, int F, int E, float *out);
/* Sample generation + encoding, train_nerf.py:289-311 + pos_encoding.py:38-70:
 * pts = o + d*t (float64), X = PE(pts) float32 [R*S][3+6E], dists [R][S] = t[s+1]-t[s], last 1e8.
 * rays_o, rays_d [R][3] float64, t [R][S] float64. Device pointers. */
LNB_API int lnb_sample_encode(lnb_ctx *ctx, const double *rays_o, const double *rays_d, const double *t,
                      int R, int S, int E, float *X, float *dists);
/* The same with the view direction (E_dir >= 0): X [R*S][(3+6E) + (3+6E_dir)] = [PE(pts, E) | PE(u, E_dir)], u the unit
 * direction of rays_d as rays mode defines it (pe_bands in lnb_step_args).  The input a features-mode step of a net with
 * view directions expects.  Device pointers. */
LNB_API int lnb_sample_encode_dirs(lnb_ctx *ctx, const double *rays_o, const double *rays_d, const double *t,
                                   int R, int S, int E, int E_dir, float *X, float *dists);

/* The rays and sample depths camera mode generates, written out (any pointer may be NULL): rays_o, rays_d [R][3], t [R][S]
 * float64.  Device pointers (cam itself is a host pointer). */
LNB_API int lnb_camera_rays(lnb_ctx *ctx, const lnb_camera *cam, int R, int S, double *rays_o, double *rays_d, double *t);

/* out[i] = (unsigned char) rint(255 * clamp(rgb[i], 0, 1)), i < n: what the hosts do before writing a PNG / video frame
 * (train_nerf.py:686-700), so that a rendered frame leaves the device as 3 bytes per pixel.  Device pointers. */
LNB_API int lnb_color_to_u8(lnb_ctx *ctx, const float *rgb, long long n, unsigned char *out);

/* c[a_h][b_w] += a[a_h][a_w] * b[a_w][b_w]; device pointers (scripts/mlp_fit.py:150-172). */
LNB_API int lnb_mult_a_b(lnb_ctx *ctx, const float *a, int a_h, int a_w, const float *b, int b_w, float *c);

/* Optimisers the reference hosts apply to the padded arrays (SURVEY.md 8 a11), n floats each.
 * lnb_adam_step reproduces AdamOptimizer.update (train_nerf.py:133-161) including its double
 * bias correction; t is the 1-based step count AFTER increment.  lnb_sgd_step: p -= lr * g
 * (fit_img.py:512-513).  Device pointers.  The hyper-parameters are doubles because the
 * reference holds them as Python floats and derives (1-beta), the bias corrections and lr_t in
 * double before they meet the float32 arrays. */
LNB_API int lnb_adam_step(lnb_ctx *ctx, float *param, const float *grad, float *m, float *v, long long n,
                  int t, double lr, double beta1, double beta2, double eps);
/* Same update with the step counter kept on the device (t = *t_dev + 1, then *t_dev += 1), so a
 * whole train step can be captured in a CUDA graph and replayed. */
LNB_API int lnb_adam_step_dev(lnb_ctx *ctx, float *param, const float *grad, float *m, float *v, long long n,
                      int *t_dev, double lr, double beta1, double beta2, double eps);
LNB_API int lnb_sgd_step(lnb_ctx *ctx, float *param, const float *grad, long long n, double lr);

/* ------------------------------------------------------------------------------------------
 * Device-resident training state (the hosts' per-chunk "grad call, then optimiser on the padded
 * arrays" loop, train_nerf.py:395-499 / fit_img.py:468-513, without leaving the GPU).
 * A batch is an lnb_step_args with DEVICE pointers; its ws, bs, d_*, loss and by-product fields are
 * ignored (the trainer supplies them).  lnb_trainer_step = gradient + optimiser update (two kernel
 * launches on the tensor-core path).  For data-parallel training split it:
 * lnb_trainer_grad -> all-reduce lnb_trainer_grad_buffer ([d_ws | d_bs | loss], written, not
 * accumulated) over the ranks -> lnb_trainer_apply.
 * ------------------------------------------------------------------------------------------ */
typedef struct lnb_trainer lnb_trainer;
enum { LNB_OPT_ADAM = 0,  /* AdamOptimizer.update, train_nerf.py:133-161 (double bias correction) */
       LNB_OPT_SGD = 1 }; /* p -= lr * g, fit_img.py:512-513                                      */
LNB_API int lnb_trainer_create(lnb_ctx *ctx, const lnb_mlp *mlp, const float *ws_host, const float *bs_host,
                       int optimizer, double lr, double beta1, double beta2, double eps, lnb_trainer **out);
LNB_API void lnb_trainer_destroy(lnb_trainer *t);
LNB_API int lnb_trainer_step(lnb_trainer *t, const lnb_step_args *batch, int nerf);
/* lnb_trainer_step, and also writes this step's forward compositing weights w_s = alpha_s * T_s (at the
 * pre-update parameters) into weights [R][S] (device, overwritten).  nerf batches only.  On the tensor-core path the fused
 * train kernel or the wide path writes them, whichever the step runs on; the fused exact kernel writes none, so an
 * exact-path step with weights runs on the layerwise fp32 kernels (the same arithmetic to <= 1e-5). */
LNB_API int lnb_trainer_step_weights(lnb_trainer *t, const lnb_step_args *batch, int nerf, float *weights);
/* the same step with the batch in HOST memory (pinned buffers are copied from directly): stages
 * host->device, steps, returns the loss through *loss_out; synchronous */
LNB_API int lnb_trainer_step_host(lnb_trainer *t, const lnb_step_args *batch, int nerf, float *loss_out);
/* PIPELINED host-buffer steps (the hosts' chunk loop, train_nerf.py:275-499, with the copy of batch i+1 under the step
 * of batch i): lnb_trainer_submit_host stages the batch on a copy stream into one of two device staging slots, enqueues the
 * step behind it and returns without waiting for the GPU.  Pinned host buffers are read by the DMA engine directly and must
 * stay unchanged until the submission after next has returned (or until lnb_trainer_wait); pageable buffers are copied to a
 * pinned bounce slot before the call returns.  lnb_trainer_wait blocks until every submitted step has finished and copies
 * the losses of the steps submitted since the previous wait, oldest first, into losses[0 .. *n_out) (at most max_losses of
 * the newest 4096; losses may be NULL).  Errors of a poisoned peer exchange surface at lnb_trainer_wait. */
LNB_API int lnb_trainer_submit_host(lnb_trainer *t, const lnb_step_args *batch, int nerf);
LNB_API int lnb_trainer_wait(lnb_trainer *t, float *losses, int max_losses, int *n_out);
LNB_API int lnb_trainer_grad(lnb_trainer *t, const lnb_step_args *batch, int nerf);
/* Composite every later nerf step of this trainer (step, step_weights, step_host, submit_host, grad) onto the background
 * colour rgb (3 floats; see lnb_composite), whichever kernels the step runs on; NULL restores the reference's compositing
 * (a trainer that never had a background set runs exactly as before).  The term is per ray, so the peer all-reduce is
 * unaffected, but every rank of a data-parallel run must set the same background.  LNB_ERR_ARG for a non-finite value. */
LNB_API int lnb_trainer_set_background(lnb_trainer *t, const float *rgb);
/* Attach a views batch (lnb_views, copied; its buffers must live as long as it is attached): from then on a nerf batch with
 * no X, rays or cam is a views batch on lnb_trainer_step, lnb_trainer_step_weights and lnb_trainer_grad (so the NCCL route
 * works too).  lnb_trainer_step_host and lnb_trainer_submit_host refuse such a batch (the scene lives on the device).  NULL
 * detaches it.  LNB_ERR_ARG for the cases lnb_views lists. */
LNB_API int lnb_trainer_set_views(lnb_trainer *t, const lnb_views *views);
LNB_API int lnb_trainer_apply(lnb_trainer *t);
LNB_API float *lnb_trainer_grad_buffer(lnb_trainer *t, long long *n_floats);
LNB_API float *lnb_trainer_params(lnb_trainer *t, long long *n_w, long long *n_b);
/* Peer-memory gradient all-reduce for the ranks of one box (one process per GPU), fused into the
 * tensor-core step's reduction kernel: every rank exports a 64-byte CUDA IPC handle of its exchange
 * buffer, the host exchanges the handles (any transport), every rank attaches all `world` handles
 * (rank-major, 64 bytes each).  From then on lnb_trainer_step[_host] sums the gradients (and the
 * loss) of all ranks over NVLink inside its second kernel -- no separate collective -- and all ranks
 * must step in lockstep; with LNB_SEED_LOSS the gradient is (sum of losses) x (sum of unit-seed
 * gradients), the reference's gradient of the whole batch.  Steps that cannot exchange in-kernel
 * (fp32 path, wide MLPs, S > 128) return LNB_ERR_UNSUPPORTED instead of updating from local
 * gradients.  A peer that stays silent for LNB_PEER_TIMEOUT_MS (default 5000) poisons that step:
 * gradients, parameters and the returned loss become NaN, lnb_trainer_step_host / lnb_trainer_read
 * return LNB_ERR_CUDA and lnb_trainer_comm_status returns 1 (0 = fine). */
LNB_API int lnb_trainer_comm_export(lnb_trainer *t, void *handle64);
LNB_API int lnb_trainer_comm_attach(lnb_trainer *t, int rank, int world, const void *handles);
LNB_API int lnb_trainer_comm_status(lnb_trainer *t);
/* synchronises; any pointer may be NULL */
LNB_API int lnb_trainer_read(lnb_trainer *t, float *ws_host, float *bs_host, float *loss_host);

/* Process-wide default context used by the compat symbols (created lazily on first call,
 * device from LOMA_NERF_B200_DEVICE or 0). Returns NULL when no CUDA device is usable. */
LNB_API lnb_ctx *lnb_default_ctx(void);

#ifdef __cplusplus
}
#endif
#endif /* LOMA_NERF_B200_H */
