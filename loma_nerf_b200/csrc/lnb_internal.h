// lnb_internal.h -- shared between the translation units of libloma_nerf_b200.so.
// Not part of the ABI (see include/loma_nerf_b200.h for that).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/loma_nerf_b200.h"

struct lnb_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;     // stream work is issued on
    cudaStream_t own_stream = nullptr; // created by lnb_create
    // device arena (grow-only), carved per call
    char *arena = nullptr;
    size_t arena_cap = 0, arena_off = 0;
    // pinned host staging (grow-only) for the *_host and compat entry points
    char *pinned = nullptr;
    size_t pinned_cap = 0, pinned_off = 0;
    // device staging that mirrors the pinned block for the *_host entry points
    char *dstage = nullptr;
    size_t dstage_cap = 0;
    long long launches = 0;
    int *tc_counter = nullptr; // tile-scheduler counter of the fused kernel (zero between launches)
    std::string err;
    // optional timing of the dominant (fused) kernel: CUDA-event pairs around each launch
    bool prof_on = false;
    std::vector<cudaEvent_t> prof_ev; // [2*i] start, [2*i+1] stop
    size_t prof_used = 0;
    std::string prof_name;
};

// time the next launch of the dominant kernel when profiling is enabled (api_flat.cu)
void lnb_prof_begin(lnb_ctx *ctx, const char *name);
void lnb_prof_end(lnb_ctx *ctx);

#define LNB_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e__);                     \
            return LNB_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

#define LNB_CHECK_LAUNCH()                                                                      \
    do {                                                                                        \
        ctx->launches++;                                                                        \
        cudaError_t e__ = cudaGetLastError();                                                   \
        if (e__ != cudaSuccess) {                                                               \
            ctx->err = std::string("kernel launch: ") + cudaGetErrorString(e__);                \
            return LNB_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

#define LNB_ARG(cond, msg)                                                                      \
    do {                                                                                        \
        if (!(cond)) {                                                                          \
            ctx->err = std::string("bad argument: ") + (msg);                                   \
            return LNB_ERR_ARG;                                                                 \
        }                                                                                       \
    } while (0)

#define LNB_TRY(call)                                                                           \
    do {                                                                                        \
        int rc__ = (call);                                                                      \
        if (rc__ != LNB_OK) return rc__;                                                        \
    } while (0)

// arena helpers (api_flat.cu).  reserve() may reallocate (synchronises the stream first) and
// resets the carve offset; take() carves 256 B aligned blocks from what reserve() guaranteed.
int lnb_arena_reserve(lnb_ctx *ctx, size_t bytes);
void *lnb_arena_take(lnb_ctx *ctx, size_t bytes);
int lnb_pinned_reserve(lnb_ctx *ctx, size_t bytes);
void *lnb_pinned_take(lnb_ctx *ctx, size_t bytes);

// activation kinds for the linear-layer epilogue
enum { ACT_NONE = 0, ACT_RELU = 1, ACT_SIGMOID = 2, ACT_NERF_HEAD = 3 };

// ---- fp32 CUDA-core kernels (kernels_f32.cu) ------------------------------------------------
// Row GEMM  C[i][n] = epi( sum_kk A[i][kk] * B(kk,n) ),  i < rows, n < n_dim, kk < k_dim with
// B(kk,n) = Bp[kk*sbk + n*sbn] (so both W and W^T are addressed from the one padded copy).
//   a_rows : rows of A that exist (rows >= a_rows multiply as zeros; nerf.py:81 vs :95)
//   bias   : added when != NULL
//   acc    : C read first and added (the reference accumulates onto the caller's scratch)
//   act    : ACT_* applied after bias (forward)
//   mask   : when != NULL the result is zeroed where mask[i][n] <= 0 (ReLU adjoint)
struct lnb_gemm_args {
    const float *A; int lda; int a_rows;
    const float *B; long long sbk, sbn;
    float *C; int ldc;
    int rows, n_dim, k_dim;
    const float *bias; int acc; int act;
    const float *mask; int ldmask;
};
int lnb_launch_row_gemm(lnb_ctx *ctx, const lnb_gemm_args &g);

// Weight-gradient contraction over rows (SURVEY.md 8 a7: d_ws[l] += H^T dZ, d_bs[l] += colsum):
// partial[z][k][j] = sum_{i in chunk z} Haug[i][k] dZ[i][j], k <= in_dim, where Haug[i][in_dim]=1
// (that extra row is the bias gradient).  partial is [n_chunks][in_dim+1][out_dim] dense.
int lnb_launch_dw_partials(lnb_ctx *ctx, const float *H, int ldh, const float *dZ, int ldz,
                           float *partial, int in_dim, int out_dim, int rows, int n_chunks);
// d_w[k*ldw + j] += scale * sum_z partial[z][k][j] (k < in_dim); d_b[j] += scale * sum_z
// partial[z][in_dim][j].  scale = seed_dev ? seed_dev[0] : 1 (then times seed_value).
int lnb_launch_dw_reduce(lnb_ctx *ctx, const float *partial, int n_chunks, int in_dim,
                         int out_dim, float *d_w, int ldw, float *d_b, float seed_value,
                         const float *seed_dev);

// compositing forward: one warp per ray (scripts/nerf.py:176-288). ray_sse[r] = sum_c (col-t)^2
// (0 when target == NULL).  Any of rgba/alpha/cumprod/weights may be NULL.  color is read first
// when color_accumulate (nerf.py:284-286 adds onto the caller's buffer).
// cx (NULL: the reference's compositing) adds the extras of lnb_composite: the background term, acc / depth outputs.
struct lnb_comp_args;
int lnb_launch_composite_fwd(lnb_ctx *ctx, const float *head, int ldh, const float *dists,
                             const float *target, int R, int S, float *rgba, float *alpha,
                             float *cumprod, float *weights, float *color, int color_accumulate,
                             float *ray_sse, const lnb_comp_args *cx = nullptr);
// compositing backward with UNIT seed (the caller scales): from head (post-activation), dists,
// the final colour and target writes dZ_head[i][0..3] = adjoint of the head's PRE-activation
// (sigmoid'/ReLU mask applied), and when non-NULL d_dists_u [R][S], d_color_u [R][3]
// (= 2 (c - t)); d_target = -d_color.
int lnb_launch_composite_bwd(lnb_ctx *ctx, const float *head, int ldh, const float *dists,
                             const float *target, const float *color, int R, int S,
                             float *dZ_head, int ldz, int out_dim, float *d_dists_u,
                             float *d_color_u, const lnb_comp_args *cx = nullptr);
// out[0] = sum_i v[i]  (fixed order, one block)
int lnb_launch_sum(lnb_ctx *ctx, const float *v, long long n, float *out);
// mlp_fit loss terms: ray_sse[r] = sum_{c<Wt} (pred[r][c]-t[r][c])^2 (scripts/mlp_fit.py:140-145)
int lnb_launch_fit_loss(lnb_ctx *ctx, const float *pred, int ldp, const float *target, int R,
                        int Wt, float *ray_sse);
// mlp_fit head adjoint, unit seed: dZ[i][j] = (i<R && j<Wt ? 2 (y-t) : 0) * y(1-y), j < out_dim,
// i < rows; d_color_u [R][Wt] = 2 (y - t) when non-NULL.
int lnb_launch_fit_head_bwd(lnb_ctx *ctx, const float *pred, int ldp, const float *target, int R,
                            int Wt, int rows, int out_dim, float *dZ, int ldz, float *d_color_u);
int lnb_launch_fill(lnb_ctx *ctx, float *p, size_t n, float v);
// dst[i*ldd + j] += sign * scale * src[i*lds + j], i < rows, j < cols; scale as in dw_reduce
int lnb_launch_axpy2d(lnb_ctx *ctx, float *dst, long long ldd, const float *src, long long lds,
                      long long rows, int cols, float sign, float seed_value,
                      const float *seed_dev);

// The per-step carrier from the entry points to each route: the compositing extras (lnb_composite) of one step as the kernels
// take them, and the per-ray poses of a views batch.  The depths are the ones the encoder used: rays mode t (float64 or
// float32), camera and views mode the camera (its depths re-derived per sample), features mode none.
struct lnb_comp_args {
    int extras = 0;                // 1: background, acc or depth asked for (the extras kernels); 0: a plain views step
    int background = 0;
    float bg[3] = {0.f, 0.f, 0.f};
    float *acc = nullptr, *depth = nullptr;
    const void *t = nullptr;       // rays mode: [R][S] sample depths
    int t_f64 = 0;
    const lnb_camera *cam = nullptr; // camera and views mode (host pointer; its pixel list is a device pointer)
    const lnb_views *views = nullptr; // views mode (host pointer): the step's cam holds the views' shared fields (views_camera)
};
// NULL when comp asks for nothing and there is no views batch (the step is then exactly lnb_nerf_step), else the carrier with
// the depth source of step a filled in; LNB_ERR_ARG for the cases lnb_composite lists (api_flat.cu)
int lnb_comp_resolve(lnb_ctx *ctx, const lnb_step_args *a, bool nerf, const lnb_composite *comp, const lnb_views *views,
                     lnb_comp_args *out, const lnb_comp_args **resolved);
// a views batch of R rays, S samples: LNB_ERR_ARG for the cases lnb_views lists (api_flat.cu)
int lnb_views_check(lnb_ctx *ctx, const lnb_views *v, int R, int S);
inline bool lnb_cx_extras(const lnb_comp_args *cx) { return cx && cx->extras; }
inline const lnb_views *lnb_cx_views(const lnb_comp_args *cx) { return cx ? cx->views : nullptr; }

// ---- fused_tc.cu ---------------------------------------------------------------------------
// Optional extras of the fused tensor-core step, used by the trainer (trainer.cu):
//   wimg            : a valid weight image (skips the per-step prep kernel)
//   overwrite_grads : d_ws / d_bs are written (=) instead of accumulated (+=)
//   fuse_adam       : the reduce kernel applies the reference's Adam update to (param, m, v) with
//                     the device step counter and refreshes `wimg_out` (the next step's image)
// peer-memory all-reduce state of one rank (trainer.cu sets it up; fused_tc.cu uses it)
struct lnb_tc_comm {
    int world = 0, rank = 0;
    int n_slot = 0;                          // gradient elements + 1 (the loss)
    unsigned long long *my_recv = nullptr;   // [2 parities][world senders][n_slot] {step<<32 | float bits}
    unsigned long long *peer_recv[8] = {};   // the same array on every rank (peer-mapped; [rank] = own)
    int *status = nullptr;                   // local, sticky: 1 after a peer timed out (that step is poisoned with NaN)
    unsigned long long timeout_ns = 5000000000ull; // LNB_PEER_TIMEOUT_MS
};

struct lnb_tc_extra {
    const lnb_tc_comm *comm = nullptr; // when set (and fuse_adam): gradients are summed over the ranks
    const void *wimg = nullptr;
    int overwrite_grads = 0;
    int fuse_adam = 0;
    float *param = nullptr, *m = nullptr, *v = nullptr; // flat [ws | bs] padded layout
    int *t_dev = nullptr;                               // incremented by the fused kernel
    double lr = 0, b1 = 0, b2 = 0, eps = 0;
    void *wimg_out = nullptr;
    float *weights = nullptr;                           // train kernels: [R][S] compositing weights w_s = alpha_s T_s
};
// cx: the compositing extras (lnb_comp_resolve), or NULL
int lnb_fused_tc_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf,
                      const lnb_tc_extra *ex, const lnb_comp_args *cx = nullptr);
// validated dispatch of one step with tensor-core extras and / or compositing extras (api_flat.cu)
int lnb_step_ex(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, const lnb_tc_extra *ex,
                const lnb_composite *comp = nullptr, const lnb_views *views = nullptr);
// layerwise tensor-core step for wide MLPs (wide_tc.cu); LNB_ERR_UNSUPPORTED when it does not apply
int lnb_wide_tc_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, const lnb_comp_args *cx = nullptr);
// padded widths of the fused kernel for this MLP, 0 when unsupported; bytes of its weight image
int lnb_tc_layout(const lnb_mlp *mlp, int *HP, int *K0P, int *wimg_bytes);
// build the weight image from fp32 padded weights (one small kernel)
int lnb_tc_prep(lnb_ctx *ctx, const lnb_mlp *mlp, const float *ws, const float *bs, void *wimg);
// Adam on the flat padded params with a device step counter (*t_dev already incremented), then
// refresh of the weight image (when wimg != NULL)
int lnb_tc_adam_img(lnb_ctx *ctx, const lnb_mlp *mlp, float *param, const float *grad, float *m, float *v,
                    const int *t_dev, double lr, double b1, double b2, double eps, void *wimg);

// ---- fused_f32.cu: the fused exact (fp32 CUDA-core) step for the reference's own network shapes; LNB_ERR_UNSUPPORTED
// when the problem (or the outputs asked for) does not fit it
// (it has no compositing extras: a step with lnb_cx_extras(cx) is LNB_ERR_UNSUPPORTED there and runs on the layerwise kernels)
int lnb_fused_f32_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, int overwrite,
                       const lnb_comp_args *cx = nullptr);
int lnb_step_f32_fused(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, int overwrite,
                       const lnb_views *views = nullptr);   // validated (api_flat.cu)

// ---- encode.cu / optim.cu ---------------------------------------------------------------------
// Rays and camera mode: the input form the MLP's input width selects (include/loma_nerf_b200.h).  Returns the direction
// band count E_d >= 0 when c_in == (3 + 6E) + (3 + 6E_d), LNB_DIRS_NONE when c_in == 3 + 6E (positions only), and
// LNB_DIRS_BAD for any other width.  One width is odd, the other even: they cannot be confused.
constexpr int LNB_DIRS_NONE = -1, LNB_DIRS_BAD = -2;
inline int lnb_rays_dir_bands(int c_in, int E)
{
    if (E < 0) return LNB_DIRS_BAD;
    const int rest = c_in - (3 + 6 * E);
    if (rest == 0) return LNB_DIRS_NONE;
    return rest >= 3 && (rest - 3) % 6 == 0 ? (rest - 3) / 6 : LNB_DIRS_BAD;
}
// Ed: direction bands (LNB_DIRS_NONE: positions only); rows are [PE(x, E) | PE(u, Ed)]
int lnb_launch_pos_encoding(lnb_ctx *ctx, const double *x, long long n, int F, int E, float *out);
int lnb_launch_sample_encode(lnb_ctx *ctx, const void *o, const void *d, const void *t, int f64,
                             int R, int S, int E, int Ed, float *X, float *dists);
int lnb_launch_sample_encode_bf16(lnb_ctx *ctx, const void *o, const void *d, const void *t, int f64,
                                  int R, int S, int E, int Ed, float *X, float *dists, void *Xb, int ldb);
// camera mode (lnb_camera): features / dists (or the wide path's bf16 rows) straight from the pose; views mode (lnb_views)
// when views != NULL, cam then holding its shared fields
int lnb_launch_camera_encode(lnb_ctx *ctx, const lnb_camera *cam, const lnb_views *views, int R, int S, int E, int Ed, float *X,
                             float *dists, void *Xb, int ldb);
int lnb_launch_adam(lnb_ctx *ctx, float *p, const float *g, float *m, float *v, long long n, int t,
                    double lr, double b1, double b2, double eps);
int lnb_launch_adam_dev(lnb_ctx *ctx, float *p, const float *g, float *m, float *v, long long n,
                        int *t_dev, double lr, double b1, double b2, double eps);
int lnb_launch_incr(lnb_ctx *ctx, int *t_dev);
int lnb_launch_adam_at(lnb_ctx *ctx, float *p, const float *g, float *m, float *v, long long n,
                       const int *t_dev, double lr, double b1, double b2, double eps);
int lnb_launch_sgd(lnb_ctx *ctx, float *p, const float *g, long long n, double lr);
