// api_flat.cu -- context management and the FLAT entry points of libloma_nerf_b200.so
// (include/loma_nerf_b200.h section 2).  The step functions follow
// /root/reference/scripts/nerf.py:67-304 and scripts/mlp_fit.py:39-147 and their reverse
// (SURVEY.md Appendix B).  There is no CPU path here: every function needs a CUDA device.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "camera.cuh"
#include "lnb_internal.h"

// ------------------------------------------------------------------------------------------------
// context / memory
// ------------------------------------------------------------------------------------------------
static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int lnb_arena_reserve(lnb_ctx *ctx, size_t bytes)
{
    ctx->arena_off = 0;
    if (bytes <= ctx->arena_cap) return LNB_OK;
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->arena) LNB_CUDA(cudaFree(ctx->arena));
    ctx->arena = nullptr;
    ctx->arena_cap = 0;
    size_t cap = align_up(bytes + bytes / 4, 1 << 20);
    LNB_CUDA(cudaMalloc((void **)&ctx->arena, cap));
    ctx->arena_cap = cap;
    return LNB_OK;
}

void *lnb_arena_take(lnb_ctx *ctx, size_t bytes)
{
    size_t off = align_up(ctx->arena_off, 256);
    if (off + bytes > ctx->arena_cap) return nullptr;
    ctx->arena_off = off + bytes;
    return ctx->arena + off;
}

int lnb_pinned_reserve(lnb_ctx *ctx, size_t bytes)
{
    ctx->pinned_off = 0;
    if (bytes <= ctx->pinned_cap) return LNB_OK;
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->pinned) LNB_CUDA(cudaFreeHost(ctx->pinned));
    ctx->pinned = nullptr;
    ctx->pinned_cap = 0;
    size_t cap = align_up(bytes + bytes / 4, 1 << 20);
    LNB_CUDA(cudaMallocHost((void **)&ctx->pinned, cap));
    ctx->pinned_cap = cap;
    return LNB_OK;
}

void *lnb_pinned_take(lnb_ctx *ctx, size_t bytes)
{
    size_t off = align_up(ctx->pinned_off, 256);
    if (off + bytes > ctx->pinned_cap) return nullptr;
    ctx->pinned_off = off + bytes;
    return ctx->pinned + off;
}

static int dstage_reserve(lnb_ctx *ctx, size_t bytes)
{
    if (bytes <= ctx->dstage_cap) return LNB_OK;
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->dstage) LNB_CUDA(cudaFree(ctx->dstage));
    ctx->dstage = nullptr;
    ctx->dstage_cap = 0;
    size_t cap = align_up(bytes + bytes / 4, 1 << 20);
    LNB_CUDA(cudaMalloc((void **)&ctx->dstage, cap));
    ctx->dstage_cap = cap;
    return LNB_OK;
}

extern "C" int lnb_abi_version(void) { return LNB_ABI_VERSION; }

extern "C" int lnb_struct_layout(int *out, int n)
{
    const int v[] = {(int)sizeof(lnb_mlp), (int)sizeof(lnb_step_args),
                     (int)offsetof(lnb_step_args, X), (int)offsetof(lnb_step_args, inter),
                     (int)offsetof(lnb_step_args, rgba), (int)offsetof(lnb_step_args, loss),
                     (int)offsetof(lnb_step_args, want_grad), (int)offsetof(lnb_step_args, d_ws),
                     (int)offsetof(lnb_step_args, path), (int)offsetof(lnb_step_args, rays_o),
                     (int)offsetof(lnb_step_args, pe_bands), (int)offsetof(lnb_step_args, cam),
                     (int)sizeof(lnb_camera), (int)offsetof(lnb_camera, pixels)};
    const int k = (int)(sizeof(v) / sizeof(v[0]));
    for (int i = 0; i < k && i < n; ++i) out[i] = v[i];
    return k;
}

extern "C" int lnb_composite_layout(int *out, int n)
{
    const int v[] = {(int)sizeof(lnb_composite), (int)offsetof(lnb_composite, background), (int)offsetof(lnb_composite, bg),
                     (int)offsetof(lnb_composite, acc), (int)offsetof(lnb_composite, depth)};
    const int k = (int)(sizeof(v) / sizeof(v[0]));
    for (int i = 0; i < k && i < n; ++i) out[i] = v[i];
    return k;
}

extern "C" int lnb_views_layout(int *out, int n)
{
    const int v[] = {(int)sizeof(lnb_views), (int)offsetof(lnb_views, poses), (int)offsetof(lnb_views, n_views),
                     (int)offsetof(lnb_views, fx), (int)offsetof(lnb_views, near), (int)offsetof(lnb_views, stratified),
                     (int)offsetof(lnb_views, seed), (int)offsetof(lnb_views, seed_dev), (int)offsetof(lnb_views, view),
                     (int)offsetof(lnb_views, pixels)};
    const int k = (int)(sizeof(v) / sizeof(v[0]));
    for (int i = 0; i < k && i < n; ++i) out[i] = v[i];
    return k;
}

int lnb_views_check(lnb_ctx *ctx, const lnb_views *v, int R, int S)
{
    LNB_ARG(v, "views: null");
    LNB_ARG(R == 0 || (v->poses && v->view && v->pixels), "views: poses, view and pixels are required");
    LNB_ARG(v->n_views >= 1, "views: n_views >= 1");
    LNB_ARG(v->width >= 2 && v->height >= 1, "views: width >= 2, height >= 1");
    LNB_ARG((long long)v->width * v->height < (1ll << 31), "views: fewer than 2^31 pixels per view");
    LNB_ARG(v->fx != 0.0 && v->fy != 0.0, "views: zero focal length");
    LNB_ARG(S <= 4096, "views: at most 4096 samples per ray");
    return LNB_OK;
}

int lnb_comp_resolve(lnb_ctx *ctx, const lnb_step_args *a, bool nerf, const lnb_composite *comp, const lnb_views *views,
                     lnb_comp_args *out, const lnb_comp_args **resolved)
{
    *resolved = nullptr;
    if (comp) {
        LNB_ARG(comp->background == 0 || comp->background == 1, "composite: background must be 0 or 1");
        if (comp->background)
            for (int c = 0; c < 3; ++c) LNB_ARG(isfinite(comp->bg[c]), "composite: non-finite background colour");
    }
    const bool extras = comp && (comp->background || comp->acc || comp->depth);
    if (!extras && !views) return LNB_OK;   // asks for nothing: the plain step
    LNB_ARG(nerf, "composite / views: a nerf-step feature");
    const bool cam = !a->X && !a->rays_o && a->cam;
    const bool rays = !a->X && (a->rays_o || cam);
    LNB_ARG(!extras || !comp->depth || rays, "composite: depth needs rays or camera mode (features mode has no sample depths)");
    *out = lnb_comp_args{};
    out->views = views;
    if (cam) out->cam = a->cam;
    else if (rays) { out->t = a->t; out->t_f64 = a->ray_dtype == LNB_RAY_F64; }
    if (extras) {
        out->extras = 1;
        out->background = comp->background;
        for (int c = 0; c < 3; ++c) out->bg[c] = comp->background ? comp->bg[c] : 0.0f;
        out->acc = comp->acc;
        out->depth = comp->depth;
    }
    *resolved = out;
    return LNB_OK;
}

extern "C" int lnb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int lnb_create(lnb_ctx **out, int device)
{
    if (!out) return LNB_ERR_ARG;
    *out = nullptr;
    int n = lnb_device_count();
    if (n <= 0) return LNB_ERR_CUDA;
    if (device < 0) {
        if (cudaGetDevice(&device) != cudaSuccess) return LNB_ERR_CUDA;
    }
    if (device >= n) return LNB_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return LNB_ERR_CUDA;
    lnb_ctx *ctx = new lnb_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return LNB_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    *out = ctx;
    return LNB_OK;
}

extern "C" void lnb_destroy(lnb_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->arena) cudaFree(ctx->arena);
    if (ctx->dstage) cudaFree(ctx->dstage);
    if (ctx->tc_counter) cudaFree(ctx->tc_counter);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    for (cudaEvent_t e : ctx->prof_ev) cudaEventDestroy(e);
    delete ctx;
}

extern "C" int lnb_set_stream(lnb_ctx *ctx, void *stream)
{
    if (!ctx) return LNB_ERR_ARG;
    // (void*)-1 selects the context's own non-blocking stream; NULL is CUDA's legacy default
    // stream (what torch.cuda.current_stream() is unless the caller changed it)
    ctx->stream = stream == (void *)-1 ? ctx->own_stream : (cudaStream_t)stream;
    return LNB_OK;
}

extern "C" int lnb_synchronize(lnb_ctx *ctx)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    return LNB_OK;
}

extern "C" const char *lnb_last_error(lnb_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }
extern "C" long long lnb_launch_count(lnb_ctx *ctx) { return ctx ? ctx->launches : 0; }

void lnb_prof_begin(lnb_ctx *ctx, const char *name)
{
    if (!ctx->prof_on) return;
    if (ctx->prof_used + 2 > ctx->prof_ev.size()) {
        cudaEvent_t a, b;
        if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
        ctx->prof_ev.push_back(a);
        ctx->prof_ev.push_back(b);
    }
    ctx->prof_name = name;
    cudaEventRecord(ctx->prof_ev[ctx->prof_used], ctx->stream);
}
void lnb_prof_end(lnb_ctx *ctx)
{
    if (!ctx->prof_on || ctx->prof_used + 2 > ctx->prof_ev.size()) return;
    cudaEventRecord(ctx->prof_ev[ctx->prof_used + 1], ctx->stream);
    ctx->prof_used += 2;
}

extern "C" int lnb_profile(lnb_ctx *ctx, int enable)
{
    if (!ctx) return LNB_ERR_ARG;
    ctx->prof_on = enable != 0;
    ctx->prof_used = 0;
    return LNB_OK;
}

extern "C" int lnb_profile_read(lnb_ctx *ctx, double *ms_total, long long *launches, char *name, int name_len)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    double tot = 0.0;
    for (size_t i = 0; i + 1 < ctx->prof_used; i += 2) {
        float ms = 0.f;
        LNB_CUDA(cudaEventElapsedTime(&ms, ctx->prof_ev[i], ctx->prof_ev[i + 1]));
        tot += ms;
    }
    if (ms_total) *ms_total = tot;
    if (launches) *launches = (long long)(ctx->prof_used / 2);
    if (name && name_len > 0) {
        strncpy(name, ctx->prof_name.c_str(), (size_t)name_len - 1);
        name[name_len - 1] = 0;
    }
    return LNB_OK;
}

extern "C" void *lnb_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
extern "C" void lnb_host_free(void *p)
{
    if (p) cudaFreeHost(p);
}

static std::mutex g_default_mu;
static lnb_ctx *g_default_ctx = nullptr;
extern "C" lnb_ctx *lnb_default_ctx(void)
{
    std::lock_guard<std::mutex> lk(g_default_mu);
    if (!g_default_ctx) {
        int dev = 0;
        const char *e = getenv("LOMA_NERF_B200_DEVICE");
        if (e && *e) dev = atoi(e);
        if (lnb_create(&g_default_ctx, dev) != LNB_OK) g_default_ctx = nullptr;
    }
    return g_default_ctx;
}

// ------------------------------------------------------------------------------------------------
// the layerwise fp32 step (device pointers)
// ------------------------------------------------------------------------------------------------
namespace {

struct StepDims {
    int L, c_in, N, M, R, S, Wt;
    int out_last;
};

int validate(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, StepDims *d)
{
    LNB_ARG(mlp && a, "null mlp/args");
    LNB_ARG(mlp->n_layers >= 1 && mlp->n_layers <= LNB_MAX_LAYERS, "n_layers out of range");
    for (int l = 0; l <= mlp->n_layers; ++l) LNB_ARG(mlp->dims[l] >= 1, "dims must be >= 1");
    for (int l = 0; l < mlp->n_layers; ++l)
        LNB_ARG(mlp->dims[l] <= mlp->max_in && mlp->dims[l + 1] <= mlp->max_out,
                "dims exceed the padded weight layout");
    LNB_ARG(a->R >= 0 && a->S >= 1, "R >= 0 and S >= 1 required");
    d->L = mlp->n_layers;
    d->c_in = mlp->dims[0];
    d->R = a->R;
    d->S = nerf ? a->S : 1;
    d->N = a->n_rows > 0 ? a->n_rows : d->R * d->S;
    d->M = a->rows > d->N ? a->rows : d->N;
    d->Wt = a->target_w > 0 ? a->target_w : 3;
    d->out_last = mlp->dims[mlp->n_layers];
    const bool cam = !a->X && !a->rays_o && a->cam;
    const bool rays = !a->X && (a->rays_o || cam);
    LNB_ARG((a->X || d->N == 0 || rays) && a->ws && a->bs, "X (or rays, or a camera), ws, bs are required");
    if (cam) {
        LNB_ARG(a->cam->width >= 2 && a->cam->height >= 1, "camera: width >= 2, height >= 1");
        LNB_ARG(a->cam->fx != 0.0 && a->cam->fy != 0.0, "camera: zero focal length");
        LNB_ARG(a->cam->pixels || (a->cam->first_pixel >= 0 && a->cam->first_pixel + d->R <= (long long)a->cam->width * a->cam->height),
                "camera: pixel range outside the grid");
        LNB_ARG(d->S <= 4096, "camera: at most 4096 samples per ray");
    }
    if (rays) {
        LNB_ARG(nerf, "rays mode is a nerf-path feature");
        LNB_ARG(cam || (a->rays_d && a->t), "rays mode needs rays_o, rays_d and t");
        LNB_ARG(lnb_rays_dir_bands(d->c_in, a->pe_bands) != LNB_DIRS_BAD,
                "rays mode: dims[0] must be 3 + 6*pe_bands, or 6 + 6*pe_bands + 6*E_dir with view directions");
        LNB_ARG(a->ray_dtype == LNB_RAY_F64 || a->ray_dtype == LNB_RAY_F32, "ray_dtype");
        LNB_ARG(!a->d_X, "d_X is not available in rays mode");
    }
    if (nerf) {
        LNB_ARG(d->out_last >= 4, "nerf head needs >= 4 output channels");
        LNB_ARG(a->dists || d->R == 0 || rays, "dists is required");
        LNB_ARG(d->N >= d->R * d->S, "n_rows < R*S");
        LNB_ARG(d->Wt == 3, "nerf target must have 3 columns");
    } else {
        LNB_ARG(d->Wt <= d->out_last, "target wider than the MLP output");
        LNB_ARG(d->N >= d->R, "n_rows < R");
    }
    if (a->inter) {
        LNB_ARG(a->inter_rows >= d->M, "inter_rows < rows");
        for (int l = 0; l < d->L; ++l) LNB_ARG(a->inter_ld >= mlp->dims[l + 1], "inter_ld too small");
    }
    if (a->want_grad) {
        LNB_ARG(a->target || d->R == 0, "target is required for the backward pass");
        LNB_ARG(a->d_ws && a->d_bs, "d_ws and d_bs are required for the backward pass");
    }
    return LNB_OK;
}

int step_layerwise(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, const lnb_comp_args *cx)
{
    StepDims d;
    LNB_TRY(validate(ctx, mlp, a, nerf, &d));
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    const int L = d.L, N = d.N, M = d.M, R = d.R, S = d.S;
    int max_w = 0;
    for (int l = 0; l <= L; ++l) max_w = mlp->dims[l] > max_w ? mlp->dims[l] : max_w;
    int n_chunks = (N + 511) / 512;
    if (n_chunks > 4 * ctx->sm_count) n_chunks = 4 * ctx->sm_count;
    if (n_chunks < 1) n_chunks = 1;

    // ---- arena plan
    const bool cam = !a->X && !a->rays_o && a->cam;
    const bool rays = !a->X && (a->rays_o || cam);
    size_t need = 4096;
    auto add = [&](size_t floats) { need += align_up(floats * sizeof(float), 256) + 256; };
    if (rays) { add((size_t)N * d.c_in); add((size_t)R * S); }
    if (!a->inter)
        for (int l = 0; l < L; ++l) add((size_t)M * mlp->dims[l + 1]);
    add((size_t)R + 1);      // ray_sse
    add((size_t)R * 3 + 4);  // colour when the caller wants none
    add(4);                  // loss
    if (a->want_grad) {
        add((size_t)N * max_w);
        add((size_t)N * max_w);
        add((size_t)n_chunks * (size_t)(mlp->max_in + 1) * mlp->max_out);
        add((size_t)N);         // d_dists unit
        add((size_t)R * d.Wt);  // d_color unit
    }
    LNB_TRY(lnb_arena_reserve(ctx, need));
    auto takef = [&](size_t floats) { return (float *)lnb_arena_take(ctx, floats * sizeof(float)); };

    // ---- rays mode: sample generation + positional encoding on the device (float64 like the reference)
    const float *X = a->X, *dists = a->dists;
    if (rays) {
        float *Xe = takef((size_t)N * d.c_in), *de = takef((size_t)R * S);
        const int Ed = lnb_rays_dir_bands(d.c_in, a->pe_bands);
        if (cam) LNB_TRY(lnb_launch_camera_encode(ctx, a->cam, lnb_cx_views(cx), R, S, a->pe_bands, Ed, Xe, de, nullptr, 0));
        else LNB_TRY(lnb_launch_sample_encode(ctx, a->rays_o, a->rays_d, a->t, a->ray_dtype == LNB_RAY_F64, R, S, a->pe_bands, Ed, Xe, de));
        X = Xe; dists = de;
    }
    // ---- forward
    std::vector<float *> Y(L);
    std::vector<int> ldy(L);
    for (int l = 0; l < L; ++l) {
        if (a->inter) {
            Y[l] = a->inter + (size_t)l * a->inter_rows * a->inter_ld;
            ldy[l] = a->inter_ld;
        } else {
            Y[l] = takef((size_t)M * mlp->dims[l + 1]);
            ldy[l] = mlp->dims[l + 1];
        }
    }
    float *ray_sse = takef((size_t)R + 1);
    float *color = a->color;
    int color_acc = a->color_accumulate;
    if (!color) { color = takef((size_t)R * 3 + 4); color_acc = 0; }
    float *loss = a->loss ? a->loss : takef(4);

    for (int l = 0; l < L; ++l) {
        lnb_gemm_args g{};
        g.A = l == 0 ? X : Y[l - 1];
        g.lda = l == 0 ? d.c_in : ldy[l - 1];
        g.a_rows = l == 0 ? N : M;
        g.B = a->ws + (size_t)l * mlp->max_in * mlp->max_out;
        g.sbk = mlp->max_out;
        g.sbn = 1;
        g.C = Y[l];
        g.ldc = ldy[l];
        g.rows = M;
        g.n_dim = mlp->dims[l + 1];
        g.k_dim = mlp->dims[l];
        g.bias = a->bs + (size_t)l * mlp->max_out;
        g.acc = (a->inter && a->inter_accumulate) ? 1 : 0;
        g.act = l < L - 1 ? ACT_RELU : (mlp->head == LNB_HEAD_NERF ? ACT_NERF_HEAD : ACT_SIGMOID);
        LNB_TRY(lnb_launch_row_gemm(ctx, g));
    }
    const float *head = Y[L - 1];
    const int ldh = ldy[L - 1];
    if (nerf) {
        LNB_TRY(lnb_launch_composite_fwd(ctx, head, ldh, dists, a->target, R, S, a->rgba,
                                         a->alpha, a->cumprod, a->weights, color, color_acc,
                                         ray_sse, cx));
    } else if (a->target) {
        LNB_TRY(lnb_launch_fit_loss(ctx, head, ldh, a->target, R, d.Wt, ray_sse));
    }
    if (a->target) LNB_TRY(lnb_launch_sum(ctx, ray_sse, R, loss));
    else if (a->loss) LNB_TRY(lnb_launch_fill(ctx, loss, 1, 0.0f));
    if (!a->want_grad || R == 0) return LNB_OK;

    // ---- backward (unit seed inside; every output scaled by the seed when accumulated)
    const float *seed_dev = a->seed_mode == LNB_SEED_LOSS ? loss : nullptr;
    const float seed_val = a->seed_mode == LNB_SEED_LOSS ? 1.0f : a->seed;
    float *dZa = takef((size_t)N * max_w), *dZb = takef((size_t)N * max_w);
    float *partial = takef((size_t)n_chunks * (size_t)(mlp->max_in + 1) * mlp->max_out);
    float *d_dists_u = takef((size_t)N), *d_color_u = takef((size_t)R * d.Wt);
    const int n_bwd = nerf ? R * S : R; // rows that carry a non-zero adjoint
    int ldz = d.out_last;
    if (nerf) {
        LNB_TRY(lnb_launch_composite_bwd(ctx, head, ldh, dists, a->target, color, R, S, dZa, ldz,
                                         d.out_last, a->d_dists ? d_dists_u : nullptr, d_color_u, cx));
        if (a->d_dists)
            LNB_TRY(lnb_launch_axpy2d(ctx, a->d_dists, S, d_dists_u, S, R, S, 1.0f, seed_val, seed_dev));
    } else {
        LNB_TRY(lnb_launch_fit_head_bwd(ctx, head, ldh, a->target, R, d.Wt, n_bwd, d.out_last, dZa,
                                        ldz, d_color_u));
    }
    if (a->d_target)
        LNB_TRY(lnb_launch_axpy2d(ctx, a->d_target, d.Wt, d_color_u, d.Wt, R, d.Wt, -1.0f, seed_val, seed_dev));
    if (a->d_color)
        LNB_TRY(lnb_launch_axpy2d(ctx, a->d_color, d.Wt, d_color_u, d.Wt, R, d.Wt, 1.0f, seed_val, seed_dev));
    float *dZ = dZa, *dZn = dZb;
    for (int l = L - 1; l >= 0; --l) {
        const int in_l = mlp->dims[l], out_l = mlp->dims[l + 1];
        const float *H = l == 0 ? X : Y[l - 1];
        const int ldhh = l == 0 ? d.c_in : ldy[l - 1];
        LNB_TRY(lnb_launch_dw_partials(ctx, H, ldhh, dZ, ldz, partial, in_l, out_l, n_bwd, n_chunks));
        LNB_TRY(lnb_launch_dw_reduce(ctx, partial, n_chunks, in_l, out_l,
                                     a->d_ws + (size_t)l * mlp->max_in * mlp->max_out, mlp->max_out,
                                     a->d_bs + (size_t)l * mlp->max_out, seed_val, seed_dev));
        if (a->d_inter)
            LNB_TRY(lnb_launch_axpy2d(ctx, a->d_inter + (size_t)l * a->inter_rows * a->inter_ld,
                                      a->inter_ld, dZ, ldz, n_bwd, out_l, 1.0f, seed_val, seed_dev));
        if (l == 0 && !a->d_X) break;
        lnb_gemm_args g{};
        g.A = dZ; g.lda = ldz; g.a_rows = n_bwd;
        g.B = a->ws + (size_t)l * mlp->max_in * mlp->max_out;
        g.sbk = 1; g.sbn = mlp->max_out;
        g.C = dZn; g.ldc = in_l;
        g.rows = n_bwd; g.n_dim = in_l; g.k_dim = out_l;
        g.act = ACT_NONE;
        if (l > 0) { g.mask = Y[l - 1]; g.ldmask = ldy[l - 1]; }
        LNB_TRY(lnb_launch_row_gemm(ctx, g));
        if (l == 0)
            LNB_TRY(lnb_launch_axpy2d(ctx, a->d_X, d.c_in, dZn, in_l, n_bwd, in_l, 1.0f, seed_val, seed_dev));
        float *t = dZ; dZ = dZn; dZn = t;
        ldz = in_l;
    }
    return LNB_OK;
}

} // namespace


// A views batch as the routes take it: the step with cam pointing at the views' shared camera fields (the per-ray poses
// travel in lnb_comp_args).  LNB_ERR_ARG for a step that has its own input or a bad lnb_views.
struct ViewsStep {
    lnb_step_args a;
    lnb_camera cam;
};
static int views_step(lnb_ctx *ctx, const lnb_step_args *a, const lnb_views *views, ViewsStep *vs)
{
    LNB_ARG(a, "null args");
    LNB_ARG(!a->X && !a->rays_o && !a->cam, "views step: the batch must have no X, rays or cam");
    LNB_TRY(lnb_views_check(ctx, views, a->R, a->S));
    vs->a = *a;
    vs->cam = views_camera(*views);
    vs->a.cam = &vs->cam;
    return LNB_OK;
}

// comp: the compositing extras (lnb_composite), resolved here against the (device-pointer) step; one that asks for nothing
// leaves the step exactly as it is without.  views: a views batch (lnb_views; a has no input of its own).
static int step_dispatch(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, const lnb_tc_extra *ex = nullptr,
                         const lnb_composite *comp = nullptr, const lnb_views *views = nullptr)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(a, "null args");
    ViewsStep vs;
    if (views) {
        LNB_TRY(views_step(ctx, a, views, &vs));
        a = &vs.a;
    }
    lnb_comp_args cxa;
    const lnb_comp_args *cx = nullptr;
    LNB_TRY(lnb_comp_resolve(ctx, a, nerf, comp, views, &cxa, &cx));
    if (a->path == LNB_PATH_F32_LAYERWISE) return step_layerwise(ctx, mlp, a, nerf, cx);
    if (a->path == LNB_PATH_F32) {
        // same arithmetic type and tolerance either way: the fused kernel when the problem and the outputs asked for fit
        // it (loss, colour, d_ws, d_bs of a 2-3 layer network of the reference's widths), else the layerwise kernels
        StepDims d;
        LNB_TRY(validate(ctx, mlp, a, nerf, &d));
        const int rc = getenv("LNB_F32_NO_FUSED") ? LNB_ERR_UNSUPPORTED : lnb_fused_f32_step(ctx, mlp, a, nerf, 0, cx);
        if (rc != LNB_ERR_UNSUPPORTED) return rc;
        return step_layerwise(ctx, mlp, a, nerf, cx);
    }
    if (a->path == LNB_PATH_TC) {
        StepDims d;
        LNB_TRY(validate(ctx, mlp, a, nerf, &d));
        int rc = lnb_fused_tc_step(ctx, mlp, a, nerf, ex, cx); // never silently changes arithmetic
        if (rc == LNB_ERR_UNSUPPORTED && !ex) {
            // wide MLPs: layerwise tensor-core path (same operand precision, same outputs)
            const std::string why = ctx->err;
            rc = lnb_wide_tc_step(ctx, mlp, a, nerf, cx);
            if (rc == LNB_ERR_UNSUPPORTED) ctx->err = why + "; " + ctx->err;
        }
        return rc;
    }
    LNB_ARG(false, "unknown path");
    return LNB_ERR_ARG;
}

// validated entry to the fused exact kernel for the trainer (overwrite: gradients written, not accumulated)
int lnb_step_f32_fused(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, int overwrite, const lnb_views *views)
{
    if (!ctx) return LNB_ERR_ARG;
    ViewsStep vs;
    if (views) {
        LNB_TRY(views_step(ctx, a, views, &vs));
        a = &vs.a;
    }
    lnb_comp_args cxa;
    const lnb_comp_args *cx = nullptr;
    LNB_TRY(lnb_comp_resolve(ctx, a, nerf, nullptr, views, &cxa, &cx));
    StepDims d;
    LNB_TRY(validate(ctx, mlp, a, nerf, &d));
    return lnb_fused_f32_step(ctx, mlp, a, nerf, overwrite, cx);
}

int lnb_step_ex(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, const lnb_tc_extra *ex,
                const lnb_composite *comp, const lnb_views *views)
{
    return step_dispatch(ctx, mlp, a, nerf, ex, comp, views);
}

extern "C" int lnb_nerf_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args)
{
    return step_dispatch(ctx, mlp, args, true);
}
extern "C" int lnb_fit_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args)
{
    return step_dispatch(ctx, mlp, args, false);
}
extern "C" int lnb_nerf_step_composite(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args, const lnb_composite *comp)
{
    return step_dispatch(ctx, mlp, args, true, nullptr, comp);
}
extern "C" int lnb_nerf_step_views(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args, const lnb_views *views,
                                   const lnb_composite *comp)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(views, "nerf_step_views: null views");
    return step_dispatch(ctx, mlp, args, true, nullptr, comp, views);
}

// ------------------------------------------------------------------------------------------------
// host-pointer variants: stage -> device step -> stage back.  Accumulating outputs (d_*) start at
// zero on the device and are added to the caller's host buffers; overwritten outputs are copied.
// ------------------------------------------------------------------------------------------------
namespace {

enum BufKind { BUF_IN, BUF_OUT, BUF_OUT_ACC, BUF_INOUT };
struct Buf {
    const void *host_in;
    void *host_out;
    size_t bytes;
    BufKind kind;
    size_t off; // in the device staging block
    void *pin;  // pinned bounce buffer (NULL when the user pointer is itself pinned)
};

bool is_pinned(const void *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

int step_host(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, const lnb_composite *comp = nullptr)
{
    if (!ctx) return LNB_ERR_ARG;
    StepDims d;
    LNB_TRY(validate(ctx, mlp, a, nerf, &d));
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    const size_t N = d.N, R = d.R, S = d.S, L = d.L;
    const size_t nW = L * (size_t)mlp->max_in * mlp->max_out, nB = L * (size_t)mlp->max_out;
    const size_t nInter = L * (size_t)a->inter_rows * a->inter_ld;
    lnb_step_args dev = *a;
    std::vector<Buf> bufs;
    std::vector<void **> slots;
    auto reg = [&](const void *hin, void *hout, size_t floats, BufKind k, void **slot) {
        bufs.push_back(Buf{hin, hout, floats * sizeof(float), k, 0, nullptr});
        slots.push_back(slot);
    };
#define IN_(field, n) if (a->field) reg(a->field, nullptr, (n), BUF_IN, (void **)&dev.field)
#define OUT_(field, n) if (a->field) reg(nullptr, a->field, (n), BUF_OUT, (void **)&dev.field)
#define ACC_(field, n) if (a->field) reg(nullptr, a->field, (n), BUF_OUT_ACC, (void **)&dev.field)
    IN_(X, N * d.c_in);
    if (!a->X && a->rays_o) {
        const size_t w = a->ray_dtype == LNB_RAY_F64 ? 2 : 1; // floats per element
        reg(a->rays_o, nullptr, R * 3 * w, BUF_IN, (void **)&dev.rays_o);
        reg(a->rays_d, nullptr, R * 3 * w, BUF_IN, (void **)&dev.rays_d);
        reg(a->t, nullptr, R * S * w, BUF_IN, (void **)&dev.t);
    }
    lnb_camera cam_dev;   // camera mode: the struct stays on the host; its pixel list (if any) is staged like an input
    const bool cam_mode = !a->X && !a->rays_o && a->cam;
    if (cam_mode) {
        cam_dev = *a->cam;
        dev.cam = &cam_dev;
        if (a->cam->pixels) reg(a->cam->pixels, nullptr, R, BUF_IN, (void **)&cam_dev.pixels);
    }
    IN_(ws, nW);
    IN_(bs, nB);
    IN_(target, R * d.Wt);
    if (nerf && !(!a->X && (a->rays_o || cam_mode))) IN_(dists, R * S);
    if (a->inter) reg(a->inter, a->inter, nInter, a->inter_accumulate ? BUF_INOUT : BUF_OUT, (void **)&dev.inter);
    if (nerf) {
        OUT_(rgba, R * S * 4);
        OUT_(alpha, R * S);
        OUT_(cumprod, R * S);
        OUT_(weights, R * S);
        if (a->color) reg(a->color, a->color, R * 3, a->color_accumulate ? BUF_INOUT : BUF_OUT, (void **)&dev.color);
    }
    lnb_composite comp_dev;   // the compositing extras: acc / depth are staged like colour
    if (comp) {
        comp_dev = *comp;
        if (nerf && comp->acc) reg(nullptr, comp->acc, R, BUF_OUT, (void **)&comp_dev.acc);
        if (nerf && comp->depth) reg(nullptr, comp->depth, R, BUF_OUT, (void **)&comp_dev.depth);
    }
    OUT_(loss, 1);
    if (a->want_grad) {
        ACC_(d_ws, nW);
        ACC_(d_bs, nB);
        ACC_(d_X, N * d.c_in);
        ACC_(d_target, R * d.Wt);
        if (nerf) ACC_(d_dists, R * S);
        ACC_(d_color, R * d.Wt);
        if (a->d_inter) reg(nullptr, a->d_inter, nInter, BUF_OUT_ACC, (void **)&dev.d_inter);
    } else {
        dev.d_ws = dev.d_bs = dev.d_X = dev.d_target = dev.d_dists = dev.d_color = dev.d_inter = nullptr;
    }
#undef IN_
#undef OUT_
#undef ACC_
    size_t dtotal = 0, ptotal = 0;
    for (auto &b : bufs) {
        b.off = dtotal;
        dtotal += align_up(b.bytes, 256);
        const void *h = b.kind == BUF_IN ? b.host_in : b.host_out;
        // outputs that accumulate must bounce (host-side +=); others go direct when pinned
        bool direct = b.kind != BUF_OUT_ACC && is_pinned(h);
        if (!direct) ptotal += align_up(b.bytes, 256) + 256;
        b.pin = direct ? nullptr : (void *)1;
    }
    LNB_TRY(dstage_reserve(ctx, dtotal + 256));
    LNB_TRY(lnb_pinned_reserve(ctx, ptotal + 256));
    for (size_t i = 0; i < bufs.size(); ++i) {
        Buf &b = bufs[i];
        if (b.pin) b.pin = lnb_pinned_take(ctx, b.bytes);
        *slots[i] = ctx->dstage + b.off;
    }
    // H2D
    for (auto &b : bufs) {
        char *dptr = ctx->dstage + b.off;
        if (b.kind == BUF_IN || b.kind == BUF_INOUT) {
            const void *src = b.host_in;
            if (b.pin) { memcpy(b.pin, b.host_in, b.bytes); src = b.pin; }
            LNB_CUDA(cudaMemcpyAsync(dptr, src, b.bytes, cudaMemcpyHostToDevice, ctx->stream));
        } else {
            // accumulating outputs start from zero; overwritten outputs too, so that the parts a
            // kernel never writes (padding columns of inter) come back as zeros, not stale bytes
            LNB_CUDA(cudaMemsetAsync(dptr, 0, b.bytes, ctx->stream));
        }
    }
    int rc = step_dispatch(ctx, mlp, &dev, nerf, nullptr, comp ? &comp_dev : nullptr);
    if (rc != LNB_OK) return rc;
    // D2H
    for (auto &b : bufs) {
        if (b.kind == BUF_IN) continue;
        void *dst = b.pin ? b.pin : b.host_out;
        LNB_CUDA(cudaMemcpyAsync(dst, ctx->dstage + b.off, b.bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    for (auto &b : bufs) {
        if (b.kind == BUF_IN || !b.pin) continue;
        if (b.kind == BUF_OUT_ACC) {
            float *o = (float *)b.host_out;
            const float *s = (const float *)b.pin;
            for (size_t i = 0, n = b.bytes / sizeof(float); i < n; ++i) o[i] += s[i];
        } else {
            memcpy(b.host_out, b.pin, b.bytes);
        }
    }
    return LNB_OK;
}

} // namespace

extern "C" int lnb_nerf_step_host(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args)
{
    return step_host(ctx, mlp, args, true);
}
extern "C" int lnb_fit_step_host(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args)
{
    return step_host(ctx, mlp, args, false);
}
extern "C" int lnb_nerf_step_composite_host(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *args, const lnb_composite *comp)
{
    return step_host(ctx, mlp, args, true, comp);
}

// ------------------------------------------------------------------------------------------------
// small flat entry points
// ------------------------------------------------------------------------------------------------
extern "C" int lnb_pos_encoding(lnb_ctx *ctx, const double *x, long long n, int F, int E, float *out)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(x && out && n >= 0 && F >= 1 && E >= 0, "pos_encoding arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    return lnb_launch_pos_encoding(ctx, x, n, F, E, out);
}

extern "C" int lnb_sample_encode(lnb_ctx *ctx, const double *rays_o, const double *rays_d,
                                 const double *t, int R, int S, int E, float *X, float *dists)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(rays_o && rays_d && t && X && R >= 0 && S >= 1 && E >= 0, "sample_encode arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    return lnb_launch_sample_encode(ctx, rays_o, rays_d, t, 1, R, S, E, LNB_DIRS_NONE, X, dists);
}

extern "C" int lnb_sample_encode_dirs(lnb_ctx *ctx, const double *rays_o, const double *rays_d,
                                      const double *t, int R, int S, int E, int E_dir, float *X, float *dists)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(rays_o && rays_d && t && X && R >= 0 && S >= 1 && E >= 0 && E_dir >= 0, "sample_encode_dirs arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    return lnb_launch_sample_encode(ctx, rays_o, rays_d, t, 1, R, S, E, E_dir, X, dists);
}

extern "C" int lnb_mult_a_b(lnb_ctx *ctx, const float *a, int a_h, int a_w, const float *b, int b_w,
                            float *c)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(a && b && c && a_h >= 0 && a_w >= 0 && b_w >= 0, "mult_a_b arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    lnb_gemm_args g{};
    g.A = a; g.lda = a_w; g.a_rows = a_h;
    g.B = b; g.sbk = b_w; g.sbn = 1;
    g.C = c; g.ldc = b_w;
    g.rows = a_h; g.n_dim = b_w; g.k_dim = a_w;
    g.acc = 1; g.act = ACT_NONE;
    return lnb_launch_row_gemm(ctx, g);
}

extern "C" int lnb_adam_step(lnb_ctx *ctx, float *param, const float *grad, float *m, float *v,
                             long long n, int t, double lr, double beta1, double beta2, double eps)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(param && grad && m && v && n >= 0 && t >= 1, "adam arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    return lnb_launch_adam(ctx, param, grad, m, v, n, t, lr, beta1, beta2, eps);
}

extern "C" int lnb_adam_step_dev(lnb_ctx *ctx, float *param, const float *grad, float *m, float *v,
                                 long long n, int *t_dev, double lr, double beta1, double beta2, double eps)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(param && grad && m && v && t_dev && n >= 0, "adam arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    return lnb_launch_adam_dev(ctx, param, grad, m, v, n, t_dev, lr, beta1, beta2, eps);
}

extern "C" int lnb_sgd_step(lnb_ctx *ctx, float *param, const float *grad, long long n, double lr)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(param && grad && n >= 0, "sgd arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    return lnb_launch_sgd(ctx, param, grad, n, lr);
}
