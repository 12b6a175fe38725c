// trainer.cu -- device-resident training state for the hot path (SURVEY.md 8f rank 1).
//
// The reference keeps the padded weights in numpy and, per chunk, calls the grad function and
// then applies AdamOptimizer.update (train_nerf.py:395-499) or SGD (fit_img.py:512-513) on the
// host.  A trainer keeps weights, optimiser state, the gradient buffer and (tensor-core path) the
// bf16 weight image on the GPU, so one train step is two kernel launches and no host traffic:
//     fused forward+backward kernel  ->  reduce partials + optimiser update + weight-image refresh
// For multi-GPU data parallelism the step splits at the gradient buffer:
//     lnb_trainer_grad -> (caller: NCCL all-reduce of lnb_trainer_grad_buffer) -> lnb_trainer_apply
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "lnb_internal.h"

struct lnb_trainer {
    lnb_ctx *ctx = nullptr;
    lnb_mlp mlp{};
    int opt = LNB_OPT_ADAM;
    double lr = 5e-4, b1 = 0.9, b2 = 0.999, eps = 1e-8;
    long long n_w = 0, n_b = 0;
    float *params = nullptr; // [ws | bs]
    float *grads = nullptr;  // [d_ws | d_bs | loss]
    float *m = nullptr, *v = nullptr;
    int *t_dev = nullptr;
    void *wimg = nullptr;    // tensor-core weight image, kept in sync with params
    bool tc_ok = false;
    bool t_bumped = false;   // the last lnb_trainer_grad already incremented *t_dev
    lnb_composite comp{};    // lnb_trainer_set_background: background 0 = the reference's compositing
    lnb_views views{};       // lnb_trainer_set_views: a nerf batch with no input of its own is a views batch
    bool has_views = false;
    // peer-memory all-reduce (lnb_trainer_comm_*): header [status | pad] + receive slots for 8 senders
    char *comm_buf = nullptr;
    size_t comm_bytes = 0;
    lnb_tc_comm comm{};
    void *peer_base[8] = {};
    // pipelined host-buffer steps (lnb_trainer_submit_host / lnb_trainer_wait)
    struct Pipe {
        static constexpr int RING = 4096;
        cudaStream_t copy_stream = nullptr;
        cudaEvent_t staged[2] = {}, consumed[2] = {};
        char *dslot[2] = {}, *pslot[2] = {};
        size_t dcap = 0, pcap = 0;
        float *loss_ring = nullptr;
        int pending = 0;
        long long seq = 0;
    } pipe;
};

static int comm_slots(const lnb_trainer *t)
{
    int n = 1;
    for (int l = 0; l < t->mlp.n_layers; ++l) n += (t->mlp.dims[l] + 1) * t->mlp.dims[l + 1];
    return n; // live gradient elements + the loss
}

extern "C" int lnb_trainer_create(lnb_ctx *ctx, const lnb_mlp *mlp, const float *ws_host, const float *bs_host,
                                  int optimizer, double lr, double beta1, double beta2, double eps, lnb_trainer **out)
{
    if (!ctx || !out) return LNB_ERR_ARG;
    *out = nullptr;
    LNB_ARG(mlp && ws_host && bs_host, "trainer: mlp, ws, bs required");
    LNB_ARG(mlp->n_layers >= 1 && mlp->n_layers <= LNB_MAX_LAYERS, "trainer: n_layers");
    LNB_ARG(optimizer == LNB_OPT_ADAM || optimizer == LNB_OPT_SGD, "trainer: optimizer");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    lnb_trainer *t = new lnb_trainer();
    t->ctx = ctx; t->mlp = *mlp; t->opt = optimizer;
    t->lr = lr; t->b1 = beta1; t->b2 = beta2; t->eps = eps;
    t->n_w = (long long)mlp->n_layers * mlp->max_in * mlp->max_out;
    t->n_b = (long long)mlp->n_layers * mlp->max_out;
    const size_t np = (size_t)(t->n_w + t->n_b);
    int wimg_bytes = 0;
    t->tc_ok = lnb_tc_layout(mlp, nullptr, nullptr, &wimg_bytes) != 0;
    bool ok = cudaMalloc((void **)&t->params, np * 4) == cudaSuccess && cudaMalloc((void **)&t->grads, (np + 1) * 4) == cudaSuccess &&
              cudaMalloc((void **)&t->m, np * 4) == cudaSuccess && cudaMalloc((void **)&t->v, np * 4) == cudaSuccess &&
              cudaMalloc((void **)&t->t_dev, 16) == cudaSuccess;
    if (ok && t->tc_ok) ok = cudaMalloc(&t->wimg, (size_t)wimg_bytes) == cudaSuccess;
    ok = ok && cudaMemcpyAsync(t->params, ws_host, (size_t)t->n_w * 4, cudaMemcpyHostToDevice, ctx->stream) == cudaSuccess &&
         cudaMemcpyAsync(t->params + t->n_w, bs_host, (size_t)t->n_b * 4, cudaMemcpyHostToDevice, ctx->stream) == cudaSuccess &&
         cudaMemsetAsync(t->grads, 0, (np + 1) * 4, ctx->stream) == cudaSuccess && cudaMemsetAsync(t->m, 0, np * 4, ctx->stream) == cudaSuccess &&
         cudaMemsetAsync(t->v, 0, np * 4, ctx->stream) == cudaSuccess && cudaMemsetAsync(t->t_dev, 0, 16, ctx->stream) == cudaSuccess;
    if (ok && t->tc_ok) ok = lnb_tc_prep(ctx, mlp, t->params, t->params + t->n_w, t->wimg) == LNB_OK;
    ok = ok && cudaStreamSynchronize(ctx->stream) == cudaSuccess; // the host buffers may go away
    if (!ok) {
        ctx->err = std::string("trainer: allocation or upload failed: ") + cudaGetErrorString(cudaGetLastError());
        lnb_trainer_destroy(t);
        return LNB_ERR_CUDA;
    }
    *out = t;
    return LNB_OK;
}

extern "C" void lnb_trainer_destroy(lnb_trainer *t)
{
    if (!t) return;
    cudaSetDevice(t->ctx->device);
    cudaStreamSynchronize(t->ctx->stream);
    for (int r = 0; r < 8; ++r)
        if (t->peer_base[r]) cudaIpcCloseMemHandle(t->peer_base[r]);
    if (t->comm_buf) cudaFree(t->comm_buf);
    if (t->pipe.copy_stream) {
        cudaStreamSynchronize(t->pipe.copy_stream);
        cudaStreamDestroy(t->pipe.copy_stream);
        for (int s = 0; s < 2; ++s) {
            cudaEventDestroy(t->pipe.staged[s]); cudaEventDestroy(t->pipe.consumed[s]);
            if (t->pipe.dslot[s]) cudaFree(t->pipe.dslot[s]);
            if (t->pipe.pslot[s]) cudaFreeHost(t->pipe.pslot[s]);
        }
        cudaFreeHost(t->pipe.loss_ring);
    }
    cudaFree(t->params); cudaFree(t->grads); cudaFree(t->m); cudaFree(t->v); cudaFree(t->t_dev);
    if (t->wimg) cudaFree(t->wimg);
    delete t;
}

// a peer never delivered its gradients: the step that noticed has poisoned the parameters with NaN
static int comm_failed(lnb_trainer *t, float *loss_out)
{
    t->ctx->err = "trainer: a peer rank did not deliver its gradients in time; the step was poisoned (NaN) instead of "
                  "applying a partial sum -- the replicas of this run are no longer usable";
    if (loss_out) *loss_out = __builtin_nanf("");
    return LNB_ERR_CUDA;
}

// weights: [R][S] compositing weights of this step's forward pass (lnb_trainer_step_weights), or NULL
static int trainer_run(lnb_trainer *t, const lnb_step_args *batch, int nerf, bool fuse_update, float *weights = nullptr)
{
    lnb_ctx *ctx = t->ctx;
    LNB_ARG(batch, "trainer: null batch");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    lnb_step_args a = *batch;
    a.ws = t->params; a.bs = t->params + t->n_w;
    a.want_grad = 1;
    a.d_ws = t->grads; a.d_bs = t->grads + t->n_w; a.loss = t->grads + t->n_w + t->n_b;
    a.d_X = a.d_target = a.d_dists = a.d_color = a.d_inter = nullptr;
    a.inter = a.rgba = a.alpha = a.cumprod = a.weights = nullptr;
    const lnb_composite *comp = (nerf && t->comp.background) ? &t->comp : nullptr;   // every route below composites onto it
    const lnb_views *views = (nerf && t->has_views && !a.X && !a.rays_o && !a.cam) ? &t->views : nullptr;
    if (a.path == LNB_PATH_TC && t->tc_ok) {
        lnb_tc_extra ex;
        ex.wimg = t->wimg; ex.overwrite_grads = 1; ex.t_dev = t->t_dev; ex.weights = weights;
        if (fuse_update) {
            if (t->comm.world > 1) ex.comm = &t->comm;
            ex.fuse_adam = 1; ex.param = t->params; ex.m = t->opt == LNB_OPT_ADAM ? t->m : nullptr; ex.v = t->v;
            ex.lr = t->lr; ex.b1 = t->b1; ex.b2 = t->b2; ex.eps = t->eps; ex.wimg_out = t->wimg;
        }
        const int rc = lnb_step_ex(ctx, &t->mlp, &a, nerf != 0, &ex, comp, views);
        if (rc == LNB_OK) { t->t_bumped = !fuse_update; return LNB_OK; }
        // the MLP fits the fused kernel but this batch does not (e.g. S > 128): the layerwise
        // tensor-core kernels below take it, exactly as lnb_nerf_step would
        if (rc != LNB_ERR_UNSUPPORTED) return rc;
    }
    // exact fp32 path, or the layerwise tensor-core path: zero the gradient buffer (those kernels
    // accumulate), step, optional update.  These steps have no fused exchange: with a peer group
    // attached they would update from local gradients only and the replicas would drift apart.
    if (fuse_update && t->comm.world > 1) {
        ctx->err = "trainer: the peer all-reduce is attached but this step (fp32 path, wide MLP or S > 128) cannot "
                   "exchange gradients in-kernel; use lnb_trainer_grad + an all-reduce of lnb_trainer_grad_buffer + lnb_trainer_apply";
        return LNB_ERR_UNSUPPORTED;
    }
    // the fused exact kernel writes no weights and has no background: a step that asks for either runs on the layerwise
    // kernels
    a.weights = weights;
    int rc = LNB_ERR_UNSUPPORTED;
    if (a.path == LNB_PATH_F32 && !comp && !getenv("LNB_F32_NO_FUSED")) {
        // fused exact kernel writing the (zero-padded, never otherwise touched) gradient buffer: no memset
        rc = lnb_step_f32_fused(ctx, &t->mlp, &a, nerf != 0, 1, views);
        if (rc != LNB_OK && rc != LNB_ERR_UNSUPPORTED) return rc;
    }
    if (rc == LNB_ERR_UNSUPPORTED) {
        LNB_CUDA(cudaMemsetAsync(t->grads, 0, (size_t)(t->n_w + t->n_b + 1) * 4, ctx->stream));
        LNB_TRY(nerf ? lnb_step_ex(ctx, &t->mlp, &a, true, nullptr, comp, views) : lnb_fit_step(ctx, &t->mlp, &a));
    }
    t->t_bumped = false;
    if (fuse_update) return lnb_trainer_apply(t);
    return LNB_OK;
}

extern "C" int lnb_trainer_grad(lnb_trainer *t, const lnb_step_args *batch, int nerf)
{
    if (!t) return LNB_ERR_ARG;
    return trainer_run(t, batch, nerf, false);
}

extern "C" int lnb_trainer_set_background(lnb_trainer *t, const float *rgb)
{
    if (!t) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    if (!rgb) { t->comp = lnb_composite{}; return LNB_OK; }
    for (int c = 0; c < 3; ++c) LNB_ARG(isfinite(rgb[c]), "trainer_set_background: non-finite colour");
    t->comp = lnb_composite{};
    t->comp.background = 1;
    for (int c = 0; c < 3; ++c) t->comp.bg[c] = rgb[c];
    return LNB_OK;
}

extern "C" int lnb_trainer_set_views(lnb_trainer *t, const lnb_views *views)
{
    if (!t) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    if (!views) { t->views = lnb_views{}; t->has_views = false; return LNB_OK; }
    LNB_TRY(lnb_views_check(ctx, views, 0, 1));
    t->views = *views;
    t->has_views = true;
    return LNB_OK;
}

extern "C" int lnb_trainer_step(lnb_trainer *t, const lnb_step_args *batch, int nerf)
{
    if (!t) return LNB_ERR_ARG;
    return trainer_run(t, batch, nerf, true);
}

extern "C" int lnb_trainer_step_weights(lnb_trainer *t, const lnb_step_args *batch, int nerf, float *weights)
{
    if (!t) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    LNB_ARG(nerf && weights, "trainer_step_weights: a nerf batch and a weights buffer");
    return trainer_run(t, batch, nerf, true, weights);
}

extern "C" int lnb_trainer_apply(lnb_trainer *t)
{
    if (!t) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    const long long np = t->n_w + t->n_b;
    if (t->tc_ok) {
        // keeps the bf16 weight image in step with the fp32 parameters
        if (!t->t_bumped && t->opt == LNB_OPT_ADAM) LNB_TRY(lnb_launch_incr(ctx, t->t_dev));
        t->t_bumped = false;
        return lnb_tc_adam_img(ctx, &t->mlp, t->params, t->grads, t->opt == LNB_OPT_ADAM ? t->m : nullptr, t->v, t->t_dev,
                               t->lr, t->b1, t->b2, t->eps, t->wimg);
    }
    if (t->opt == LNB_OPT_SGD) return lnb_launch_sgd(ctx, t->params, t->grads, np, t->lr);
    if (t->t_bumped) { // counter already advanced: use the host-free variant that reads it as is
        t->t_bumped = false;
        return lnb_launch_adam_at(ctx, t->params, t->grads, t->m, t->v, np, t->t_dev, t->lr, t->b1, t->b2, t->eps);
    }
    return lnb_launch_adam_dev(ctx, t->params, t->grads, t->m, t->v, np, t->t_dev, t->lr, t->b1, t->b2, t->eps);
}

// ---- host-buffer steps ---------------------------------------------------------------------------
// The batch's inputs as (pointer slot, bytes) pairs; `a` is the caller's batch copied, `cam_dev` the
// copy of its camera (camera mode: only the optional pixel list and the targets cross the bus).
struct HostIn { const void **slot; size_t bytes; };
static int host_inputs(lnb_trainer *t, lnb_step_args &a, lnb_camera &cam_dev, int nerf, HostIn *ins, int *n_in_out)
{
    lnb_ctx *ctx = t->ctx;
    const size_t R = (size_t)a.R, S = nerf ? (size_t)a.S : 1, N = a.n_rows > 0 ? (size_t)a.n_rows : R * S;
    const size_t c_in = (size_t)t->mlp.dims[0], Wt = a.target_w > 0 ? (size_t)a.target_w : 3;
    const bool rays = !a.X && a.rays_o;
    const bool cam = !a.X && !a.rays_o && a.cam;
    const size_t rw = a.ray_dtype == LNB_RAY_F64 ? 8 : 4;
    int n_in = 0;
    if (cam) {
        cam_dev = *a.cam;
        a.cam = &cam_dev;
        if (cam_dev.pixels) ins[n_in++] = HostIn{(const void **)&cam_dev.pixels, R * sizeof(int)};
    } else if (rays) {
        ins[n_in++] = HostIn{&a.rays_o, R * 3 * rw};
        ins[n_in++] = HostIn{&a.rays_d, R * 3 * rw};
        ins[n_in++] = HostIn{&a.t, R * S * rw};
    } else {
        LNB_ARG(a.X || !nerf || !t->has_views, "trainer: a views batch (lnb_trainer_set_views) has its scene on the device; "
                                                "the host-buffer steps do not take it");
        LNB_ARG(a.X, "trainer: X or rays required");
        ins[n_in++] = HostIn{(const void **)&a.X, N * c_in * 4};
        if (nerf) { LNB_ARG(a.dists, "trainer: dists required"); ins[n_in++] = HostIn{(const void **)&a.dists, R * S * 4}; }
    }
    LNB_ARG(a.target, "trainer: target required");
    ins[n_in++] = HostIn{(const void **)&a.target, R * Wt * 4};
    *n_in_out = n_in;
    return LNB_OK;
}

static bool host_pinned(const void *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost) return true;
    cudaGetLastError();
    return false;
}

// Host-buffer step: stages the batch (pinned buffers are copied directly, pageable ones bounce
// through the context's pinned block), runs lnb_trainer_step, returns the loss.  Synchronous.
extern "C" int lnb_trainer_step_host(lnb_trainer *t, const lnb_step_args *batch, int nerf, float *loss_out)
{
    if (!t) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    LNB_ARG(batch, "trainer: null batch");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    lnb_step_args a = *batch;
    lnb_camera cam_dev;
    HostIn ins[6];
    int n_in = 0;
    LNB_TRY(host_inputs(t, a, cam_dev, nerf, ins, &n_in));
    size_t dtotal = 0, ptotal = 0;
    bool direct[6];
    for (int i = 0; i < n_in; ++i) {
        direct[i] = host_pinned(*ins[i].slot);
        if (!direct[i]) ptotal += (ins[i].bytes + 255) / 256 * 256 + 256;
        dtotal += (ins[i].bytes + 255) / 256 * 256;
    }
    if (dtotal + 256 > ctx->dstage_cap) {
        LNB_CUDA(cudaStreamSynchronize(ctx->stream));
        if (ctx->dstage) LNB_CUDA(cudaFree(ctx->dstage));
        ctx->dstage = nullptr; ctx->dstage_cap = 0;
        const size_t cap = (dtotal + dtotal / 4 + (1 << 20)) / (1 << 20) * (1 << 20);
        LNB_CUDA(cudaMalloc((void **)&ctx->dstage, cap));
        ctx->dstage_cap = cap;
    }
    LNB_TRY(lnb_pinned_reserve(ctx, ptotal + 256));
    size_t off = 0;
    for (int i = 0; i < n_in; ++i) {
        const void *src = *ins[i].slot;
        if (!direct[i]) {
            void *pin = lnb_pinned_take(ctx, ins[i].bytes);
            memcpy(pin, src, ins[i].bytes);
            src = pin;
        }
        LNB_CUDA(cudaMemcpyAsync(ctx->dstage + off, src, ins[i].bytes, cudaMemcpyHostToDevice, ctx->stream));
        *ins[i].slot = ctx->dstage + off;
        off += (ins[i].bytes + 255) / 256 * 256;
    }
    LNB_TRY(trainer_run(t, &a, nerf, true));
    float *pl = (float *)lnb_pinned_take(ctx, 16);
    if (!pl) { LNB_TRY(lnb_pinned_reserve(ctx, 4096)); pl = (float *)lnb_pinned_take(ctx, 16); }
    LNB_CUDA(cudaMemcpyAsync(pl, t->grads + t->n_w + t->n_b, 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (t->comm.world > 1) LNB_CUDA(cudaMemcpyAsync(pl + 1, t->comm.status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (loss_out) *loss_out = *pl;
    if (t->comm.world > 1 && *reinterpret_cast<const int *>(pl + 1) != 0) return comm_failed(t, loss_out);
    return LNB_OK;
}

// Pipelined host-buffer steps.  Two device staging slots and a copy stream: the host->device copy of
// batch i+1 runs under the step of batch i, and nothing waits for the GPU until lnb_trainer_wait.
//   copy stream : wait(consumed[slot]) -> H2D of the batch -> record(staged[slot])
//   step stream : wait(staged[slot])   -> the step -> D2H of its loss into a pinned ring -> record(consumed[slot])
// Pageable host buffers are copied into a pinned bounce slot at once (the call then waits for the H2D
// that last read that slot, two submissions ago); pinned buffers are read by the DMA engine directly
// and must stay unchanged until the submission after next has returned (or lnb_trainer_wait).
extern "C" int lnb_trainer_submit_host(lnb_trainer *t, const lnb_step_args *batch, int nerf)
{
    if (!t) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    LNB_ARG(batch, "trainer: null batch");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    lnb_trainer::Pipe &pp = t->pipe;
    if (!pp.copy_stream) {
        LNB_CUDA(cudaStreamCreateWithFlags(&pp.copy_stream, cudaStreamNonBlocking));
        for (int s = 0; s < 2; ++s) {
            LNB_CUDA(cudaEventCreateWithFlags(&pp.staged[s], cudaEventDisableTiming));
            LNB_CUDA(cudaEventCreateWithFlags(&pp.consumed[s], cudaEventDisableTiming));
        }
        LNB_CUDA(cudaMallocHost((void **)&pp.loss_ring, lnb_trainer::Pipe::RING * sizeof(float)));
    }
    if (pp.pending == lnb_trainer::Pipe::RING) {   // the ring of undelivered losses is full: drain the GPU, keep the newest
        LNB_CUDA(cudaStreamSynchronize(ctx->stream));
        pp.pending = 0;
    }
    lnb_step_args a = *batch;
    lnb_camera cam_dev;
    HostIn ins[6];
    int n_in = 0;
    LNB_TRY(host_inputs(t, a, cam_dev, nerf, ins, &n_in));
    const int slot = (int)(pp.seq & 1);
    size_t dtotal = 0, ptotal = 0;
    bool direct[6];
    for (int i = 0; i < n_in; ++i) {
        direct[i] = host_pinned(*ins[i].slot);
        if (!direct[i]) ptotal += (ins[i].bytes + 255) / 256 * 256;
        dtotal += (ins[i].bytes + 255) / 256 * 256;
    }
    if (dtotal > pp.dcap || ptotal > pp.pcap) {    // grow (rare): drain both streams first
        LNB_CUDA(cudaStreamSynchronize(pp.copy_stream));
        LNB_CUDA(cudaStreamSynchronize(ctx->stream));
        if (dtotal > pp.dcap) {
            const size_t cap = (dtotal + dtotal / 4 + (1 << 20)) / (1 << 20) * (1 << 20);
            for (int s = 0; s < 2; ++s) {
                if (pp.dslot[s]) LNB_CUDA(cudaFree(pp.dslot[s]));
                pp.dslot[s] = nullptr;
                LNB_CUDA(cudaMalloc((void **)&pp.dslot[s], cap));
            }
            pp.dcap = cap;
        }
        if (ptotal > pp.pcap) {
            const size_t cap = (ptotal + ptotal / 4 + (1 << 20)) / (1 << 20) * (1 << 20);
            for (int s = 0; s < 2; ++s) {
                if (pp.pslot[s]) LNB_CUDA(cudaFreeHost(pp.pslot[s]));
                pp.pslot[s] = nullptr;
                LNB_CUDA(cudaMallocHost((void **)&pp.pslot[s], cap));
            }
            pp.pcap = cap;
        }
    }
    if (ptotal && pp.seq >= 2) LNB_CUDA(cudaEventSynchronize(pp.staged[slot]));   // the DMA that last read this bounce slot
    if (pp.seq >= 2) LNB_CUDA(cudaStreamWaitEvent(pp.copy_stream, pp.consumed[slot], 0));
    size_t off = 0, poff = 0;
    for (int i = 0; i < n_in; ++i) {
        const void *src = *ins[i].slot;
        if (!direct[i]) {
            memcpy(pp.pslot[slot] + poff, src, ins[i].bytes);
            src = pp.pslot[slot] + poff;
            poff += (ins[i].bytes + 255) / 256 * 256;
        }
        LNB_CUDA(cudaMemcpyAsync(pp.dslot[slot] + off, src, ins[i].bytes, cudaMemcpyHostToDevice, pp.copy_stream));
        *ins[i].slot = pp.dslot[slot] + off;
        off += (ins[i].bytes + 255) / 256 * 256;
    }
    LNB_CUDA(cudaEventRecord(pp.staged[slot], pp.copy_stream));
    LNB_CUDA(cudaStreamWaitEvent(ctx->stream, pp.staged[slot], 0));
    LNB_TRY(trainer_run(t, &a, nerf, true));
    LNB_CUDA(cudaMemcpyAsync(pp.loss_ring + pp.pending, t->grads + t->n_w + t->n_b, 4, cudaMemcpyDeviceToHost, ctx->stream));
    LNB_CUDA(cudaEventRecord(pp.consumed[slot], ctx->stream));
    pp.pending++;
    pp.seq++;
    return LNB_OK;
}

// Waits for every submitted step; copies the losses of the steps submitted since the previous wait
// (oldest first, at most max_losses of the newest RING) and returns their number through *n_out.
extern "C" int lnb_trainer_wait(lnb_trainer *t, float *losses, int max_losses, int *n_out)
{
    if (!t) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    lnb_trainer::Pipe &pp = t->pipe;
    int st = 0;
    if (t->comm.world > 1) LNB_CUDA(cudaMemcpyAsync(&st, t->comm.status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    int n = pp.pending;
    if (n > max_losses) n = max_losses < 0 ? 0 : max_losses;
    if (losses) for (int i = 0; i < n; ++i) losses[i] = pp.loss_ring[pp.pending - n + i];
    if (n_out) *n_out = n;
    pp.pending = 0;
    if (st != 0) return comm_failed(t, nullptr);
    return LNB_OK;
}

// ---- peer-memory all-reduce set-up: export my comm buffer, attach everybody's -------------------
extern "C" int lnb_trainer_comm_export(lnb_trainer *t, void *handle64)
{
    if (!t || !handle64) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    LNB_ARG(t->tc_ok, "peer all-reduce is part of the tensor-core trainer step");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    if (!t->comm_buf) {
        t->comm_bytes = 256 + 2 * 8 * (size_t)comm_slots(t) * sizeof(unsigned long long);
        LNB_CUDA(cudaMalloc((void **)&t->comm_buf, t->comm_bytes));
        LNB_CUDA(cudaMemset(t->comm_buf, 0, t->comm_bytes));
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t h;
    LNB_CUDA(cudaIpcGetMemHandle(&h, t->comm_buf));
    memcpy(handle64, &h, 64);
    return LNB_OK;
}

extern "C" int lnb_trainer_comm_attach(lnb_trainer *t, int rank, int world, const void *handles)
{
    if (!t || !handles) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    LNB_ARG(world >= 1 && world <= 8 && rank >= 0 && rank < world, "comm: 1 <= world <= 8");
    LNB_ARG(t->comm_buf, "comm: call lnb_trainer_comm_export first");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    const int n_slot = comm_slots(t);
    lnb_tc_comm c{};
    c.world = world; c.rank = rank; c.n_slot = n_slot;
    if (const char *e = getenv("LNB_PEER_TIMEOUT_MS")) { const long long ms = atoll(e); if (ms > 0) c.timeout_ns = (unsigned long long)ms * 1000000ull; }
    c.status = reinterpret_cast<int *>(t->comm_buf);
    c.my_recv = reinterpret_cast<unsigned long long *>(t->comm_buf + 256);
    for (int r = 0; r < world; ++r) {
        char *base = t->comm_buf;
        if (r != rank) {
            cudaIpcMemHandle_t h;
            memcpy(&h, (const char *)handles + (size_t)r * 64, 64);
            void *p = nullptr;
            LNB_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
            t->peer_base[r] = p;
            base = (char *)p;
        }
        c.peer_recv[r] = reinterpret_cast<unsigned long long *>(base + 256);
    }
    t->comm = c;
    return LNB_OK;
}

// 0 = fine; 1 = a peer's words never arrived and that step was poisoned with NaN. Synchronises.
extern "C" int lnb_trainer_comm_status(lnb_trainer *t)
{
    if (!t || !t->comm_buf) return 0;
    int st = 0;
    cudaSetDevice(t->ctx->device);
    cudaStreamSynchronize(t->ctx->stream);
    cudaMemcpy(&st, t->comm_buf, 4, cudaMemcpyDeviceToHost);
    return st;
}

extern "C" float *lnb_trainer_grad_buffer(lnb_trainer *t, long long *n_floats)
{
    if (!t) return nullptr;
    if (n_floats) *n_floats = t->n_w + t->n_b + 1;
    return t->grads;
}

extern "C" float *lnb_trainer_params(lnb_trainer *t, long long *n_w, long long *n_b)
{
    if (!t) return nullptr;
    if (n_w) *n_w = t->n_w;
    if (n_b) *n_b = t->n_b;
    return t->params;
}

extern "C" int lnb_trainer_read(lnb_trainer *t, float *ws_host, float *bs_host, float *loss_host)
{
    if (!t) return LNB_ERR_ARG;
    lnb_ctx *ctx = t->ctx;
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    if (ws_host) LNB_CUDA(cudaMemcpyAsync(ws_host, t->params, (size_t)t->n_w * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (bs_host) LNB_CUDA(cudaMemcpyAsync(bs_host, t->params + t->n_w, (size_t)t->n_b * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (loss_host) LNB_CUDA(cudaMemcpyAsync(loss_host, t->grads + t->n_w + t->n_b, 4, cudaMemcpyDeviceToHost, ctx->stream));
    int st = 0;
    if (t->comm.world > 1) LNB_CUDA(cudaMemcpyAsync(&st, t->comm.status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    LNB_CUDA(cudaStreamSynchronize(ctx->stream));
    if (st != 0) return comm_failed(t, loss_host);
    return LNB_OK;
}
