// fused_tc.cu -- the fused tensor-core train / render step for small coordinate MLPs (sm_100a).
//
// Two kernels share this file's machinery (PTX wrappers, slab layout, weight image, reduce + Adam + peer all-reduce):
//   fused_v1_kernel  (below)        one 128-sample tile per 128-thread CTA.  Its FWD instantiation is the forward-only
//                                   (render) kernel: hidden activations live in tensor memory and registers only.
//   fused_mg_kernel  (fused_mg.cuh) the train step: one CTA per SM, up to seven 128-thread groups, adjoints in place.
//
// ONE kernel does, per 128-sample tile held by a persistent CTA (or group):
//   features -> bf16 A tile in shared memory            (scripts/nerf.py layer_input)
//   L x [ tcgen05.mma (M=128 samples, N=width, fp32 accumulators in TMEM)
//         -> tcgen05.ld epilogue: +bias, ReLU -> bf16 -> next layer's A tile ]  (nerf.py:67-146)
//   head: sigmoid rgb / ReLU sigma (nerf.py:147-167) or sigmoid (mlp_fit.py:121-132)
//   per-ray compositing with warp-shuffle product scans (nerf.py:176-288), SSE loss (:297-302)
//   reverse: compositing adjoint (reverse affine scan, no division), then per layer
//         dH = dZ W^T on tcgen05 (the SAME shared-memory copy of W, addressed MN-major),
//         ReLU mask from the stored activations, and
//         dW_l += H_l^T dZ_l on tcgen05 with the contraction over the tile's 128 samples,
//         accumulated in TMEM across ALL tiles of the CTA (bias gradient = an all-ones feature).
//   one write of the CTA's dW / loss partials at the end; a tiny second kernel reduces the
//   partials over CTAs in a fixed order and applies the seed (SURVEY.md 8 a7: grads are linear
//   in _dreturn, the hosts pass the loss).
//
// Operands are bf16 (8-bit mantissa), accumulation fp32: this is LNB_PATH_TC, with the error
// bound stated in DESIGN.md and asserted in tests/test_gpu_tc.py.  The exact fp32 path is
// kernels_f32.cu.
//
// Shared-memory operand layout ("slab" layout, no swizzle): a [128 rows][F features] bf16 matrix
// is stored as F/8 slabs of 2048 B; slab c holds features 8c..8c+7 of every row, row r at byte
// r*16.  One 8x8 block (8 rows x 16 B) is exactly a UMMA core matrix, so the same bytes are
//   * a K-major  operand with rows as M/N   (SBO = 128 B between 8-row groups, LBO = slab stride)
//   * an MN-major operand with rows as K    (SBO = slab stride, LBO = 128 B)
// which is what lets H_l serve as A for the forward MMA and as A^T for the dW MMA, and W_l as B
// for forward and B^T for backward, without any transposed copy.
#include <cuda_bf16.h>
#include <stdio.h>
#include <stdlib.h>

#include <type_traits>
#include <vector>

#include "camera.cuh"
#include "lnb_internal.h"
#include "tc_ptx.cuh"

namespace {

constexpr int TILE = 128;          // samples per tile = UMMA M
constexpr int SLAB = TILE * 16;    // bytes per 8-feature slab
constexpr int MAXL = 4;            // layers supported by the fused kernel

// camera mode in float32 (the tensor-core path): see camera.cuh / lnb_camera
struct CamF32 {
    float c2w[12];
    float inv_fx, inv_fy, cx, cy, step, near, far, dt_lin, dt_str;   // dt_lin = (far-near)/(S-1), dt_str = (far-near)/S
    long long first_pixel;
    const int *pixels;
    unsigned long long seed;
    unsigned long long w_magic;      // floor(2^64 / width) + 1 (width >= 2): q / width = umul64hi(q, w_magic) for every 32-bit q
    int width, stratified;
    // views mode (the RAYS == 2 instantiations; lnb_views): pixels is the views' pixel list
    const double *poses;
    const int *view;
    const unsigned long long *seed_dev;
    long long P;
    int n_views;
};

struct alignas(16) TcParams {   // 16: the kernel parameters after it keep their alignment
    const float *X, *dists, *target, *ws, *bs;
    float *color;      // [R][3] or NULL
    float *part;       // [grid][part_stride]
    float *dbg;        // optional [N][4] head outputs (debug)
    const void *wimg;  // weight image built by tc_prep_kernel (ImgMap)
    // rays mode (X == NULL): features are computed in the kernel from rays and sample depths
    const void *rays_o, *rays_d, *tvals; // [R][3], [R][3], [R][S]; float64 when ray_f64 else float32
    int ray_f64, pe_bands;
    int dir_bands;     // view-direction bands E_d of a DIRS instantiation (dims[0] == 6 + 6 pe_bands + 6 E_d)
    int cam_mode;      // rays and depths generated from `cam` instead of read from rays_o / rays_d / tvals
    CamF32 cam;
    int *t_dev;        // optimiser step counter, incremented once per launch (or NULL)
    int *tile_counter; // dynamic tile scheduler: tiles beyond the first are claimed with atomicAdd
    long long N;       // samples (rows of X)
    int R, S, G, rows_per_tile, n_tiles;
    int L, dims[MAXL + 1], max_in, max_out;
    int K0P;           // padded input width (multiple of 16, <= 64)
    int head, want_grad, Wt;
    int part_stride;
    int part_off[MAXL]; // offset of layer l's [(in_l+1) x out_l] block inside a partial
    float *weights;     // [R][S] compositing weights of a train step (lnb_trainer_step_weights), or NULL
    // compositing extras (lnb_composite), read by the EXT instantiations only
    float *acc, *depth; // [R] opacity / expected depth, or NULL
    int background;     // 1: colour += (1 - acc) bg
    float bg[3];
};

// ---------------------------------------------------------------------------------------------
// PTX wrappers of these kernels only (the shared ones are in tc_ptx.cuh)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0;
    unsigned long long t0 = 0;
    for (uint32_t it = 0; !done; ++it) {
        // the suspend-time hint lets the warp sleep in hardware instead of burning issue slots
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity), "r"(100000u) : "memory");
        if (!done && (it & 0x3FFu) == 0x3FFu) {
            // never hang the GPU: a lost arrival is a bug, fail loudly (10 s by the global timer)
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 10000000000ull) __trap();
        }
    }
}
// The forward-only kernel's wait for an MMA stage: nine CTAs share an SM and a stage takes ~1 us there, during which the
// hardware-suspended try_wait comes back ~10 times (any barrier event of the SM wakes it).  The render kernel is bound by
// instruction issue and these polls were 30 % of its instructions at nine per iteration (counter, time-out test, sleep);
// here an iteration is the try_wait and one branch, the counter ticks once per four polls.  The multi-group train kernel's
// groups wait with it too: with seven groups on an SM a hardware-suspended try_wait is woken by the other groups' barrier
// traffic and re-polls several times per wait (an explicit __nanosleep between polls, tried before, does not actually sleep
// there and costs five instructions).
__device__ __forceinline__ void mbar_wait_tight(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        ".reg .u32 n;\n\t"
        "mov.u32 n, 0;\n"
        "LNB_WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra LNB_WAIT_DONE;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra LNB_WAIT_DONE;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra LNB_WAIT_DONE;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra LNB_WAIT_DONE;\n\t"
        "add.u32 n, n, 1;\n\t"
        "setp.lt.u32 q, n, 0x1000000;\n\t"
        "@q bra LNB_WAIT_LOOP;\n\t"
        "trap;\n"                       // never hang the GPU: a lost arrival is a bug, fail loudly (seconds)
        "LNB_WAIT_DONE:\n\t"
        "}"
        :: "r"(bar), "r"(parity), "r"(100000u) : "memory");
}

// A operand from tensor memory (M = 128 rows = TMEM lanes; a 16-bit K-step of 16 is 8 columns, element 2c in the low half
// of column c), B from shared memory
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// named barrier of the 128 threads of one tile: id 0 in the one-tile-per-CTA kernel (the whole CTA, = __syncthreads()),
// g + 1 for group g of the multi-group kernel
__device__ __forceinline__ void bar_tile(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(TILE) : "memory"); }

// UMMA shared-memory descriptor, SWIZZLE_NONE (cute::UMMA::SmemDescriptor): start>>4 [0,14),
// LBO>>4 [16,30), SBO>>4 [32,46), version=1 [46,48), layout_type=0 [61,64)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo)
{
    return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) | (1ull << 46);
}

__device__ __forceinline__ float sigmoid_f(float z) { return __fdividef(1.0f, 1.0f + __expf(0.0f - z)); }
// two floats -> packed bf16 pair (lo = first), with ReLU: ONE instruction (F2FP.RELU.BF16)
__device__ __forceinline__ uint32_t pack_relu_bf16(float lo, float hi)
{
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// 0xFFFF per half where the bf16 half is > 0 (post-ReLU activations are >= 0)
__device__ __forceinline__ uint32_t gt0_mask_bf16x2(uint32_t h)
{
    uint32_t r;
    asm("set.gt.u32.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(h), "r"(0u));
    return r;
}


// sin / cos of a sample coordinate for the positional encoding: one Cody-Waite step to [-pi, pi], then the
// MUFU approximations (abs. error ~2^-21 there); doubled E-1 times this stays far below the bf16 operand step
__device__ __forceinline__ void pe_sincos(float x, float *s, float *c)
{
    const float k = rintf(x * 0.15915494309189535f);
    float r = fmaf(k, -6.28318548202514648f, x);
    r = fmaf(k, 1.7484555e-7f, r);
    __sincosf(r, s, c);
}

// ---------------------------------------------------------------------------------------------
// the kernel.  HP = padded hidden width (16/32/64): every hidden layer has width+1 <= HP.
// 128 threads: thread r owns row r of the tile (TMEM lane r).  Thread 0 issues the MMAs and the
// bulk-async (TMA) copies: the weight image once, the next tile's features every tile.
//
// Shared memory, in this order so that an M=64 MN-major read of A_l (8 slabs from its start)
// always stays inside live shared memory:
//   A0 [K0P/8 slabs] | A1 .. A_{L-1} [HP/8 slabs each] | dZ_0 .. dZ_{L-2} [HP/8 each] | dZ_{L-1} [2]
//   | weight image: W_0 .. W_{L-1} (bf16 slabs), biases (fp32)      <- one TMA per CTA
//   | stage: fp32 features of the next tile                          <- one TMA per tile
//   | compositing scratch | mbarriers
// TMEM (128 columns for 3 layers of width <= 31): [0,HP) holds each layer's output / dH in turn
// (its epilogue drains it before the next MMA is issued); [HP, HP+ndw) holds ONE concatenated
// weight-gradient accumulator: all A_l buffers are contiguous in shared memory and so are all
// dZ_l buffers, so a single M=128 x N=ndw MMA per 16-sample K-step computes
// [A_0|A_1|..]^T [dZ_0|dZ_1|..]; the blocks (A_l, dZ_l) on its diagonal are the dW_l (the
// off-diagonal blocks are never read).  8 MMAs per tile instead of 8 per layer.
// Every MMA's operands are tile-invariant, so the descriptors are computed once per CTA into a
// shared-memory "MMA program"; issuing a stage is a loop of (load 32 B record, tcgen05.mma).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// tensor-memory allocation for `need` columns: a power of two, at least 32
__host__ __device__ inline uint32_t tmem_alloc_cols(int need)
{
    return need <= 32 ? 32 : (need <= 64 ? 64 : (need <= 128 ? 128 : (need <= 256 ? 256 : 512)));
}

// The weight image every CTA of the fused kernels copies: [W_0 .. W_{L-1} bf16 slabs][bias fp32 MAXL x HP], built by
// tc_prep_kernel in global memory and refreshed in place by the fused Adam update.  W_l holds Kp = kp(l) input rows
// (K0P for the first layer, HP after) of Np = np(l) columns (HP, 16 for the head) in the slab layout.  The A operands carry
// an all-ones feature at column in_l (it exists for the bias gradient), so row in_l of a HIDDEN layer's W holds the bias
// b_l (the MMA adds it) and, at column out_l, a 1.0 that re-creates the ones feature in the layer's output: the hidden-layer
// epilogue is then just ReLU + pack.  The head keeps its bias in the fp32 tail [MAXL][HP] (zero for hidden layers).  In
// the adjoint pass these extra entries only feed column in_l of dH_l, which becomes the ones column of dZ_{l-1}: it meets
// zero weight columns and lands in weight-gradient entries nobody reads.
struct ImgMap {
    int L, HP, K0P;
    int dims[MAXL + 1];
    __host__ __device__ int np(int l) const { return l < L - 1 ? HP : 16; }
    __host__ __device__ int kp(int l) const { return l == 0 ? K0P : HP; }
    __host__ __device__ int w_off(int l) const
    {
        int o = 0;
        for (int i = 0; i < l; ++i) o += np(i) * kp(i) * 2;
        return o;
    }
    __host__ __device__ int bytes() const { return w_off(L) + MAXL * HP * 4; }
    __device__ float *bias(uint8_t *img) const { return reinterpret_cast<float *>(img + w_off(L)); }
    __device__ void put_w(uint8_t *img, int l, int k, int j, float v) const
    {
        reinterpret_cast<__nv_bfloat16 *>(img + w_off(l))[(k >> 3) * (np(l) * 8) + j * 8 + (k & 7)] = __float2bfloat16_rn(v);
    }
    __device__ void put_b(uint8_t *img, int l, int j, float v) const
    {
        if (l < L - 1) put_w(img, l, dims[l], j, v);   // hidden layers: bias row of the MMA operand
        else bias(img)[l * HP + j] = v;                 // head: fp32
    }
};

template <int HP>
struct TcLayout {
    static constexpr int HSL = HP / 8;
    // TMEM columns: [0,HP) the layer output / dH region (drained by its epilogue before the next
    // MMA is issued), [HP, HP + ndw) the concatenated dW accumulator (see issue of the dW stage)
    __host__ __device__ static int ndw(int L) { return (L - 1) * HP + 16; }
    // forward only (render): no adjoint buffers, no dW accumulator -> more CTAs per SM
    __host__ __device__ static uint32_t tmem_cols(int L, bool grad = true)
    {
        return tmem_alloc_cols(grad ? HP + ndw(L) : HP + HP / 2);   // forward only: result columns + the next layer's bf16 A operand
    }
    static constexpr int MAX_STAGES = 2 * MAXL + 1; // records of the per-CTA MMA program
    __host__ __device__ static int a_off(int l, int K0P) { return l == 0 ? 0 : (K0P / 8 + (l - 1) * HSL) * SLAB; }
    __host__ __device__ static int dz_off(int l, int L, int K0P) { return (K0P / 8 + (L - 1) * HSL + l * HSL) * SLAB; }
    // forward only (render): nothing is kept for a weight gradient, so only A_0 is in shared memory; the hidden activations
    // go from the epilogue's registers straight into TENSOR MEMORY (tcgen05.st) and the next layer's MMA takes its A operand
    // from there: no shared-memory store, no operand fetch.  A_0 is followed by two slabs of per-ray colour / target scratch.
    __host__ __device__ static int fwd_slabs(int K0P) { return K0P / 8; }
    __host__ __device__ static int act_bytes(int L, int K0P, bool grad = true)
    {
        return grad ? (K0P / 8 + 2 * (L - 1) * HSL + 2) * SLAB : (fwd_slabs(K0P) + 2) * SLAB;
    }
    // the weight image of this width (ImgMap)
    __host__ __device__ static int np(int l, int L) { return ImgMap{L, HP, 0, {}}.np(l); }
    __host__ __device__ static int kp(int l, int K0P) { return ImgMap{0, HP, K0P, {}}.kp(l); }
    __host__ __device__ static int w_off(int l, int L, int K0P) { return ImgMap{L, HP, K0P, {}}.w_off(l); }
    __host__ __device__ static int wimg_bytes(int L, int K0P) { return ImgMap{L, HP, K0P, {}}.bytes(); }
    __host__ __device__ static int stage_bytes(int c_in, int K0P) { return (TILE * c_in * 4 + 32 + K0P * 4 + 15) / 16 * 16; }
    static constexpr int SCRATCH_FLOATS = 48; // colour + target per ray, scan carries, loss
    __host__ __device__ static size_t total(int L, int K0P, int c_in, bool rays = false, bool grad = true)
    {
        // the concatenated dW MMA reads 16 slabs (M = 128 features) from the start of shared
        // memory whatever the real feature count: keep that inside the allocation
        const size_t t = (size_t)act_bytes(L, K0P, grad) + wimg_bytes(L, K0P) + (rays ? 0 : stage_bytes(c_in, K0P)) + SCRATCH_FLOATS * 4 + 64 + MAX_STAGES * 48;
        return (grad && t < 16 * SLAB) ? 16 * SLAB : t;
    }
};

// fp32 padded weights and biases -> the weight image (ImgMap)
__global__ void tc_prep_kernel(const TcParams p, const ImgMap im, uint8_t *__restrict__ img)
{
    const int L = im.L;
    for (int l = 0; l < L; ++l) {
        const int in_l = im.dims[l], out_l = im.dims[l + 1], Np = im.np(l), Kp = im.kp(l);
        const float *wl = p.ws + (size_t)l * p.max_in * p.max_out;
        const float *bl = p.bs + (size_t)l * p.max_out;
        for (int e = threadIdx.x; e < Np * Kp; e += blockDim.x) {
            const int k = e / Np, j = e % Np; // consecutive threads -> consecutive j (coalesced reads)
            if (k == in_l && l < L - 1) im.put_b(img, l, j, j < out_l ? __ldg(bl + j) : (j == out_l ? 1.0f : 0.0f));
            else im.put_w(img, l, k, j, k < in_l && j < out_l ? __ldg(wl + (size_t)k * p.max_out + j) : 0.0f);
        }
    }
    for (int e = threadIdx.x; e < MAXL * im.HP; e += blockDim.x) {
        const int l = e / im.HP, j = e % im.HP;
        im.bias(img)[e] = (l == L - 1 && j < im.dims[l + 1]) ? __ldg(p.bs + (size_t)l * p.max_out + j) : 0.0f;
    }
}

// ---------------------------------------------------------------------------------------------
// Per-tile stages of the one-tile-per-CTA kernel (below) and the multi-group train kernel (fused_mg.cuh).  Thread tid of a
// tile's 128 owns row tid: sample smp of the tile's ray ray_l.
// ---------------------------------------------------------------------------------------------

// TMA source of a tile's features (16 B aligned start, `lead` floats in front of the tile)
__device__ __forceinline__ const void *x_src(const TcParams &p, int tile, int c_in, int &lead, uint32_t &bytes)
{
    const long long row0 = (long long)tile * p.rows_per_tile;
    long long rem = p.N - row0;
    const int valid = rem < p.rows_per_tile ? (int)rem : p.rows_per_tile;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p.X + row0 * c_in);
    const uintptr_t a16 = a & ~(uintptr_t)15;
    lead = (int)((a - a16) >> 2);
    bytes = (uint32_t)(((a - a16) + (uintptr_t)valid * c_in * 4 + 15) & ~(uintptr_t)15);
    return reinterpret_cast<const void *>(a16);
}

// This row's inputs other than its features, loaded early (latency-tolerant, consumed after the MLP forward): the sample
// spacing `dist` and, at a ray's first sample, the ray's target colour.  From rays (RAYS) also the sample point x:
// pts = o + d t (train_nerf.py:289-299), dist = t[s+1] - t[s], last 1e8 (train_nerf.py:306-311).  x and dist stay 0 in a
// row past the tile's live samples.  DIRS: also the ray's unit direction u = d / |d| (0 in a row that is not live).
// RAYS: 0 features, 1 rays or camera mode (p.cam_mode), 2 views mode (a separate instantiation, so that the camera prologue
// of the others stays as it was).
template <int RAYS, bool DIRS>
__device__ __forceinline__ void sample_inputs(const TcParams &p, long long row0, int ray0, int tid, int smp, int ray_l, bool live,
                                              float (&x)[3], float &dist, float (&tg)[3], float (&u)[3])
{
    const int S = p.S;
    dist = 0.0f;
    tg[0] = tg[1] = tg[2] = 0.0f;
    if (p.head == LNB_HEAD_NERF && live) {
        if (!RAYS) dist = __ldg(p.dists + row0 + tid);
        if (p.target && smp == 0) {
            const float *t = p.target + (size_t)(ray0 + ray_l) * 3;   // a tile holds G whole rays: ray0 = row0 / S (R is an int)
            tg[0] = __ldg(t); tg[1] = __ldg(t + 1); tg[2] = __ldg(t + 2);
        }
    }
    x[0] = x[1] = x[2] = 0.0f;
    if (DIRS) u[0] = u[1] = u[2] = 0.0f;
    if (!RAYS || !live) return;
    const long long ray = ray0 + ray_l;
    if (RAYS == 2) {
        // views mode: camera mode's ray of pixel q = pixels[r] under the pose poses[view[r]] (rounded to float32 as camera
        // mode rounds its c2w), the jitter keyed by g = view[r] * P + q under seed'.  An out-of-range index makes x and
        // dist NaN (dist too, so the colour is NaN whatever the MLP makes of x) and reads the table's first pose.
        const CamF32 &c = p.cam;
        const int v = __ldg(c.view + ray), q = __ldg(c.pixels + ray);
        const bool ok = (unsigned)v < (unsigned)c.n_views && (long long)(unsigned)q < c.P;
        const double *m = c.poses + 12 * (ok ? v : 0);
        const unsigned long long seed = c.seed_dev ? __ldg(c.seed_dev) : c.seed;
        const long long g = (long long)v * c.P + q;
        const unsigned uq = (unsigned)q, row = (unsigned)__umul64hi((unsigned long long)uq, c.w_magic), col = uq - row * (unsigned)c.width;
        const float fi = col == (unsigned)c.width - 1 ? 1.0f : (float)col * c.step, fj = row == (unsigned)c.width - 1 ? 1.0f : (float)row * c.step;
        const float dx = (fi - c.cx) * c.inv_fx, dy = (c.cy - fj) * c.inv_fy;
        float tt, tn;
        if (c.stratified) {
            tt = fmaf((float)smp + (float)lnb_uniform_bits(seed, g, smp) * (1.0f / 16777216.0f), c.dt_str, c.near);
            tn = fmaf((float)(smp + 1) + (float)lnb_uniform_bits(seed, g, smp + 1) * (1.0f / 16777216.0f), c.dt_str, c.near);
        } else {
            tt = smp == S - 1 && S > 1 ? c.far : fmaf((float)smp, c.dt_lin, c.near);
            tn = smp + 1 == S - 1 ? c.far : fmaf((float)(smp + 1), c.dt_lin, c.near);
        }
        dist = smp + 1 < S ? tn - tt : 1e8f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float dk = fmaf(dx, (float)__ldg(m + 4 * k), fmaf(dy, (float)__ldg(m + 4 * k + 1), 0.0f - (float)__ldg(m + 4 * k + 2)));
            x[k] = fmaf(dk, tt, (float)__ldg(m + 4 * k + 3));
            if (DIRS) u[k] = dk;
        }
        if (!ok) x[0] = x[1] = x[2] = dist = __int_as_float(0x7fc00000);
    } else if (p.cam_mode) {
        // ray of pixel q and depth of sample smp straight from the pose (get_rays, train_nerf.py:23-62; linspace /
        // stratified depths, train_nerf.py:289-311): no per-ray or per-sample input at all
        const CamF32 &c = p.cam;
        const long long q = c.pixels ? (long long)__ldg(c.pixels + ray) : c.first_pixel + ray;
        // q / width by the 64-bit reciprocal the launcher computed (exact for every 32-bit q)
        const unsigned uq = (unsigned)q, row = c.width == 1 ? uq : (unsigned)__umul64hi((unsigned long long)uq, c.w_magic), col = uq - row * (unsigned)c.width;
        const float fi = col == (unsigned)c.width - 1 ? 1.0f : (float)col * c.step, fj = row == (unsigned)c.width - 1 ? 1.0f : (float)row * c.step;
        const float dx = (fi - c.cx) * c.inv_fx, dy = (c.cy - fj) * c.inv_fy;
        float tt, tn;
        if (c.stratified) {
            tt = fmaf((float)smp + (float)lnb_uniform_bits(c.seed, q, smp) * (1.0f / 16777216.0f), c.dt_str, c.near);
            tn = fmaf((float)(smp + 1) + (float)lnb_uniform_bits(c.seed, q, smp + 1) * (1.0f / 16777216.0f), c.dt_str, c.near);
        } else {
            tt = smp == S - 1 && S > 1 ? c.far : fmaf((float)smp, c.dt_lin, c.near);
            tn = smp + 1 == S - 1 ? c.far : fmaf((float)(smp + 1), c.dt_lin, c.near);
        }
        dist = smp + 1 < S ? tn - tt : 1e8f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float dk = fmaf(dx, c.c2w[4 * k], fmaf(dy, c.c2w[4 * k + 1], 0.0f - c.c2w[4 * k + 2]));
            x[k] = fmaf(dk, tt, c.c2w[4 * k + 3]);
            if (DIRS) u[k] = dk;
        }
    } else if (p.ray_f64) {
        const double *o = reinterpret_cast<const double *>(p.rays_o) + ray * 3;
        const double *d = reinterpret_cast<const double *>(p.rays_d) + ray * 3;
        const double *tv = reinterpret_cast<const double *>(p.tvals) + row0 + tid;
        const double tt = __ldg(tv);
        dist = smp + 1 < S ? (float)(__ldg(tv + 1) - tt) : 1e8f;
#pragma unroll
        for (int c = 0; c < 3; ++c) x[c] = (float)(__ldg(o + c) + __ldg(d + c) * tt);
        if (DIRS)
            for (int c = 0; c < 3; ++c) u[c] = (float)__ldg(d + c);
    } else {
        const float *o = reinterpret_cast<const float *>(p.rays_o) + ray * 3;
        const float *d = reinterpret_cast<const float *>(p.rays_d) + ray * 3;
        const float *tv = reinterpret_cast<const float *>(p.tvals) + row0 + tid;
        const float tt = __ldg(tv);
        dist = smp + 1 < S ? __ldg(tv + 1) - tt : 1e8f;
#pragma unroll
        for (int c = 0; c < 3; ++c) x[c] = fmaf(__ldg(d + c), tt, __ldg(o + c));
        if (DIRS)
            for (int c = 0; c < 3; ++c) u[c] = __ldg(d + c);
    }
    if (DIRS) {
        const float inv = rsqrtf(fmaf(u[0], u[0], fmaf(u[1], u[1], u[2] * u[2])));
#pragma unroll
        for (int c = 0; c < 3; ++c) u[c] *= inv;
    }
}

// The positional encoding (pos_encoding.py:38-70) of the sample point x into this row's first `live_slabs` slabs of A_0,
// through store(slab, its 16 bytes of the row).  sn / cs: sin / cos of x (pe_sincos); the higher bands by angle doubling
// (sin 2a = 2 s c, cos 2a = 1 - 2 s^2), which amplifies the base error by 2^(E-1): ~1e-6 at E = 5, far below the bf16
// operand rounding.  Feature f = 3 * slot + coord: x0 x1 | x2 s0 | s1 s2 | c0 c1 | c2 s0' | ... as bf16 pairs (pair j =
// features 2j, 2j+1); band i fills pairs 1+3i .. 3+3i and leaves its last cosine pending; the ones column (feature 3 + 6E,
// odd) closes the pending pair.  Four pairs make a slab's 16 bytes, stored as soon as they are complete.
template <class Store>
__device__ __forceinline__ void pack_pe(const float (&x)[3], float (&sn)[3], float (&cs)[3], int pe_bands, int live_slabs, Store &&store)
{
    uint32_t q4[4] = {pack_bf16(x[0], x[1]), 0u, 0u, 0u};
    float pend = x[2];
    bool closed = false;
    auto put = [&](int j, uint32_t v) {            // j is a compile-time constant at every call site
        q4[j & 3] = v;
        if ((j & 3) == 3) {
            if ((j >> 2) < live_slabs) store(j >> 2, make_uint4(q4[0], q4[1], q4[2], q4[3]));
            q4[0] = q4[1] = q4[2] = q4[3] = 0u;
        }
    };
    // warp-uniform branches: the bands that are off cost nothing
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        if (i < pe_bands) {
            put(1 + 3 * i, pack_bf16(pend, sn[0]));
            put(2 + 3 * i, pack_bf16(sn[1], sn[2]));
            put(3 + 3 * i, pack_bf16(cs[0], cs[1]));
            pend = cs[2];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float s2 = 2.0f * sn[c] * cs[c], c2 = fmaf(-2.0f * sn[c], sn[c], 1.0f);
                sn[c] = s2; cs[c] = c2;
            }
        } else {
            if (closed && ((1 + 3 * i) >> 2) >= live_slabs) break;   // no live slab left to store (slab 7 then is not live either)
            put(1 + 3 * i, closed ? 0u : pack_bf16(pend, 1.0f));
            put(2 + 3 * i, 0u);
            put(3 + 3 * i, 0u);
            closed = true;
        }
    }
    put(31, closed ? 0u : pack_bf16(pend, 1.0f));
}

// The same with the view direction (rays / camera mode with dims[0] = (3 + 6E) + (3 + 6E_d)): the stream of 3-vectors
// x, its 2E band slots, u, its 2E_d band slots, then the ones column, into this row's first (dims[0] + 8) / 8 slabs of A_0.
// x starts a pair, so its bands leave their last cosine pending as in pack_pe; the position part is odd-long, so u starts
// mid-pair (pend, u0) (u1, u2) and its bands pair up without a pending element; the ones column (feature dims[0], even)
// opens a pair.  The pair index depends on E, so the four pairs of a slab are selected at run time.  u = d rsqrt(d.d) in
// fp32 is within ~1e-7 of the float64 unit vector, and |u| <= 1 keeps pe_sincos at its base error (~2^-21) without
// range reduction; angle doubling amplifies that by 2^(E_d - 1) <= 8 for E_d <= 4: ~1e-6, far below the bf16 step.
template <class Store>
__device__ __forceinline__ void pack_pe_dirs(const float (&x)[3], const float (&u)[3], int pe_bands, int dir_bands, Store &&store)
{
    uint32_t q4[4] = {0u, 0u, 0u, 0u};
    int j = 0;                                     // the next pair (features 2j, 2j+1)
    auto put = [&](uint32_t v) {
        const int k = j & 3;
        q4[0] = k == 0 ? v : q4[0];
        q4[1] = k == 1 ? v : q4[1];
        q4[2] = k == 2 ? v : q4[2];
        q4[3] = k == 3 ? v : q4[3];
        if (k == 3) {
            store(j >> 2, make_uint4(q4[0], q4[1], q4[2], q4[3]));
            q4[0] = q4[1] = q4[2] = q4[3] = 0u;
        }
        ++j;
    };
    float sn[3], cs[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) pe_sincos(x[c], &sn[c], &cs[c]);
    put(pack_bf16(x[0], x[1]));
    float pend = x[2];
    for (int i = 0; i < pe_bands; ++i) {
        put(pack_bf16(pend, sn[0]));
        put(pack_bf16(sn[1], sn[2]));
        put(pack_bf16(cs[0], cs[1]));
        pend = cs[2];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float s2 = 2.0f * sn[c] * cs[c], c2 = fmaf(-2.0f * sn[c], sn[c], 1.0f);
            sn[c] = s2; cs[c] = c2;
        }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) pe_sincos(u[c], &sn[c], &cs[c]);
    put(pack_bf16(pend, u[0]));
    put(pack_bf16(u[1], u[2]));
    for (int i = 0; i < dir_bands; ++i) {
        put(pack_bf16(sn[0], sn[1]));
        put(pack_bf16(sn[2], cs[0]));
        put(pack_bf16(cs[1], cs[2]));
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float s2 = 2.0f * sn[c] * cs[c], c2 = fmaf(-2.0f * sn[c], sn[c], 1.0f);
            sn[c] = s2; cs[c] = c2;
        }
    }
    put(pack_bf16(1.0f, 0.0f));
    while (j & 3) put(0u);
}

// Features mode: this row's c_in fp32 features (xr) -> its first (c_in + 8) / 8 slabs of A_0, through store(slab, its
// 16 bytes of the row): full slabs, then the last one with the ones column (feature c_in, the bias-gradient feature)
// written explicitly and zeros after it.  A row past the tile's valid ones stores zeros.
template <class Store>
__device__ __forceinline__ void pack_features(const float *xr, int c_in, bool row_live, Store &&store)
{
    // the slab count from an opaque copy of c_in: otherwise the compiler hoists the loop's trip-count arithmetic out of the
    // caller's tile loop, where it holds registers for the whole tile (a dozen more in the one-tile-per-CTA kernel)
    int n = c_in;
    asm volatile("" : "+r"(n));
    const int a0s = (n + 8) >> 3;
    for (int c8 = 0; c8 < a0s - 1; ++c8) {         // (a0s - 1) * 8 <= c_in: every column of these slabs is a feature
        uint4 q = make_uint4(0, 0, 0, 0);
        if (row_live) {
            float f[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) f[j] = xr[c8 * 8 + j];
            q = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
        }
        store(c8, q);
    }
    const int c8 = a0s - 1;
    uint4 q = make_uint4(0, 0, 0, 0);
    if (row_live) {
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { const int c = c8 * 8 + j; f[j] = c < c_in ? xr[c] : (c == c_in ? 1.0f : 0.0f); }
        q = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
    }
    store(c8, q);
}

// shared-memory scratch of the head and compositing stage of one tile
struct CompScratch {
    float *color, *tgt;             // [rays of the tile][3]: colour sums, targets
    float *ext;                     // EXT: [rays of the tile][2]: acc and depth sums
    float *tailp;                   // [4] inclusive product at lane 31 of each warp
    int *tail_s;                    // [4] sample index at lane 31
    float *headq, *headA, *headB;   // [5] q at lane 0 of each warp; the affine suffix scan's head of each warp
};

// Depth t_s of sample smp of ray `ray` (row `row` of the batch) for the depth map: re-loaded (rays mode) or re-derived from
// the camera exactly as sample_inputs forms it, at the compositing stage rather than held in a register across the MMAs.
template <bool VIEWS>
__device__ __forceinline__ float tile_sample_depth(const TcParams &p, long long ray, int smp, long long row)
{
    if (VIEWS) {   // views mode: camera mode's depth under the ray's jitter key g = view * P + q and seed'
        const CamF32 &c = p.cam;
        if (!c.stratified) return smp == p.S - 1 && p.S > 1 ? c.far : fmaf((float)smp, c.dt_lin, c.near);
        const long long g = (long long)__ldg(c.view + ray) * c.P + __ldg(c.pixels + ray);
        const unsigned long long seed = c.seed_dev ? __ldg(c.seed_dev) : c.seed;
        return fmaf((float)smp + (float)lnb_uniform_bits(seed, g, smp) * (1.0f / 16777216.0f), c.dt_str, c.near);
    }
    if (p.cam_mode) {
        const CamF32 &c = p.cam;
        const long long q = c.pixels ? (long long)__ldg(c.pixels + ray) : c.first_pixel + ray;
        if (c.stratified) return fmaf((float)smp + (float)lnb_uniform_bits(c.seed, q, smp) * (1.0f / 16777216.0f), c.dt_str, c.near);
        return smp == p.S - 1 && p.S > 1 ? c.far : fmaf((float)smp, c.dt_lin, c.near);
    }
    return p.ray_f64 ? (float)__ldg(reinterpret_cast<const double *>(p.tvals) + row) : __ldg(reinterpret_cast<const float *>(p.tvals) + row);
}

// The head on the last layer's pre-activations hz, the loss (added to loss_acc) and, with GRAD, dz = the adjoint of hz
// (unit seed).  `bar` is the tile's named barrier (bar_tile).  EXT (the extras instantiations): the compositing weights of
// live rows go to p.weights when it is set (lnb_trainer_step_weights), acc and depth ride in the segmented colour sum as
// two more channels (p.acc / p.depth), and with p.background the colour gets (1 - acc) bg before the loss, the weight
// adjoint uses rgb - bg.  A separate instantiation, so the plain train and render kernels stay as they were.
template <bool GRAD, bool EXT = false, bool VIEWS = false>
__device__ __forceinline__ void head_and_composite(const TcParams &p, const CompScratch &s, int bar, const float (&hz)[4], float dist,
                                                   const float (&tg)[3], long long row0, int ray0, int valid, int tid, int smp,
                                                   int ray_l, bool live, float &loss_acc, float (&dz)[4])
{
    const int warp = tid >> 5, lane = tid & 31, S = p.S;
    dz[0] = dz[1] = dz[2] = dz[3] = 0.0f;
    if (p.head == LNB_HEAD_SIGMOID) {
        // mlp_fit: row r <-> target row (scripts/mlp_fit.py:121-145)
        if (tid < valid && row0 + tid < p.R) {
            const float *t = p.target + (row0 + tid) * p.Wt;
            for (int c = 0; c < p.Wt && c < 4; ++c) {
                float y = sigmoid_f(hz[c]);
                float d = y - __ldg(t + c);
                loss_acc = fmaf(d, d, loss_acc);
                dz[c] = 2.0f * d * (y * (1.0f - y));
            }
        }
        return;
    }
    // Compositing with one thread per sample (thread r <-> sample r of the tile): segmented warp-shuffle scans inside each
    // warp, carries across the 4 warps through shared memory.  scripts/nerf.py:176-288 and its reverse (SURVEY.md
    // Appendix B).
    const float cr = sigmoid_f(hz[0]), cg = sigmoid_f(hz[1]), cb = sigmoid_f(hz[2]);
    const float sg = fmaxf(hz[3], 0.0f);
    const float e = __expf((0.0f - sg) * dist);
    const float a = 1.0f - e;
    const float qv = live ? (1.0f - a) + 1e-10f : 1.0f;
    float pr = qv;                                   // segmented inclusive product
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        float o = __shfl_up_sync(0xffffffffu, pr, d);
        if (lane >= d && smp >= d) pr *= o;
    }
    if (lane == 31) { s.tailp[warp] = pr; s.tail_s[warp] = smp; }
    if (lane == 0) s.headq[warp] = qv;
    if (live && smp == 0) {
        s.color[ray_l * 3] = 0.f; s.color[ray_l * 3 + 1] = 0.f; s.color[ray_l * 3 + 2] = 0.f;
        if (EXT) { s.ext[ray_l * 2] = 0.f; s.ext[ray_l * 2 + 1] = 0.f; }
        s.tgt[ray_l * 3] = tg[0]; s.tgt[ray_l * 3 + 1] = tg[1]; s.tgt[ray_l * 3 + 2] = tg[2];
    }
    bar_tile(bar);
    float carry = 1.0f;                              // product of this ray's samples in earlier warps
    if (smp > lane) {
        for (int w2 = warp - 1; w2 >= 0; --w2) {
            carry *= s.tailp[w2];
            if (s.tail_s[w2] < 32) break;            // that warp's last segment started inside it
        }
    }
    const float Cpre = pr * carry;                   // true inclusive product prod_{k<=s} q_k
    const float T = (smp == 0) ? 1.0f : Cpre;
    const float wgt = a * T;
    if (EXT && live && p.weights) p.weights[row0 + tid] = wgt;
    {   // colour: segmented inclusive sums, one shared-memory atomic per (warp, ray) segment
        float s0 = live ? wgt * cr : 0.f, s1 = live ? wgt * cg : 0.f, s2 = live ? wgt * cb : 0.f;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            float o0 = __shfl_up_sync(0xffffffffu, s0, d), o1 = __shfl_up_sync(0xffffffffu, s1, d), o2 = __shfl_up_sync(0xffffffffu, s2, d);
            if (lane >= d && smp >= d) { s0 += o0; s1 += o1; s2 += o2; }
        }
        if (live && (lane == 31 || smp == S - 1)) {
            atomicAdd(s.color + ray_l * 3, s0); atomicAdd(s.color + ray_l * 3 + 1, s1); atomicAdd(s.color + ray_l * 3 + 2, s2);
        }
        if (EXT) {   // acc = sum w, depth = sum w t: the same segmented sum
            float s3 = live ? wgt : 0.f, s4 = (live && p.depth) ? wgt * tile_sample_depth<VIEWS>(p, ray0 + ray_l, smp, row0 + tid) : 0.f;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                float o3 = __shfl_up_sync(0xffffffffu, s3, d), o4 = __shfl_up_sync(0xffffffffu, s4, d);
                if (lane >= d && smp >= d) { s3 += o3; s4 += o4; }
            }
            if (live && (lane == 31 || smp == S - 1)) { atomicAdd(s.ext + ray_l * 2, s3); atomicAdd(s.ext + ray_l * 2 + 1, s4); }
        }
    }
    bar_tile(bar);
    float dc0 = 0.f, dc1 = 0.f, dc2 = 0.f;
    if (live) {
        float c0 = s.color[ray_l * 3], c1 = s.color[ray_l * 3 + 1], c2 = s.color[ray_l * 3 + 2];
        if (EXT) {
            const float acc = s.ext[ray_l * 2];
            if (p.background) {
                const float tr = 1.0f - acc;   // the light that reaches the background
                c0 = fmaf(tr, p.bg[0], c0); c1 = fmaf(tr, p.bg[1], c1); c2 = fmaf(tr, p.bg[2], c2);
            }
            if (smp == 0 && p.acc) p.acc[ray0 + ray_l] = acc;
            if (smp == 0 && p.depth) p.depth[ray0 + ray_l] = s.ext[ray_l * 2 + 1];
        }
        if (smp == 0 && p.color) {
            float *co = p.color + (size_t)(ray0 + ray_l) * 3;
            co[0] = c0; co[1] = c1; co[2] = c2;
        }
        // a train step always has a target (the launcher refuses a gradient without one); a forward-only call may pass none
        if (GRAD || p.target) {
            const float d0 = c0 - s.tgt[ray_l * 3], d1 = c1 - s.tgt[ray_l * 3 + 1], d2 = c2 - s.tgt[ray_l * 3 + 2];
            if (smp == 0) loss_acc += d0 * d0 + d1 * d1 + d2 * d2;
            dc0 = 2.0f * d0; dc1 = 2.0f * d1; dc2 = 2.0f * d2;
        }
    }
    if (!GRAD) return;
    // G_s = dT_s + q_{s+1} G_{s+1}: suffix scan of affine maps; B = 0 at a ray's last sample
    const float d_w = (EXT && p.background) ? (cr - p.bg[0]) * dc0 + (cg - p.bg[1]) * dc1 + (cb - p.bg[2]) * dc2
                                            : cr * dc0 + cg * dc1 + cb * dc2;
    const float dT = (smp == 0 || !live) ? 0.0f : d_w * a;
    float qn = __shfl_down_sync(0xffffffffu, qv, 1);
    if (lane == 31) qn = warp < 3 ? s.headq[warp + 1] : 0.0f;
    float Aa = dT, Bb = (live && smp + 1 < S) ? qn : 0.0f;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        float A2 = __shfl_down_sync(0xffffffffu, Aa, d);
        float B2 = __shfl_down_sync(0xffffffffu, Bb, d);
        if (lane + d < 32) { Aa = fmaf(Bb, A2, Aa); Bb = Bb * B2; }
    }
    if (lane == 0) { s.headA[warp] = Aa; s.headB[warp] = Bb; }
    bar_tile(bar);
    float Gn = 0.0f;                                 // G at lane 0 of the next warp
    for (int w2 = 3; w2 > warp; --w2) Gn = fmaf(s.headB[w2], Gn, s.headA[w2]);
    const float Gv = fmaf(Bb, Gn, Aa);
    float Cm1 = __shfl_up_sync(0xffffffffu, Cpre, 1);
    if (lane == 0) Cm1 = carry;
    if (smp == 0) Cm1 = 1.0f;
    const float d_alpha = d_w * T - Cm1 * Gv;
    if (live) {
        dz[0] = (wgt * dc0) * (cr * (1.0f - cr));
        dz[1] = (wgt * dc1) * (cg * (1.0f - cg));
        dz[2] = (wgt * dc2) * (cb * (1.0f - cb));
        dz[3] = sg > 0.0f ? d_alpha * e * dist : 0.0f;
    }
}

// One stage of an MMA program, built once per CTA (group) in shared memory: the MMAs of a stage differ only by constant
// increments of the descriptors' start-address fields (the K-steps).  With a_tmem set, `a` is the tensor-memory column of
// the A operand (8 columns per K-step) instead of a shared-memory descriptor.
struct StageRec { uint64_t a, b; uint32_t inc_a, inc_b, idesc, dcol; uint32_t count, a_tmem, pad0, pad1; };

// issue K-steps [k0, min(k1, count)) of a stage (one thread): the first accumulates into D when `acc` is set, the others
// always.  TS: the program has stages that take A from tensor memory.
template <bool TS>
__device__ __forceinline__ void issue_steps(const StageRec *rec, uint32_t tmem, uint32_t k0, uint32_t k1, uint32_t acc)
{
    const uint4 r0 = *reinterpret_cast<const uint4 *>(rec);
    const uint4 r1 = *(reinterpret_cast<const uint4 *>(rec) + 1);
    const uint4 r2 = *(reinterpret_cast<const uint4 *>(rec) + 2);
    if (k1 > r2.x) k1 = r2.x;
    uint32_t alo = r0.x + k0 * r1.x, blo = r0.z + k0 * r1.y;
    const uint32_t ahi = r0.y, bhi = r0.w;
    const uint32_t d = tmem + r1.w;
    if (TS && r2.y) {
        for (uint32_t k = k0; k < k1; ++k) {
            umma_bf16_ts(d, tmem + alo, ((uint64_t)bhi << 32) | blo, r1.z, acc);
            alo += r1.x; blo += r1.y; acc = 1u;
        }
        return;
    }
    for (uint32_t k = k0; k < k1; ++k) {
        umma_bf16(d, ((uint64_t)ahi << 32) | alo, ((uint64_t)bhi << 32) | blo, r1.z, acc);
        alo += r1.x; blo += r1.y; acc = 1u;
    }
}

// The ReLU adjoint of one row: dz = dH_l (the fp32 TMEM values v, rounded to bf16) where the stored bf16 activation a of
// A_l is positive, 0 elsewhere; 8 features per uint4.  Post-ReLU values are >= 0, so positive <=> non-zero halfword.
template <int HP>
__device__ __forceinline__ void relu_adjoint(const uint32_t (&v)[HP / 16][16], const uint4 (&a)[HP / 8], uint4 (&dz)[HP / 8])
{
#pragma unroll
    for (int c8 = 0; c8 < HP / 8; ++c8) {
        const uint32_t hw[4] = {a[c8].x, a[c8].y, a[c8].z, a[c8].w};
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int e = (c8 & 1) * 8 + 2 * j;
            o[j] = pack_bf16(__uint_as_float(v[c8 >> 1][e]), __uint_as_float(v[c8 >> 1][e + 1])) & gt0_mask_bf16x2(hw[j]);
        }
        dz[c8] = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// ---------------------------------------------------------------------------------------------
// the one-tile-per-CTA kernel.
// FWD: the forward-only (render) form, compiled separately: nothing of the backward pass in its register budget.  Its
// launch bounds are the CTAs per SM that tensor memory admits (512 columns / 64 per CTA = 8; 4 for the 64-wide form), not
// more: a ninth CTA could never allocate its columns and the tighter register budget only bought a spill.
// EXT: the extras instantiations (head_and_composite); its acc / depth scratch follows the colour / target scratch.
template <int RAYS, int HP, bool FWD, bool DIRS = false, bool EXT = false>
__global__ void __launch_bounds__(TILE, FWD ? (HP == 64 ? 4 : 8) : 1) fused_v1_kernel(const TcParams p)
{
    using LY = TcLayout<HP>;
    extern __shared__ __align__(1024) uint8_t smem[];
#ifdef LNB_TC_CLK
    const long long clk_start = clock64();
    unsigned long long gt_start;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt_start));
#endif
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = p.L, K0P = p.K0P, c_in = p.dims[0], S = p.S;
    const int act_bytes = LY::act_bytes(L, K0P, !FWD);
    uint8_t *const Wbase = smem + act_bytes;
    const float *const bias_s = reinterpret_cast<const float *>(Wbase + LY::w_off(L, L, K0P));
    float *const stage = reinterpret_cast<float *>(Wbase + LY::wimg_bytes(L, K0P));
    const int stage_sz = RAYS ? 0 : LY::stage_bytes(c_in, K0P);
    // per-ray colour / target scratch aliases dZ_0: it is dead from the top of a tile (the previous
    // tile's dW MMAs have been awaited) until the last backward epilogue writes it
    constexpr bool fwd_only = FWD;
    float *const color_s = reinterpret_cast<float *>(smem + (fwd_only ? LY::fwd_slabs(K0P) * SLAB : LY::dz_off(0, L, K0P)));
    float *const tgt_s = color_s + TILE * 3;
    float *const tailp = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(stage) + stage_sz); // [4] inclusive product at lane 31
    int *const tail_s = reinterpret_cast<int *>(tailp + 4);  // [4] sample index at lane 31
    float *const headq = tailp + 8;                          // [5] q at lane 0 of each warp
    float *const headA = tailp + 13;                         // [5]
    float *const headB = tailp + 18;                         // [5]
    float *const red_s = tailp + 24;                         // [8]
    uint64_t *const bar_p = reinterpret_cast<uint64_t *>(tailp + 48);
    uint32_t *const tmem_slot = reinterpret_cast<uint32_t *>(bar_p + 4);
    const uint32_t bar_mma = smem_u32(bar_p), bar_x = smem_u32(bar_p + 1), bar_w = smem_u32(bar_p + 2), bar_dw = smem_u32(bar_p + 3);
    // EXT: [TILE][2] more floats: colour, target and these fill the forward form's two scratch slabs exactly, and the train
    // form's dZ region (>= 4 slabs) has room to spare
    const CompScratch scratch{color_s, tgt_s, tgt_s + TILE * 3, tailp, tail_s, headq, headA, headB};
    StageRec *const prog = reinterpret_cast<StageRec *>(reinterpret_cast<uint8_t *>(bar_p) + 64);   // the MMA program

    // ---- one-time setup: zero activations, then TMA the weight image and the first tile
    // (every activation / adjoint buffer is fully rewritten each tile before it is read, except
    // the upper 8 features of dZ_{L-1}, which must stay zero)
    for (uint8_t *z = smem + LY::dz_off(L - 1, L, K0P) + tid * 16; z < smem + act_bytes; z += TILE * 16) *reinterpret_cast<uint4 *>(z) = make_uint4(0, 0, 0, 0);
    // A_0: only the slabs holding live features are rewritten per tile; its K padding, which the layer-0 MMA reads from
    // shared memory, must be zero
    for (uint8_t *z = smem + tid * 16; z < smem + (fwd_only ? LY::fwd_slabs(K0P) * SLAB : LY::a_off(1, K0P)); z += TILE * 16) *reinterpret_cast<uint4 *>(z) = make_uint4(0, 0, 0, 0);
    if (tid == 0) {
        mbar_init(bar_mma, 1);
        mbar_init(bar_x, 1);
        mbar_init(bar_w, 1);
        mbar_init(bar_dw, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // ---- build the MMA program.  Stages: fwd l (0..L-1), dH l (L+l, l = 1..L-1), dW (2L)
        for (int l = 0; l < L; ++l) {          // D[128 x Np] = A_l[128 x Kp] * W_l   (A, B K-major)
            const int Np = LY::np(l, L), Kp = LY::kp(l, K0P);
            const uint32_t a0 = smem_u32(smem + (fwd_only ? 0 : LY::a_off(l, K0P))), b0 = smem_u32(Wbase + LY::w_off(l, L, K0P));
            prog[l] = StageRec{smem_desc(a0, SLAB, 128), smem_desc(b0, Np * 16, 128), (uint32_t)(2 * SLAB) >> 4, (uint32_t)(2 * Np * 16) >> 4,
                               instr_desc(128, Np, 0, 0), 0u, (uint32_t)(Kp / 16), 0u, 0u, 0u};
            if (fwd_only && l > 0) { prog[l].a = (uint64_t)HP; prog[l].inc_a = 8u; prog[l].a_tmem = 1u; }   // A from TMEM, 8 columns per K-step
        }
        for (int l = 1; l < L; ++l) {          // dH_l[128 x Kp] = dZ_l[128 x Np] * W_l^T (same W bytes, MN-major)
            const int Np = LY::np(l, L), Kp = LY::kp(l, K0P);
            const uint32_t a0 = smem_u32(smem + LY::dz_off(l, L, K0P)), b0 = smem_u32(Wbase + LY::w_off(l, L, K0P));
            prog[L + l] = StageRec{smem_desc(a0, SLAB, 128), smem_desc(b0, 128, Np * 16), (uint32_t)(2 * SLAB) >> 4, 256u >> 4,
                                   instr_desc(128, Kp, 0, 1), 0u, (uint32_t)(Np / 16), 0u, 0u, 0u};
        }
        {                                      // dW: [all A]^T [all dZ], K = 128 samples, both MN-major
            const uint32_t a0 = smem_u32(smem), b0 = smem_u32(smem + LY::dz_off(0, L, K0P));
            prog[2 * L] = StageRec{smem_desc(a0, 128, SLAB), smem_desc(b0, 128, SLAB), 256u >> 4, 256u >> 4,
                                   instr_desc(128, LY::ndw(L), 1, 1), (uint32_t)HP, (uint32_t)(TILE / 16), 0u, 0u, 0u};
        }
    }
    if (warp == 0) tmem_alloc(smem_u32(tmem_slot), LY::tmem_cols(L, !FWD));
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // Programmatic dependent launch: everything above (shared-memory zeroing, barrier init, TMEM
    // allocation, the MMA program) overlaps the tail of the previous kernel in the stream; from here
    // on we read what it produced (weight image, tile counter, step counter).
    pdl_wait();
    pdl_trigger();
    if (tid == 0) {
        const uint32_t wb = (uint32_t)LY::wimg_bytes(L, K0P);
        mbar_expect_tx(bar_w, wb);
        bulk_g2s(smem_u32(Wbase), p.wimg, wb, bar_w);
        if (!RAYS) {
            int lead; uint32_t bytes;
            const void *src = x_src(p, blockIdx.x, c_in, lead, bytes);
            mbar_expect_tx(bar_x, bytes);
            bulk_g2s(smem_u32(stage), src, bytes, bar_x);
        }
    }
    const uint32_t tmem = *tmem_slot;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    uint32_t phase = 0, xphase = 0;
    float loss_acc = 0.0f;
    bool dw_started = false, dw_pending = false;
    uint32_t dwphase = 0;
    mbar_wait(bar_w, 0); // weights + biases have landed

    auto a_buf = [&](int l) { return smem + (fwd_only ? 0 : LY::a_off(l, K0P)); };
    auto dz_buf = [&](int l) { return smem + LY::dz_off(l, L, K0P); };
    auto row_ptr = [&](uint8_t *buf, int slab) { return reinterpret_cast<uint4 *>(buf + slab * SLAB + tid * 16); };
    // issue all K-steps of one stage of the MMA program (thread 0 only); the weight gradient accumulates across tiles
    auto issue_stage = [&](int stage_id, uint32_t acc) { issue_steps<FWD>(prog + stage_id, tmem, 0u, 64u, acc); };
    auto commit_and_wait = [&]() {
        if (tid == 0) umma_commit(bar_mma);
        if (FWD) mbar_wait_tight(bar_mma, phase);
        else
            mbar_wait(bar_mma, phase);
        phase ^= 1;
        tc_fence_after();
    };
    auto publish_smem = [&]() { // generic-proxy smem writes -> visible to the tensor core, all threads
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    };

#ifdef LNB_TC_CLK
    long long clk_acc[24] = {0}, clk_t = clock64();
    clk_acc[14] = clk_t - clk_start;
#define CLK(i) do { long long t_ = clock64(); clk_acc[i] += t_ - clk_t; clk_t = t_; } while (0)
#else
#define CLK(i)
#endif
    int *const next_tile_s = reinterpret_cast<int *>(tailp + 32);
    const int smp = tid % S, ray_l = tid / S;            // this thread's sample within its ray (the same in every tile)
    for (int tile = blockIdx.x; tile < p.n_tiles;) {
        const long long row0 = (long long)tile * p.rows_per_tile;
        long long rem = p.N - row0;
        const int valid = rem < p.rows_per_tile ? (int)rem : p.rows_per_tile;
        const int rays_here = valid == p.rows_per_tile ? p.G : valid / S;
        const int ray0 = tile * p.G;      // = row0 / S: a tile holds G whole rays (R is an int)
        CLK(15);
        const bool live = tid < rays_here * S;
        float x[3], my_dist, tg[3], u[3];
        sample_inputs<RAYS, DIRS>(p, row0, ray0, tid, smp, ray_l, live, x, my_dist, tg, u);
        auto store_a0 = [&](int c8, uint4 q) { *row_ptr(a_buf(0), c8) = q; };
        const int a0s = (c_in + 8) >> 3;   // slabs holding features 0..c_in (the ones column included)
        if (RAYS) {
            // ---- features from rays: the positional encoding, written straight into A_0
            float sn[3], cs[3];
            if (!DIRS) {
#pragma unroll
                for (int c = 0; c < 3; ++c) pe_sincos(x[c], &sn[c], &cs[c]);
            }
            if (dw_pending) { mbar_wait(bar_dw, dwphase); dwphase ^= 1; dw_pending = false; tc_fence_after(); }
            CLK(12);
            if (DIRS) pack_pe_dirs(x, u, p.pe_bands, p.dir_bands, store_a0);
            else pack_pe(x, sn, cs, p.pe_bands, a0s, store_a0);
        } else {
            // ---- features: wait for the TMA, convert this thread's row to bf16 slabs
            int lead; uint32_t bytes;
            (void)x_src(p, tile, c_in, lead, bytes);
            mbar_wait(bar_x, xphase);
            xphase ^= 1;
            CLK(0);
            if (dw_pending) { mbar_wait(bar_dw, dwphase); dwphase ^= 1; dw_pending = false; tc_fence_after(); }
            CLK(12);
            pack_features(stage + lead + tid * c_in, c_in, tid < valid, store_a0);
        }
        publish_smem(); // also: every thread is done reading `stage`
        CLK(1);
        if (tid == 0) {
            // claim the next tile now (so its features can be prefetched); CTAs that started late or
            // run slow simply claim fewer tiles
            const int nt = atomicAdd(p.tile_counter, 1) + (int)gridDim.x;
            *next_tile_s = nt;
            if (!RAYS && nt < p.n_tiles) {
                int lead; uint32_t bytes;
                const void *src = x_src(p, nt, c_in, lead, bytes);
                mbar_expect_tx(bar_x, bytes);
                bulk_g2s(smem_u32(stage), src, bytes, bar_x);
            }
        }
        // ---- forward
        float hz[4];
        for (int l = 0; l < L; ++l) {
            if (tid == 0) issue_stage(l, 0u);
            CLK(2);
            commit_and_wait();
            CLK(3);
            const float *bl = bias_s + l * HP;
            if (l < L - 1) {
                uint8_t *an = a_buf(l + 1);
                uint32_t v[HP / 16][16];
#pragma unroll
                for (int c16 = 0; c16 < HP / 16; ++c16) tmem_ld16(tmem + lane_base + c16 * 16, v[c16]);
                tmem_ld_wait();
                // the hidden layers' bias and the all-ones feature of the next layer's input came out of the MMA (see
                // tc_prep_kernel): ReLU + round + pack is one instruction per pair
#pragma unroll
                for (int c16 = 0; c16 < HP / 16; ++c16) {
                    uint32_t o[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = pack_relu_bf16(__uint_as_float(v[c16][2 * j]), __uint_as_float(v[c16][2 * j + 1]));
                    if (FWD) {
                        tmem_st8(tmem + lane_base + (uint32_t)(HP + c16 * 8), o);
                    } else {
                        *row_ptr(an, c16 * 2) = make_uint4(o[0], o[1], o[2], o[3]);
                        *row_ptr(an, c16 * 2 + 1) = make_uint4(o[4], o[5], o[6], o[7]);
                    }
                }
                CLK(4);
                if (FWD) {              // nothing went to shared memory: the activations are in tensor memory
                    tmem_st_wait();
                    tc_fence_before();
                    __syncthreads();
                    tc_fence_after();
                } else
                    publish_smem();
                CLK(5);
            } else {
                uint32_t v[16];
                tmem_ld16(tmem + lane_base, v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 4; ++j) hz[j] = __uint_as_float(v[j]) + bl[j];
            }
        }
        CLK(16);
        // ---- head + loss + adjoint of the head's pre-activation (unit seed)
        float dz[4];
        head_and_composite<!FWD, EXT, RAYS == 2>(p, scratch, 0, hz, my_dist, tg, row0, ray0, valid, tid, smp, ray_l, live, loss_acc, dz);
        CLK(17);
        if (FWD) { __syncthreads(); tile = *next_tile_s; continue; }
        // ---- backward.  dZ_{L-1}: 4 live features, the rest of the 16 stay zero
        *row_ptr(dz_buf(L - 1), 0) = make_uint4(pack_bf16(dz[0], dz[1]), pack_bf16(dz[2], dz[3]), 0u, 0u);
        publish_smem();
        CLK(7);
        for (int l = L - 1; l >= 1; --l) {
            if (tid == 0) issue_stage(L + l, 0u);
            CLK(8);
            commit_and_wait();
            CLK(9);
            uint8_t *al = a_buf(l), *dzn = dz_buf(l - 1);
            uint32_t v[HP / 16][16];
#pragma unroll
            for (int c16 = 0; c16 < HP / 16; ++c16) tmem_ld16(tmem + lane_base + c16 * 16, v[c16]);
            uint4 hm[HP / 8];
#pragma unroll
            for (int c8 = 0; c8 < HP / 8; ++c8) hm[c8] = *row_ptr(al, c8);
            tmem_ld_wait();
            uint4 oz[HP / 8];
            relu_adjoint<HP>(v, hm, oz);
#pragma unroll
            for (int c8 = 0; c8 < HP / 8; ++c8) *row_ptr(dzn, c8) = oz[c8];
            CLK(10);
            publish_smem();
            CLK(11);
        }
        // all dZ_l are in shared memory: the weight-gradient MMAs run in the background; their
        // completion is awaited only before A_0 is overwritten by the next tile (or at the end)
        if (tid == 32) { issue_stage(2 * L, dw_started ? 1u : 0u); umma_commit(bar_dw); } // warp 1 issues; warp 0 moves on
        dw_pending = true;
        CLK(13);
        tile = *next_tile_s; // written before this tile's forward; several block barriers ago
        dw_started = true;
    }

    // ---- epilogue: this CTA's partials.  loss, then per layer the valid (in_l+1) x out_l block.
    if (dw_pending) { mbar_wait(bar_dw, dwphase); dwphase ^= 1; }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    float *part = p.part + (size_t)blockIdx.x * p.part_stride;
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) loss_acc += __shfl_xor_sync(0xffffffffu, loss_acc, d);
    if (lane == 0) red_s[warp] = loss_acc;
    __syncthreads();
    if (tid == 0) part[0] = red_s[0] + red_s[1] + red_s[2] + red_s[3];
    if (tid == 0 && blockIdx.x == 0 && p.t_dev) p.t_dev[0] += 1; // read by the kernels that follow in the stream
    if (!FWD) {
        // accumulator row (TMEM lane) = feature index over the concatenated A buffers; thread tid
        // owns row tid: find the layer whose feature range contains it
        for (int l = 0; l < L; ++l) {
            const int rowbase = LY::a_off(l, K0P) / SLAB * 8;
            const int in_l = p.dims[l], out_l = p.dims[l + 1], Np = LY::np(l, L);
            const int row = tid - rowbase;
            const int colbase = HP + l * HP;
            float *o = part + p.part_off[l];
#pragma unroll
            for (int c16 = 0; c16 < HP / 16; ++c16) {
                if (c16 * 16 >= Np) break;
                uint32_t v[16];
                tmem_ld16(tmem + lane_base + (uint32_t)(colbase + c16 * 16), v);
                tmem_ld_wait();
                if (row >= 0 && row <= in_l) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        int col = c16 * 16 + j;
                        if (col < out_l) o[row * out_l + col] = dw_started ? __uint_as_float(v[j]) : 0.0f;
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, LY::tmem_cols(L, !FWD));
#ifdef LNB_TC_CLK
    clk_acc[13] += clock64() - clk_t; // (issue dW slot reused: epilogue after the last tile)
    unsigned long long gt_end;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt_end));
    if (p.dbg && tid == 0) {
        unsigned long long *tt = reinterpret_cast<unsigned long long *>(p.dbg + (size_t)gridDim.x * 24);
        tt[blockIdx.x * 2] = gt_start; tt[blockIdx.x * 2 + 1] = gt_end;
    }
    if (p.dbg && tid == 0) for (int i = 0; i < 24; ++i) p.dbg[blockIdx.x * 24 + i] = (float)clk_acc[i];
#endif
}

#include "fused_mg.cuh"

struct AdamArgs {
    float *param, *m, *v;
    const int *t_dev;
    double lr, b1, b2, eps;
    uint8_t *wimg;
    long long n_w; // floats in the padded ws block (biases follow)
    int sgd;       // 1: param -= lr * g (fit_img.py:512-513) instead of Adam
};

// the reference's AdamOptimizer.update (train_nerf.py:133-161, double bias correction kept) on
// one parameter; python-float scalars meet float32 arrays exactly as in optim.cu
// the step's scalar factors: Python doubles in the reference (lr_t = lr * sqrt(1 - b2^t) / (1 - b1^t)), rounded to float32
// once where they meet the arrays; computed by ONE thread per block, beside the gather (see tc_reduce_kernel).
struct AdamScalars { float lr_t, c1, c2; };
// beta^t for an integer step count by squaring: ~2 log2(t) dependent double multiplies where pow() is ~1 us of dependent
// arithmetic (it was hidden behind the gather: the step time did not change).  Both are within a few ulps of double; the
// results are rounded to float32.
__device__ __forceinline__ double pow_int(double b, int t)
{
    double r = 1.0;
    for (; t > 0; t >>= 1) {
        if (t & 1) r *= b;
        b *= b;
    }
    return r;
}
__device__ __forceinline__ AdamScalars adam_scalars(const AdamArgs &a)
{
    if (a.sgd) return AdamScalars{0.f, 1.f, 1.f};
    const int t = a.t_dev[0];
    const double c1 = 1.0 - pow_int(a.b1, t), c2 = 1.0 - pow_int(a.b2, t);
    return AdamScalars{(float)(a.lr * (sqrt(c2) / c1)), (float)c1, (float)c2};
}
// p0, m0, v0: the element's parameter and moments, loaded by the caller (early, off the critical path)
__device__ __forceinline__ float adam_one(const AdamArgs &a, long long i, float g, const AdamScalars &sc, float p0, float m0, float v0)
{
    if (a.sgd) {
        const float pn = p0 - (float)a.lr * g;
        a.param[i] = pn;
        return pn;
    }
    const float mi = (float)a.b1 * m0 + (float)(1.0 - a.b1) * g;
    const float vi = (float)a.b2 * v0 + (float)(1.0 - a.b2) * (g * g);
    a.m[i] = mi;
    a.v[i] = vi;
    const float pnew = p0 - sc.lr_t * (mi / sc.c1) / (sqrtf(vi / sc.c2) + (float)a.eps);
    a.param[i] = pnew;
    return pnew;
}

// One-shot all-reduce over NVLink peer memory, fused into the gradient reduction (SURVEY.md 8e:
// 12 KB per step, latency-bound).  Every rank writes its reduced gradient into its own comm buffer
// (double-buffered by step parity), publishes the step number with a system-scope release, waits
// for every peer's flag with system-scope acquires, and sums all ranks' vectors IN RANK ORDER so
// that every rank computes bit-identical totals; the optimiser update follows in the same kernel.
__device__ __forceinline__ void st_release_sys(unsigned *p, unsigned v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// element e0 of a partial's gradient block (the loss before it not counted): layer l, input row k (k == dims[l]: the
// bias), output column j, and its index `off` in the padded ws block (is_w) or bs block
struct PartElem { int l, k, j; bool is_w; long long off; };
__device__ __forceinline__ PartElem part_elem(const TcParams &p, int e0)
{
    int e = e0 + 1, l = 0;
    while (l + 1 < p.L && e >= p.part_off[l + 1]) ++l;
    e -= p.part_off[l];
    const int out_l = p.dims[l + 1], k = e / out_l, j = e % out_l;
    const bool is_w = k < p.dims[l];
    return PartElem{l, k, j, is_w, is_w ? ((long long)l * p.max_in + k) * p.max_out + j : (long long)l * p.max_out + j};
}

// reduce the per-CTA partials in a fixed order; apply the seed; accumulate into (or overwrite) the
// caller's buffers; optionally apply Adam to the parameter and refresh the bf16 weight image
__global__ void __launch_bounds__(1024) tc_reduce_kernel(const float *__restrict__ part, int n_part, int part_stride, TcParams p,
                                 float *__restrict__ d_ws, float *__restrict__ d_bs, float *__restrict__ loss,
                                 float seed_value, int seed_is_loss, int overwrite, int fuse_adam, AdamArgs ad, ImgMap im,
                                 lnb_tc_comm cm)
{
    __shared__ float sloss;
    __shared__ AdamScalars s_adam;
    pdl_wait();      // the fused kernel's partials are complete
    pdl_trigger();   // the next step may start its prologue
    // Three things run side by side, one barrier at the end: warp 31 sums the loss partials (every block itself, same order
    // everywhere, so the seed needs no second pass), one thread of warp 30 derives the Adam scalars (two double-precision
    // pow()), warps 0-29 gather the gradient partials: 32 consecutive elements per block (one coalesced 128 B line per
    // partial), the warps stride over the partials with all their loads in flight, fixed-order combine through shared memory.
    __shared__ float acc[30][33];
    const int el = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int n_el = part_stride - 1;
    const int e_glob = blockIdx.x * 32 + el;
    // the element this thread of warp 0 will update: its parameter and moments are fetched now, under the gather
    const bool mine_el = grp == 0 && e_glob < n_el && d_ws;
    PartElem me{};
    long long m_pi = 0;
    float *m_dst = nullptr;
    float pf_p = 0.0f, pf_m = 0.0f, pf_v = 0.0f, pf_d = 0.0f;
    if (mine_el) {
        me = part_elem(p, e_glob);
        m_dst = (me.is_w ? d_ws : d_bs) + me.off;
        m_pi = me.is_w ? me.off : ad.n_w + me.off;
        if (!overwrite) pf_d = *m_dst;
        if (fuse_adam) { pf_p = ad.param[m_pi]; if (!ad.sgd) { pf_m = ad.m[m_pi]; pf_v = ad.v[m_pi]; } }
    }
    if (grp == 31) {
        float s = 0.0f;
#pragma unroll 5
        for (int i = el; i < n_part; i += 32) s += part[(size_t)i * part_stride];
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        if (el == 0) {
            sloss = s;
            if (blockIdx.x == 0 && loss) loss[0] = s;
            if (blockIdx.x == 0 && p.tile_counter) p.tile_counter[0] = 0; // ready for the next launch
        }
    } else if (grp == 30) {
        if (fuse_adam && el == 0 && d_ws) s_adam = adam_scalars(ad);
    } else if (d_ws) {
        float s = 0.0f;
        if (e_glob < n_el) {
            const float *src = part + 1 + e_glob;
#pragma unroll 5
            for (int i = grp; i < n_part; i += 30) s += src[(size_t)i * part_stride];
        }
        acc[grp][el] = s;
    }
    __syncthreads();
    if (!d_ws) return;
    const float scale = seed_is_loss ? sloss * seed_value : seed_value;
    float g_local = 0.0f, s = 0.0f;
    if (grp == 0) {
#pragma unroll
        for (int w2 = 0; w2 < 30; ++w2) s += acc[w2][el];
        g_local = scale * s;
    }
    float loss_total = sloss;
    if (cm.world > 1) {
        // ---- exchange (low-latency push): every element travels as one 8-byte {value, step} word
        // written straight into each peer's receive slot; the receiver polls its LOCAL slot until the
        // step tag matches -- no fences, no separate flags, one NVLink traversal.  Slots are double-
        // buffered by step parity; ranks cannot drift more than one step apart (each needs every
        // peer's words of step s to finish step s).
        // The words carry UNIT-seed gradients; with seed = loss (train_nerf.py:477) the reference's
        // gradient of the whole batch is (sum of the ranks' losses) x (sum of the ranks' unit-seed
        // gradients), so every block also collects the ranks' losses and scales afterwards.
        // A peer that does not show up within LNB_PEER_TIMEOUT_NS of %globaltimer POISONS the step:
        // the element (and through it the parameter) becomes NaN and the sticky status word is set,
        // which lnb_trainer_step_host / lnb_trainer_read / lnb_trainer_comm_status report as an error.
        __shared__ float s_loss_all;
        const unsigned step = (unsigned)ad.t_dev[0], par = step & 1u;
        const bool mine = grp == 0 && e_glob < n_el;
        const bool loss_thread = threadIdx.x == 32;        // every block reads the losses; block 0 publishes
        if (mine || loss_thread) {
            const int slot = mine ? e_glob : n_el;
            const float val = mine ? (seed_is_loss ? seed_value * s : g_local) : sloss;
            const unsigned long long word = ((unsigned long long)step << 32) | (unsigned long long)__float_as_uint(val);
            const size_t off = ((size_t)par * cm.world + cm.rank) * cm.n_slot + slot;
            if (mine || blockIdx.x == 0)
                for (int r = 0; r < cm.world; ++r)
                    if (r != cm.rank) asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(cm.peer_recv[r] + off), "l"(word) : "memory");
            // poll ALL peers' slots side by side (one L2 round trip per sweep instead of one per peer: at 8 GPUs the serial
            // form cost seven dependent ~0.3 us system-scope loads even when every word had already landed), then add in
            // rank order
            unsigned long long w[8];
            unsigned pending = 0;
            for (int r = 0; r < cm.world; ++r)
                if (r != cm.rank) pending |= 1u << r;
            unsigned long long t0 = 0;
            for (unsigned spins = 0; pending; ++spins) {
#pragma unroll
                for (int r = 0; r < 8; ++r)
                    if (pending >> r & 1u) {
                        const unsigned long long *src = cm.my_recv + ((size_t)par * cm.world + r) * cm.n_slot + slot;
                        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(w[r]) : "l"(src) : "memory");
                    }
#pragma unroll
                for (int r = 0; r < 8; ++r)
                    if ((pending >> r & 1u) && (unsigned)(w[r] >> 32) == step) pending &= ~(1u << r);
                if (pending && (spins & 1023u) == 1023u) {       // a lost peer must not hang the GPU
                    unsigned long long now;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                    if (t0 == 0) t0 = now;
                    else if (now - t0 > cm.timeout_ns) {
                        *cm.status = 1;
#pragma unroll
                        for (int r = 0; r < 8; ++r)
                            if (pending >> r & 1u) w[r] = 0x7FC00000ull;     // NaN: the step is poisoned, not silently partial
                        pending = 0;
                    }
                }
            }
            float tot = 0.0f;
#pragma unroll
            for (int r = 0; r < 8; ++r)
                if (r < cm.world) tot += r == cm.rank ? val : __uint_as_float((unsigned)w[r]);
            if (mine) g_local = tot;
            else { loss_total = tot; s_loss_all = tot; if (blockIdx.x == 0 && loss) loss[0] = tot; }
        }
        if (seed_is_loss) {
            __syncthreads();
            g_local *= s_loss_all;
        }
    }
    (void)loss_total;
    if (mine_el) {
        const float g = overwrite ? g_local : pf_d + g_local;
        *m_dst = g;
        if (fuse_adam) {
            const float pn = adam_one(ad, m_pi, g, s_adam, pf_p, pf_m, pf_v);
            if (ad.wimg) { if (me.is_w) im.put_w(ad.wimg, me.l, me.k, me.j, pn); else im.put_b(ad.wimg, me.l, me.j, pn); }
        }
    }
}

// stand-alone Adam + image refresh over the live (non-padding) parameters, one thread each
__global__ void tc_adam_img_kernel(TcParams p, const float *__restrict__ grad, AdamArgs ad, ImgMap im, int n_el)
{
    const int e0 = blockIdx.x * blockDim.x + threadIdx.x;
    if (e0 >= n_el) return;
    const PartElem me = part_elem(p, e0);
    const long long pi = me.is_w ? me.off : ad.n_w + me.off;
    const float pn = adam_one(ad, pi, grad[pi], adam_scalars(ad), ad.param[pi], ad.sgd ? 0.0f : ad.m[pi], ad.sgd ? 0.0f : ad.v[pi]);
    if (ad.wimg) { if (me.is_w) im.put_w(ad.wimg, me.l, me.k, me.j, pn); else im.put_b(ad.wimg, me.l, me.j, pn); }
}

// the padded widths of the fused kernels for this MLP: HP (hidden width + the ones feature, 16 / 32 / 64) and K0P (input
// width + the ones feature, a multiple of 16).  Returns NULL, or why the MLP does not fit the fused kernels.
const char *tc_pick(const lnb_mlp *mlp, int *HP, int *K0P)
{
    const int L = mlp->n_layers;
    if (L < 2 || L > MAXL) return "needs 2..4 layers";
    int hw = 0;
    for (int l = 1; l < L; ++l) hw = mlp->dims[l] > hw ? mlp->dims[l] : hw;
    *HP = hw + 1 <= 16 ? 16 : (hw + 1 <= 32 ? 32 : (hw + 1 <= 64 ? 64 : 0));
    *K0P = (mlp->dims[0] + 1 + 15) / 16 * 16;
    if (!*HP) return "hidden width + 1 must be <= 64";
    if (*K0P > 64) return "input width + 1 must be <= 64";
    if (mlp->dims[L] > 16) return "more than 16 output channels";
    return nullptr;
}

void fill_layout(TcParams &p, const lnb_mlp *mlp, int K0P)
{
    const int L = mlp->n_layers;
    p.L = L;
    for (int l = 0; l <= L; ++l) p.dims[l] = mlp->dims[l];
    p.max_in = mlp->max_in; p.max_out = mlp->max_out;
    p.K0P = K0P;
    int off = 1;
    for (int l = 0; l < L; ++l) { p.part_off[l] = off; off += (mlp->dims[l] + 1) * mlp->dims[l + 1]; }
    p.part_stride = off;
}

ImgMap img_map(const lnb_mlp *mlp, int HP, int K0P)
{
    ImgMap im{mlp->n_layers, HP, K0P, {}};
    for (int l = 0; l <= mlp->n_layers; ++l) im.dims[l] = mlp->dims[l];
    return im;
}

// f(std::integral_constant<int, HP>()) for a padded hidden width HP of 16, 32 or 64: the kernels and their layouts are
// compiled per width
template <class F>
auto with_hp(int HP, F &&f)
{
    if (HP == 16) return f(std::integral_constant<int, 16>());
    if (HP == 32) return f(std::integral_constant<int, 32>());
    return f(std::integral_constant<int, 64>());
}

} // namespace

// Returns LNB_ERR_UNSUPPORTED when the problem does not fit the fused tensor-core kernel.
int lnb_tc_layout(const lnb_mlp *mlp, int *HP, int *K0P, int *wimg_bytes)
{
    int hp = 0, k0p = 0;
    if (tc_pick(mlp, &hp, &k0p)) return 0;
    if (HP) *HP = hp;
    if (K0P) *K0P = k0p;
    if (wimg_bytes) *wimg_bytes = img_map(mlp, hp, k0p).bytes();
    return 1;
}

int lnb_tc_prep(lnb_ctx *ctx, const lnb_mlp *mlp, const float *ws, const float *bs, void *wimg)
{
    int HP = 0, K0P = 0;
    if (tc_pick(mlp, &HP, &K0P)) { ctx->err = "fused tensor-core path: MLP shape not supported"; return LNB_ERR_UNSUPPORTED; }
    TcParams p{};
    fill_layout(p, mlp, K0P);
    p.ws = ws; p.bs = bs;
    tc_prep_kernel<<<1, 256, 0, ctx->stream>>>(p, img_map(mlp, HP, K0P), (uint8_t *)wimg);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_tc_adam_img(lnb_ctx *ctx, const lnb_mlp *mlp, float *param, const float *grad, float *m, float *v,
                    const int *t_dev, double lr, double b1, double b2, double eps, void *wimg)
{
    int HP = 0, K0P = 0;
    if (tc_pick(mlp, &HP, &K0P)) { ctx->err = "fused tensor-core path: MLP shape not supported"; return LNB_ERR_UNSUPPORTED; }
    TcParams p{};
    fill_layout(p, mlp, K0P);
    AdamArgs ad{param, m, v, t_dev, lr, b1, b2, eps, (uint8_t *)wimg, (long long)mlp->n_layers * mlp->max_in * mlp->max_out, m == nullptr};
    const int n_el = p.part_stride - 1;
    tc_adam_img_kernel<<<(n_el + 255) / 256, 256, 0, ctx->stream>>>(p, grad, ad, img_map(mlp, HP, K0P), n_el);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_fused_tc_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, const lnb_tc_extra *ex,
                      const lnb_comp_args *cx)
{
    const int L = mlp->n_layers;
    auto unsupported = [&](const char *why) {
        ctx->err = std::string("fused tensor-core path: ") + why;
        return LNB_ERR_UNSUPPORTED;
    };
    int HP = 0, K0P = 0;
    if (const char *why = tc_pick(mlp, &HP, &K0P)) return unsupported(why);
    if (a->inter || a->rgba || a->alpha || a->cumprod || a->weights || a->d_X || a->d_target || a->d_dists ||
        a->d_color || a->d_inter)
        return unsupported("only loss, colour, d_ws and d_bs are produced (use the fp32 path for the rest)");
    if (a->color && a->color_accumulate) return unsupported("colour accumulation");
    const int R = a->R, S = nerf ? a->S : 1;
    const long long N = a->n_rows > 0 ? a->n_rows : (long long)R * S;
    if (nerf && (S > TILE || N != (long long)R * S)) return unsupported("needs S <= 128 and n_rows == R*S");
    const bool cam = a->X == nullptr && a->rays_o == nullptr && a->cam != nullptr;
    const bool rays = a->X == nullptr && (a->rays_o != nullptr || cam);
    const int dir_bands = rays ? lnb_rays_dir_bands(mlp->dims[0], a->pe_bands) : LNB_DIRS_NONE;
    if (rays && (!nerf || (!cam && (!a->rays_d || !a->t)) || dir_bands == LNB_DIRS_BAD))
        return unsupported("rays mode needs rays_o, rays_d, t (or a camera) and dims[0] == 3 + 6 * pe_bands (+ 3 + 6 * E_dir)");
    const bool dirs = dir_bands >= 0;
    if (cam && (long long)a->cam->width * a->cam->height >= (1ll << 31)) return unsupported("camera: more than 2^31 pixels");
    const lnb_views *views = cam ? lnb_cx_views(cx) : nullptr;   // views mode: the RAYS == 2 instantiations
    if (!nerf && N != R) return unsupported("needs n_rows == R");
    if (a->rows > N) return unsupported("rows > n_rows");
    if (!nerf && (a->target_w > 4)) return unsupported("target wider than 4");
    if (a->want_grad && !a->target && N > 0) return unsupported("gradient without target");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;

    TcParams p{};
    fill_layout(p, mlp, K0P);
    p.X = a->X; p.dists = a->dists; p.target = a->target; p.ws = a->ws; p.bs = a->bs;
    p.rays_o = a->rays_o; p.rays_d = a->rays_d; p.tvals = a->t; p.ray_f64 = a->ray_dtype == LNB_RAY_F64; p.pe_bands = a->pe_bands;
    p.dir_bands = dirs ? dir_bands : 0;
    if (cam) {
        const lnb_camera &c = *a->cam;
        p.cam_mode = 1;
        for (int i = 0; i < 12; ++i) p.cam.c2w[i] = (float)c.c2w[i];
        p.cam.inv_fx = (float)(1.0 / c.fx); p.cam.inv_fy = (float)(1.0 / c.fy); p.cam.cx = (float)c.cx; p.cam.cy = (float)c.cy;
        p.cam.step = (float)(1.0 / (double)(c.width - 1)); p.cam.near = (float)c.near; p.cam.far = (float)c.far;
        p.cam.dt_lin = (float)((c.far - c.near) / (double)(a->S > 1 ? a->S - 1 : 1)); p.cam.dt_str = (float)((c.far - c.near) / (double)a->S);
        p.cam.first_pixel = c.first_pixel; p.cam.pixels = c.pixels; p.cam.seed = c.seed; p.cam.width = c.width; p.cam.stratified = c.stratified;
        p.cam.w_magic = c.width >= 2 ? ~0ull / (unsigned long long)c.width + 1ull : 0ull;
        if (views) {
            p.cam.poses = views->poses; p.cam.view = views->view; p.cam.seed_dev = views->seed_dev;
            p.cam.P = (long long)views->width * views->height; p.cam.n_views = views->n_views;
        }
    }
    p.color = nerf ? a->color : nullptr;
    p.N = N; p.R = R; p.S = S;
    p.G = nerf ? TILE / S : TILE;
    p.rows_per_tile = p.G * S;
    p.n_tiles = (int)((N + p.rows_per_tile - 1) / p.rows_per_tile);
    p.head = mlp->head; p.want_grad = a->want_grad; p.Wt = a->target_w > 0 ? a->target_w : 3;

    const int c_in = mlp->dims[0];
    const bool grad = a->want_grad != 0;
    if (!rays && (reinterpret_cast<uintptr_t>(a->X) & 3) != 0) return unsupported("X must be 4-byte aligned");
    // Train steps run on the multi-group kernel (fused_mg.cuh: one CTA per SM, up to seven 128-thread groups, adjoints in
    // place); forward-only launches and LNB_TC_V1=1 on the one-tile-per-CTA kernel above.
    const bool mg = grad && getenv("LNB_TC_V1") == nullptr && (!nerf || S >= 2);
    // the extras instantiations: lnb_trainer_step_weights, and any step with compositing extras (lnb_composite)
    const bool ext = nerf && ((grad && ex && ex->weights) || lnb_cx_extras(cx));
    if (views && grad && !mg) return unsupported("views mode trains on the multi-group kernel (S >= 2, LNB_TC_V1 unset)");
    if (grad && !mg) {   // the one-tile-per-CTA kernel computes all weight gradients with ONE concatenated M = 128 MMA per K-step
        if (K0P / 8 + (L - 1) * (HP / 8) > 16) return unsupported("input + hidden widths exceed 128 features in total");
        if ((L - 1) * HP + 16 > 256) return unsupported("hidden widths exceed 256 gradient columns");
    }
    const int in_kind = views ? (dirs ? 4 : 3) : (dirs ? 2 : (rays ? 1 : 0));   // the input form, as mg_regs lists them
    void (*const kern)(TcParams) = with_hp(HP, [&](auto hp) -> void (*)(TcParams) {
        constexpr int H = decltype(hp)::value;
        if (views) {
            if (mg && ext) return dirs ? fused_mg_kernel<2, H, true, true> : fused_mg_kernel<2, H, false, true>;
            if (mg) return dirs ? fused_mg_kernel<2, H, true> : fused_mg_kernel<2, H>;
            if (ext) return dirs ? fused_v1_kernel<2, H, true, true, true> : fused_v1_kernel<2, H, true, false, true>;
            return dirs ? fused_v1_kernel<2, H, true, true> : fused_v1_kernel<2, H, true>;
        }
        if (mg && ext) return dirs ? fused_mg_kernel<true, H, true, true> : rays ? fused_mg_kernel<true, H, false, true> : fused_mg_kernel<false, H, false, true>;
        if (mg) return dirs ? fused_mg_kernel<true, H, true> : rays ? fused_mg_kernel<true, H> : fused_mg_kernel<false, H>;
        if (grad && ext)
            return dirs ? fused_v1_kernel<true, H, false, true, true> : rays ? fused_v1_kernel<true, H, false, false, true> : fused_v1_kernel<false, H, false, false, true>;
        if (grad) return dirs ? fused_v1_kernel<true, H, false, true> : rays ? fused_v1_kernel<true, H, false> : fused_v1_kernel<false, H, false>;
        if (ext)
            return dirs ? fused_v1_kernel<true, H, true, true, true> : rays ? fused_v1_kernel<true, H, true, false, true> : fused_v1_kernel<false, H, true, false, true>;
        return dirs ? fused_v1_kernel<true, H, true, true> : rays ? fused_v1_kernel<true, H, true> : fused_v1_kernel<false, H, true>;
    });
    size_t smem = 0;
    int grid = 0, ng = 1;
    if (mg) {
        ng = with_hp(HP, [&](auto hp) {
            using MG = MgLayout<decltype(hp)::value>;
            int n = mg_max_groups<decltype(hp)::value>();
            while (n > 1 && (MG::total(L, c_in, K0P, rays, n) > 232448 || MG::tmem_need(L, K0P, n) > 512)) --n;
            return n;
        });
        // registers per thread of each instantiation ([extras] (features, rays, rays + directions, views, views + directions)),
        // asked once
        static int mg_regs[2][5][3] = {};
        int &regs = mg_regs[ext][in_kind][HP / 32];
        if (regs == 0) {
            cudaFuncAttributes fa;
            LNB_CUDA(cudaFuncGetAttributes(&fa, kern));
            regs = fa.numRegs;
        }
        while (ng > 1 && (long long)ng * TILE * ((regs + 7) / 8 * 8) > 65536) --ng;
        if (const char *e = getenv("LNB_TC_GROUPS")) { const int v = atoi(e); if (v >= 1 && v < ng) ng = v; }
        const int per_sm = (p.n_tiles + ctx->sm_count - 1) / ctx->sm_count;   // small batches: no idle groups
        if (ng > per_sm) ng = per_sm < 1 ? 1 : per_sm;
        grid = (p.n_tiles + ng - 1) / ng;
        if (grid > ctx->sm_count) grid = ctx->sm_count;
        if (grid < 1) grid = 1;
        smem = with_hp(HP, [&](auto hp) { return MgLayout<decltype(hp)::value>::total(L, c_in, K0P, rays, ng); });
        if (smem > 232448) return unsupported("shared memory");
    } else {
        int tmem_cols = 0;
        with_hp(HP, [&](auto hp) {
            using LY = TcLayout<decltype(hp)::value>;
            smem = LY::total(L, K0P, c_in, rays, grad);
            tmem_cols = (int)LY::tmem_cols(L, grad);
        });
        int per_sm = 512 / tmem_cols;
        int by_smem = (int)((228 * 1024) / (smem + 1024));
        if (by_smem < per_sm) per_sm = by_smem;
        if (per_sm < 1) return unsupported("shared memory");
        if (const char *e = getenv("LNB_TC_CTAS_PER_SM")) { int v = atoi(e); if (v >= 1 && v < per_sm) per_sm = v; }
        grid = ctx->sm_count * per_sm;
        if (grid > p.n_tiles) grid = p.n_tiles;
        if (grid < 1) grid = 1;
    }
    const ImgMap im = img_map(mlp, HP, K0P);
    const int wimg_bytes = im.bytes();
    LNB_TRY(lnb_arena_reserve(ctx, (size_t)grid * p.part_stride * sizeof(float) + wimg_bytes + 8192));
    p.part = (float *)lnb_arena_take(ctx, (size_t)grid * p.part_stride * sizeof(float));
    uint8_t *wimg = (uint8_t *)lnb_arena_take(ctx, wimg_bytes);
    p.wimg = (ex && ex->wimg) ? ex->wimg : wimg;
    p.t_dev = ex ? ex->t_dev : nullptr;
    p.weights = (ext && ex) ? ex->weights : nullptr;
    if (cx) {
        p.acc = cx->acc; p.depth = cx->depth; p.background = cx->background;
        for (int c = 0; c < 3; ++c) p.bg[c] = cx->bg[c];
    }
    if (!ctx->tc_counter) {
        LNB_CUDA(cudaMalloc((void **)&ctx->tc_counter, 256));
        LNB_CUDA(cudaMemsetAsync(ctx->tc_counter, 0, 256, ctx->stream));
    }
    p.tile_counter = ctx->tc_counter;
    float *loss = a->loss ? a->loss : (float *)lnb_arena_take(ctx, 16);
#ifdef LNB_TC_CLK
    float *dbg_dev = nullptr;
    cudaMalloc(&dbg_dev, (size_t)grid * 28 * sizeof(float) * 8);
    cudaMemset(dbg_dev, 0, (size_t)grid * 28 * sizeof(float) * 8);
    p.dbg = dbg_dev;
#endif
    cudaLaunchAttribute pdl_attr[1];
    pdl_attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl_attr[0].val.programmaticStreamSerializationAllowed = 1;
    const bool use_pdl = getenv("LNB_NO_PDL") == nullptr;
    if (N > 0) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(mg ? ng * TILE : TILE); cfg.dynamicSmemBytes = smem; cfg.stream = ctx->stream;
        cfg.attrs = pdl_attr; cfg.numAttrs = use_pdl ? 1 : 0;
        if (!(ex && ex->wimg)) {
            tc_prep_kernel<<<1, 256, 0, ctx->stream>>>(p, im, wimg);
            LNB_CHECK_LAUNCH();
        }
        // the dynamic shared-memory limit of each kernel instantiation (kind, input, HP) on each device: raised only when it grows
        static size_t smem_set[2][3][5][3][64] = {};
        size_t &lim = smem_set[ext][mg ? 0 : (grad ? 1 : 2)][in_kind][HP / 32][ctx->device & 63];
        if (smem > lim || ctx->device > 63) { LNB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); lim = smem; }
        // the symbols ncu lists; "+extras": an extras instantiation (weights / acc / depth / background)
        static const char *const names[2][2][3] = {{{"fused_v1_kernel<features>", "fused_v1_kernel<rays>", "fused_v1_kernel<views>"},
                                                    {"fused_mg_kernel<features>", "fused_mg_kernel<rays>", "fused_mg_kernel<views>"}},
                                                   {{"fused_v1_kernel<features>+extras", "fused_v1_kernel<rays>+extras", "fused_v1_kernel<views>+extras"},
                                                    {"fused_mg_kernel<features>+extras", "fused_mg_kernel<rays>+extras", "fused_mg_kernel<views>+extras"}}};
        lnb_prof_begin(ctx, names[ext][mg][views ? 2 : rays]);
        LNB_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
        lnb_prof_end(ctx);
        LNB_CHECK_LAUNCH();
    } else {
        grid = 0;
        if (p.t_dev) LNB_TRY(lnb_launch_incr(ctx, p.t_dev)); // an empty shard still takes the step (and publishes zeros)
    }
#ifdef LNB_TC_CLK
    {
        cudaStreamSynchronize(ctx->stream);
        std::vector<float> h((size_t)grid * 28);
        if (!mg) {
            cudaMemcpy(h.data(), dbg_dev, h.size() * sizeof(float), cudaMemcpyDeviceToHost);
            cudaFree(dbg_dev);
        }
        static int calls = 0;
        if (mg) {
            std::vector<unsigned long long> hs((size_t)grid * ng * 8);
            cudaMemcpy(hs.data(), dbg_dev, hs.size() * 8, cudaMemcpyDeviceToHost);
            cudaFree(dbg_dev);
            if (++calls % 50 == 20) {
                unsigned long long t0 = ~0ull;
                for (size_t i = 0; i < hs.size(); i += 8) t0 = hs[i] < t0 ? hs[i] : t0;
                const char *nm[8] = {"CTA start", "prologue done", "weights landed", "first tile done", "last tile done", "all groups done", "end", "partials written"};
                fprintf(stderr, "[mg clk] grid %d x %d groups, %d tiles: us from the first CTA start (min / mean / max over groups that have the stamp)\n", grid, ng, p.n_tiles);
                for (int k = 0; k < 8; ++k) {
                    double mn = 1e30, mx = 0, sum = 0; int n = 0;
                    for (size_t i = 0; i < hs.size(); i += 8) if (hs[i + k]) { const double v = (hs[i + k] - t0) * 1e-3; mn = v < mn ? v : mn; mx = v > mx ? v : mx; sum += v; ++n; }
                    if (n) fprintf(stderr, "   %-16s %7.2f %7.2f %7.2f   (%d)\n", nm[k], mn, sum / n, mx, n);
                }
            }
        } else if (++calls % 150 == 20) {
            double acc[24] = {0};
            for (int b = 0; b < grid; ++b) for (int i = 0; i < 24; ++i) acc[i] += h[(size_t)b * 24 + i];
            const char *nm[24] = {"wait X", "convert+publish", "issue fwd", "wait fwd mma", "fwd epilogue", "fwd publish", "", "dz publish",
                                  "issue bwd", "wait bwd mma", "bwd epilogue", "bwd publish", "wait dW", "issue dW + final epilogue", "prologue", "loop top",
                                  "head ld+bias", "compositing", "", "", "", "", "", ""};
            double tot = 0; for (int i = 0; i < 24; ++i) tot += acc[i];
            fprintf(stderr, "[tc clk] grid %d tiles %d: cycles per tile (thread 0), total %.0f\n", grid, p.n_tiles, tot / p.n_tiles);
            {
                const unsigned long long *tt = reinterpret_cast<const unsigned long long *>(h.data() + (size_t)grid * 24);
                unsigned long long s0 = ~0ull, s1 = 0, e0 = ~0ull, e1 = 0;
                for (int b = 0; b < grid; ++b) {
                    s0 = tt[2 * b] < s0 ? tt[2 * b] : s0; s1 = tt[2 * b] > s1 ? tt[2 * b] : s1;
                    e0 = tt[2 * b + 1] < e0 ? tt[2 * b + 1] : e0; e1 = tt[2 * b + 1] > e1 ? tt[2 * b + 1] : e1;
                }
                fprintf(stderr, "   CTA start spread %.1f us, first end at %.1f us, last end at %.1f us (from first start)\n",
                        (s1 - s0) * 1e-3, (e0 - s0) * 1e-3, (e1 - s0) * 1e-3);
            }
            for (int i = 0; i < 24; ++i) if (acc[i] > 0) fprintf(stderr, "   %-22s %8.0f\n", nm[i], acc[i] / p.n_tiles);
        }
    }
#endif
    const int n_el = p.part_stride - 1;
    const int seed_is_loss = a->seed_mode == LNB_SEED_LOSS;
    const float seed_val = seed_is_loss ? 1.0f : a->seed;
    int blocks = a->want_grad ? (n_el + 31) / 32 : 1;
    AdamArgs ad{};
    const int fuse = ex && ex->fuse_adam && a->want_grad;
    if (fuse) ad = AdamArgs{ex->param, ex->m, ex->v, ex->t_dev, ex->lr, ex->b1, ex->b2, ex->eps, (uint8_t *)ex->wimg_out,
                            (long long)L * mlp->max_in * mlp->max_out, ex->m == nullptr};
    {
        cudaLaunchConfig_t rc{};
        rc.gridDim = dim3((unsigned)blocks); rc.blockDim = dim3(1024); rc.dynamicSmemBytes = 0; rc.stream = ctx->stream;
        rc.attrs = pdl_attr; rc.numAttrs = use_pdl ? 1 : 0;
        const lnb_tc_comm comm_arg = (ex && ex->comm && fuse) ? *ex->comm : lnb_tc_comm{};
        LNB_CUDA(cudaLaunchKernelEx(&rc, tc_reduce_kernel, (const float *)p.part, grid, p.part_stride, p,
                                    a->want_grad ? a->d_ws : (float *)nullptr, a->want_grad ? a->d_bs : (float *)nullptr, loss,
                                    seed_val, seed_is_loss, ex ? ex->overwrite_grads : 0, fuse, ad, im, comm_arg));
    }
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}
