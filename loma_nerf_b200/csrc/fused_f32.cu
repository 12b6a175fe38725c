// fused_f32.cu -- the fused EXACT step: IEEE fp32 on the CUDA cores, one kernel from features to weight gradients.
//
// LNB_PATH_F32 for the reference's own network shapes (2 or 3 layers, input width <= 35, hidden width <= 31, <= 4 outputs:
// 33 -> 30 -> 30 -> 4 of train_nerf.py, 22 -> 16 -> 16 -> 3 of fit_img.py) when only loss, colour, d_ws and d_bs are asked
// for.  Everything else (intermediates, d_layer_input, wider / deeper networks) stays on the layerwise kernels of
// kernels_f32.cu, which materialise every array the compat ABI hands back; both are held to <= 1e-5 of the reference.
//
// Per 128-sample tile of a persistent CTA (128 threads, static tile -> CTA assignment, so results are reproducible bit
// for bit):
//   features -> shared memory A_0 [128][36] (row stride 36 floats: 16-byte accesses of consecutive rows fall into
//     distinct banks), an all-ones column at c_in (its weight-gradient row is the bias gradient)
//   hidden layers: register-tiled GEMM, thread = 4 samples x 8 outputs, k in ascending order like the reference's
//     loops (scripts/nerf.py:67-146); 3 shared-memory loads (one activation quad, two weight quads) per 32 FMAs
//   head + compositing with one thread per sample: warp-shuffle product / sum / affine-suffix scans (nerf.py:176-288
//     and its reverse), accurate expf
//   backward per layer, while A_l and dZ_l are both in shared memory:
//     dW_l += A_l^T dZ_l   -- each warp contracts its own 32 samples into 32 + 4 register accumulators per thread that
//                             live across ALL tiles of the CTA (north_star item 4: one write per CTA at the end)
//     dZ_{l-1} = relu'(A_l) . (dZ_l W_l^T), written in place of A_l
//   one partial [loss | dW_0 | db_0 | ...] per CTA; fused_f32_reduce_kernel sums the partials in a fixed order, applies
//   the seed (SURVEY.md 8 a7: gradients are linear in _dreturn) and accumulates into d_ws / d_bs.
// The weights (and W^T for the adjoint GEMMs) sit in shared memory for the CTA's lifetime: 72 KB per CTA, three per SM.
#include <stdlib.h>

#include "lnb_internal.h"

namespace {

constexpr int FT = 128;   // samples per tile = threads per CTA
constexpr int LD = 36;    // activation row stride in floats
constexpr int HW = 32;    // padded hidden width (hidden + ones column <= 32)
constexpr int K0 = 36;    // padded input width (c_in + ones column <= 36)

struct F32Params {
    const float *X, *dists, *target, *ws, *bs;
    float *color;     // [R][3] or NULL
    float *part;      // [grid][part_stride]
    long long N;
    int R, S, rows_per_tile, n_tiles;
    int L, dims[4], max_in, max_out, head, want_grad, Wt;
    int part_stride, part_off[3];
    int x_vec4;               // every tile of X starts on a 16-byte boundary
    unsigned c_in_magic;      // ceil(2^32 / c_in)
};

__device__ __forceinline__ float sigmoid_exact(float z) { return 1.0f / (1.0f + expf(0.0f - z)); }
__device__ __forceinline__ float comp(const float4 &v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : (k == 2 ? v.z : v.w)); }

// Two IEEE fp32 FMAs per instruction (SASS FFMA2; the scalar operand is broadcast by the instruction itself): the same
// roundings as two fmaf, half the issue slots -- the kernel is issue-bound, not FMA-pipe-bound.
__device__ __forceinline__ void fma2(float &c0, float &c1, float a, float b0, float b1)
{
    const float2 r = __ffma2_rn(make_float2(a, a), make_float2(b0, b1), make_float2(c0, c1));
    c0 = r.x; c1 = r.y;
}

// acc[s][j] += sum_k A[row_s][k] * W[k][8 warp + j], rows row_s = lane + 32 s, k ascending
template <int KP>
__device__ __forceinline__ void gemm_4x8(const float *__restrict__ A, const float *__restrict__ W, int warp, int lane, float (&acc)[4][8])
{
#pragma unroll 3
    for (int k4 = 0; k4 < KP; k4 += 4) {
        float4 a[4];
#pragma unroll
        for (int s = 0; s < 4; ++s) a[s] = *reinterpret_cast<const float4 *>(A + (lane + 32 * s) * LD + k4);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const float4 w0 = *reinterpret_cast<const float4 *>(W + (k4 + kk) * HW + 8 * warp);
            const float4 w1 = *reinterpret_cast<const float4 *>(W + (k4 + kk) * HW + 8 * warp + 4);
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const float av = comp(a[s], kk);
                fma2(acc[s][0], acc[s][1], av, w0.x, w0.y); fma2(acc[s][2], acc[s][3], av, w0.z, w0.w);
                fma2(acc[s][4], acc[s][5], av, w1.x, w1.y); fma2(acc[s][6], acc[s][7], av, w1.z, w1.w);
            }
        }
    }
}

// dZ_{l-1} = relu'(A) . acc, in place of A (columns >= width, i.e. the ones column and the padding, become 0)
__device__ __forceinline__ void store_masked(float *A, int warp, int lane, const float (&acc)[4][8])
{
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        float *row = A + (lane + 32 * s) * LD + 8 * warp;
        const float4 m0 = *reinterpret_cast<const float4 *>(row), m1 = *reinterpret_cast<const float4 *>(row + 4);
        *reinterpret_cast<float4 *>(row) = make_float4(m0.x > 0.f ? acc[s][0] : 0.f, m0.y > 0.f ? acc[s][1] : 0.f,
                                                       m0.z > 0.f ? acc[s][2] : 0.f, m0.w > 0.f ? acc[s][3] : 0.f);
        *reinterpret_cast<float4 *>(row + 4) = make_float4(m1.x > 0.f ? acc[s][4] : 0.f, m1.y > 0.f ? acc[s][5] : 0.f,
                                                           m1.z > 0.f ? acc[s][6] : 0.f, m1.w > 0.f ? acc[s][7] : 0.f);
    }
}

// this warp's 32 samples: g[i][j] += A[s][8 gi + i] * D[s][4 gj + j]   (lane = 8 gi + gj)
__device__ __forceinline__ void dw_8x4(const float *__restrict__ A, const float *__restrict__ D, int ldd, int warp, int lane, float (&g)[8][4])
{
    const int gi = lane >> 3, gj = lane & 7;
#pragma unroll 2
    for (int s = 32 * warp; s < 32 * warp + 32; ++s) {
        const float4 a0 = *reinterpret_cast<const float4 *>(A + s * LD + 8 * gi), a1 = *reinterpret_cast<const float4 *>(A + s * LD + 8 * gi + 4);
        const float4 d = *reinterpret_cast<const float4 *>(D + s * ldd + 4 * gj);
        const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) { fma2(g[i][0], g[i][1], av[i], d.x, d.y); fma2(g[i][2], g[i][3], av[i], d.z, d.w); }
    }
}

__global__ void __launch_bounds__(FT, 3) fused_f32_kernel(const F32Params p)
{
    extern __shared__ __align__(16) float sm[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int L = p.L, c_in = p.dims[0], S = p.S, out_last = p.dims[L];
    const bool three = L == 3;
    // ---- shared memory
    float *A0 = sm, *A1 = A0 + FT * LD, *A2 = A1 + FT * LD;            // A2 only when L == 3
    float *Zh = three ? A2 + FT * LD : A2;                              // [128][4] head pre-activation adjoints
    float *W0 = Zh + FT * 4;                                            // [36][32]
    float *W1 = W0 + K0 * HW;                                           // [32][32]  (L == 3)
    float *Wl = three ? W1 + HW * HW : W1;                              // [32][4]   last layer
    float *WT1 = Wl + HW * 4;                                           // [32][32]  W_1^T (L == 3)
    float *WTl = three ? WT1 + HW * HW : WT1;                           // [4][32]   last layer, transposed
    float *bias = WTl + 4 * HW;                                         // [3][32]
    float *scr = bias + 3 * HW;                                         // compositing scratch
    float *color_s = scr, *tgt_s = scr + 192, *tailp = scr + 384;
    int *tail_s = reinterpret_cast<int *>(tailp + 4);
    float *headq = tailp + 8, *headA = tailp + 13, *headB = tailp + 18, *red_s = tailp + 24;
    float *const Alast = three ? A2 : A1;                               // input of the last layer
    const int h0 = p.dims[1], h1 = three ? p.dims[2] : 0;

    // ---- weights into shared memory, zero padded (padding rows / columns must be exact zeros)
    for (int e = tid; e < K0 * HW; e += FT) { const int k = e / HW, j = e % HW; W0[e] = (k < c_in && j < h0) ? __ldg(p.ws + (size_t)k * p.max_out + j) : 0.0f; }
    if (three)
        for (int e = tid; e < HW * HW; e += FT) {
            const int k = e / HW, j = e % HW;
            const float v = (k < h0 && j < h1) ? __ldg(p.ws + ((size_t)p.max_in + k) * p.max_out + j) : 0.0f;
            W1[e] = v; WT1[j * HW + k] = v;
        }
    {
        const int hin = three ? h1 : h0;
        const float *wl = p.ws + (size_t)(L - 1) * p.max_in * p.max_out;
        for (int e = tid; e < HW * 4; e += FT) {
            const int k = e / 4, j = e % 4;
            const float v = (k < hin && j < out_last) ? __ldg(wl + (size_t)k * p.max_out + j) : 0.0f;
            Wl[e] = v; WTl[j * HW + k] = v;
        }
    }
    for (int e = tid; e < 3 * HW; e += FT) { const int l = e / HW, j = e % HW; bias[e] = (l < L && j < p.dims[l + 1]) ? __ldg(p.bs + (size_t)l * p.max_out + j) : 0.0f; }
    __syncthreads();

    // weight-gradient accumulators of this thread (its warp's samples of every tile of this CTA)
    float g0[8][4] = {}, g0x[4] = {}, g1[8][4] = {}, gl[4] = {};
    float loss_acc = 0.0f;

    for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const long long row0 = (long long)tile * p.rows_per_tile;
        const long long rem = p.N - row0;
        const int valid = rem < p.rows_per_tile ? (int)rem : p.rows_per_tile;
        const int rays_here = valid / S;
        const int smp = tid % S, ray_l = tid / S;
        const bool live = tid < rays_here * S;
        float my_dist = 0.0f, tg0 = 0.0f, tg1 = 0.0f, tg2 = 0.0f;
        if (p.head == LNB_HEAD_NERF && live) {
            my_dist = __ldg(p.dists + row0 + tid);
            if (p.target && smp == 0) {
                const float *tg = p.target + (row0 / S + ray_l) * 3;
                tg0 = __ldg(tg); tg1 = __ldg(tg + 1); tg2 = __ldg(tg + 2);
            }
        }
        // ---- features: the tile is valid * c_in contiguous floats; coalesced 16-byte loads (all issued before the first use),
        // scattered into the padded rows.  e / c_in by multiply-high (exact for e < 2^16).
        {
            const float *src = p.X + row0 * c_in;
            const int n_el = valid * c_in;
            if (p.x_vec4) {
                float4 v[9];
#pragma unroll
                for (int i = 0; i < 9; ++i) {
                    const int e = 4 * (tid + FT * i);
                    v[i] = e + 3 < n_el ? __ldg(reinterpret_cast<const float4 *>(src + e))
                                        : make_float4(e < n_el ? __ldg(src + e) : 0.f, e + 1 < n_el ? __ldg(src + e + 1) : 0.f, e + 2 < n_el ? __ldg(src + e + 2) : 0.f, 0.f);
                }
#pragma unroll
                for (int i = 0; i < 9; ++i) {
                    const int e = 4 * (tid + FT * i);
                    if (e < FT * c_in) {
                        int row = (int)__umulhi((unsigned)e, p.c_in_magic), col = e - row * c_in;
                        const float f[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            if (e + j < FT * c_in) A0[row * LD + col] = f[j];
                            if (++col == c_in) { col = 0; ++row; }
                        }
                    }
                }
            } else {
                int row = tid / c_in, col = tid % c_in;
                const int drow = FT / c_in, dcol = FT % c_in;
                for (int e = tid; e < FT * c_in; e += FT) {
                    A0[row * LD + col] = e < n_el ? __ldg(src + e) : 0.0f;
                    row += drow; col += dcol;
                    if (col >= c_in) { col -= c_in; ++row; }
                }
            }
            for (int c = c_in; c < K0; ++c) A0[tid * LD + c] = (c == c_in && tid < valid) ? 1.0f : 0.0f;
        }
        __syncthreads();
        // ---- hidden layers
        {
            float acc[4][8] = {};
            gemm_4x8<K0>(A0, W0, warp, lane, acc);
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                float v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) { const int c = 8 * warp + j; const float z = acc[s][j] + bias[c]; v[j] = c < h0 ? fmaxf(z, 0.0f) : (c == h0 ? 1.0f : 0.0f); }
                float *row = A1 + (lane + 32 * s) * LD + 8 * warp;
                *reinterpret_cast<float4 *>(row) = make_float4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<float4 *>(row + 4) = make_float4(v[4], v[5], v[6], v[7]);
            }
        }
        __syncthreads();
        if (three) {
            float acc[4][8] = {};
            gemm_4x8<HW>(A1, W1, warp, lane, acc);
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                float v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) { const int c = 8 * warp + j; const float z = acc[s][j] + bias[HW + c]; v[j] = c < h1 ? fmaxf(z, 0.0f) : (c == h1 ? 1.0f : 0.0f); }
                float *row = A2 + (lane + 32 * s) * LD + 8 * warp;
                *reinterpret_cast<float4 *>(row) = make_float4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<float4 *>(row + 4) = make_float4(v[4], v[5], v[6], v[7]);
            }
            __syncthreads();
        }
        // ---- last layer: thread = sample
        float hz[4] = {0.f, 0.f, 0.f, 0.f};
        {
            const float *row = Alast + tid * LD;
#pragma unroll 2
            for (int k4 = 0; k4 < HW; k4 += 4) {
                const float4 a = *reinterpret_cast<const float4 *>(row + k4);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const float4 w = *reinterpret_cast<const float4 *>(Wl + (k4 + kk) * 4);
                    const float av = comp(a, kk);
                    fma2(hz[0], hz[1], av, w.x, w.y); fma2(hz[2], hz[3], av, w.z, w.w);
                }
            }
            const float *bl = bias + (L - 1) * HW;
#pragma unroll
            for (int j = 0; j < 4; ++j) hz[j] += bl[j];
        }
        // ---- head + loss + adjoint of the head's pre-activation (unit seed)
        float dz[4] = {0.f, 0.f, 0.f, 0.f};
        if (p.head == LNB_HEAD_SIGMOID) {
            // mlp_fit: row r <-> target row (scripts/mlp_fit.py:121-145)
            if (tid < valid && row0 + tid < p.R && p.target) {
                const float *tg = p.target + (row0 + tid) * p.Wt;
                for (int c = 0; c < p.Wt && c < 4; ++c) {
                    const float y = sigmoid_exact(hz[c]);
                    const float d = y - __ldg(tg + c);
                    loss_acc = fmaf(d, d, loss_acc);
                    dz[c] = (2.0f * d) * (y * (1.0f - y));
                }
            }
        } else {
            // compositing with one thread per sample: segmented warp-shuffle scans inside each warp, carries across the four
            // warps through shared memory (scripts/nerf.py:176-288 and its reverse; the reverse sweep multiplies, never divides)
            const float cr = sigmoid_exact(hz[0]), cg = sigmoid_exact(hz[1]), cb = sigmoid_exact(hz[2]);
            const float sg = fmaxf(hz[3], 0.0f);
            const float e = expf((0.0f - sg) * my_dist);
            const float a = 1.0f - e;
            const float qv = live ? (1.0f - a) + 1e-10f : 1.0f;
            float pr = qv;                                   // segmented inclusive product
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const float o = __shfl_up_sync(0xffffffffu, pr, d);
                if (lane >= d && smp >= d) pr *= o;
            }
            if (lane == 31) { tailp[warp] = pr; tail_s[warp] = smp; }
            if (lane == 0) headq[warp] = qv;
            if (live && smp == 0) {
                color_s[ray_l * 3] = 0.f; color_s[ray_l * 3 + 1] = 0.f; color_s[ray_l * 3 + 2] = 0.f;
                tgt_s[ray_l * 3] = tg0; tgt_s[ray_l * 3 + 1] = tg1; tgt_s[ray_l * 3 + 2] = tg2;
            }
            __syncthreads();
            float carry = 1.0f;                              // product of this ray's samples in earlier warps
            if (smp > lane) {
                for (int w2 = warp - 1; w2 >= 0; --w2) {
                    carry *= tailp[w2];
                    if (tail_s[w2] < 32) break;              // that warp's last segment started inside it
                }
            }
            const float Cpre = pr * carry;                   // inclusive product prod_{k<=s} q_k
            const float T = (smp == 0) ? 1.0f : Cpre;
            const float wgt = a * T;
            {   // colour: segmented inclusive sums; the (warp, ray) segments of a ray are added in warp order (two barriers
                // below make the order fixed: one segment per warp per ray, ascending warps)
                float s0 = live ? wgt * cr : 0.f, s1 = live ? wgt * cg : 0.f, s2 = live ? wgt * cb : 0.f;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const float o0 = __shfl_up_sync(0xffffffffu, s0, d), o1 = __shfl_up_sync(0xffffffffu, s1, d), o2 = __shfl_up_sync(0xffffffffu, s2, d);
                    if (lane >= d && smp >= d) { s0 += o0; s1 += o1; s2 += o2; }
                }
                for (int w2 = 0; w2 < 4; ++w2) {             // fixed order: reproducible colours
                    if (warp == w2 && live && (lane == 31 || smp == S - 1)) {
                        color_s[ray_l * 3] += s0; color_s[ray_l * 3 + 1] += s1; color_s[ray_l * 3 + 2] += s2;
                    }
                    __syncthreads();
                }
            }
            float dc0 = 0.f, dc1 = 0.f, dc2 = 0.f;
            if (live) {
                const float c0 = color_s[ray_l * 3], c1 = color_s[ray_l * 3 + 1], c2 = color_s[ray_l * 3 + 2];
                if (smp == 0 && p.color) {
                    float *co = p.color + (row0 / S + ray_l) * 3;
                    co[0] = c0; co[1] = c1; co[2] = c2;
                }
                if (p.target) {
                    const float d0 = c0 - tgt_s[ray_l * 3], d1 = c1 - tgt_s[ray_l * 3 + 1], d2 = c2 - tgt_s[ray_l * 3 + 2];
                    if (smp == 0) loss_acc += d0 * d0 + d1 * d1 + d2 * d2;
                    dc0 = 2.0f * d0; dc1 = 2.0f * d1; dc2 = 2.0f * d2;
                }
            }
            if (p.want_grad) {
                // G_s = dT_s + q_{s+1} G_{s+1}: suffix scan of affine maps; B = 0 at a ray's last sample
                const float d_w = cr * dc0 + cg * dc1 + cb * dc2;
                const float dT = (smp == 0 || !live) ? 0.0f : d_w * a;
                float qn = __shfl_down_sync(0xffffffffu, qv, 1);
                if (lane == 31) qn = warp < 3 ? headq[warp + 1] : 0.0f;
                float Aa = dT, Bb = (live && smp + 1 < S) ? qn : 0.0f;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const float A2 = __shfl_down_sync(0xffffffffu, Aa, d);
                    const float B2 = __shfl_down_sync(0xffffffffu, Bb, d);
                    if (lane + d < 32) { Aa = fmaf(Bb, A2, Aa); Bb = Bb * B2; }
                }
                if (lane == 0) { headA[warp] = Aa; headB[warp] = Bb; }
                __syncthreads();
                float Gn = 0.0f;                             // G at lane 0 of the next warp
                for (int w2 = 3; w2 > warp; --w2) Gn = fmaf(headB[w2], Gn, headA[w2]);
                const float Gv = fmaf(Bb, Gn, Aa);
                float Cm1 = __shfl_up_sync(0xffffffffu, Cpre, 1);
                if (lane == 0) Cm1 = carry;
                if (smp == 0) Cm1 = 1.0f;
                const float d_alpha = d_w * T - Cm1 * Gv;
                if (live) {
                    dz[0] = (wgt * dc0) * (cr * (1.0f - cr));
                    dz[1] = (wgt * dc1) * (cg * (1.0f - cg));
                    dz[2] = (wgt * dc2) * (cb * (1.0f - cb));
                    dz[3] = sg > 0.0f ? d_alpha * e * my_dist : 0.0f;
                }
            }
        }
        if (!p.want_grad) { __syncthreads(); continue; }
        // ---- backward
        *reinterpret_cast<float4 *>(Zh + tid * 4) = make_float4(dz[0], dz[1], dz[2], dz[3]);
        __syncthreads();
        {   // last layer: dW = Alast^T dZ (thread: input row `lane`, 4 outputs; its warp's 32 samples), then dH
            const float *col = Alast + lane;
#pragma unroll 4
            for (int s = 32 * warp; s < 32 * warp + 32; ++s) {
                const float av = col[s * LD];
                const float4 d = *reinterpret_cast<const float4 *>(Zh + s * 4);
                fma2(gl[0], gl[1], av, d.x, d.y); fma2(gl[2], gl[3], av, d.z, d.w);
            }
            __syncthreads();                                 // every warp is done reading Alast: it becomes dZ
            float acc[4][8] = {};
            float4 z[4];
#pragma unroll
            for (int s = 0; s < 4; ++s) z[s] = *reinterpret_cast<const float4 *>(Zh + (lane + 32 * s) * 4);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 w0 = *reinterpret_cast<const float4 *>(WTl + j * HW + 8 * warp), w1 = *reinterpret_cast<const float4 *>(WTl + j * HW + 8 * warp + 4);
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const float zv = comp(z[s], j);
                    fma2(acc[s][0], acc[s][1], zv, w0.x, w0.y); fma2(acc[s][2], acc[s][3], zv, w0.z, w0.w);
                    fma2(acc[s][4], acc[s][5], zv, w1.x, w1.y); fma2(acc[s][6], acc[s][7], zv, w1.z, w1.w);
                }
            }
            store_masked(Alast, warp, lane, acc);
            __syncthreads();
        }
        if (three) {   // layer 1: dW_1 = A_1^T dZ_1 (dZ_1 sits in A_2), then dZ_0 in place of A_1
            dw_8x4(A1, A2, LD, warp, lane, g1);
            __syncthreads();
            float acc[4][8] = {};
            gemm_4x8<HW>(A2, WT1, warp, lane, acc);
            store_masked(A1, warp, lane, acc);
            __syncthreads();
        }
        {   // layer 0: dW_0 = A_0^T dZ_0 (dZ_0 sits in A_1); rows 32..35 of A_0 (the ones column among them) on the side
            dw_8x4(A0, A1, LD, warp, lane, g0);
#pragma unroll 4
            for (int s = 32 * warp; s < 32 * warp + 32; ++s) {
                const float4 a = *reinterpret_cast<const float4 *>(A0 + s * LD + 32);
                const float d = A1[s * LD + lane];
                fma2(g0x[0], g0x[1], d, a.x, a.y); fma2(g0x[2], g0x[3], d, a.z, a.w);
            }
        }
        __syncthreads();                                     // the next tile overwrites A_0 / A_1
    }

    // ---- this CTA's partial: the four warps' accumulators are added in warp order into shared memory, then written out
    float *D0 = sm;                    // [36][32]
    float *D1 = D0 + K0 * HW;          // [32][32]
    float *Dl = D1 + HW * HW;          // [32][4]
    __syncthreads();
    for (int e = tid; e < K0 * HW + HW * HW + HW * 4; e += FT) sm[e] = 0.0f;
    __syncthreads();
    if (p.want_grad) {
        const int gi = lane >> 3, gj = lane & 7;
        for (int w2 = 0; w2 < 4; ++w2) {
            if (warp == w2) {
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        D0[(8 * gi + i) * HW + 4 * gj + j] += g0[i][j];
                        D1[(8 * gi + i) * HW + 4 * gj + j] += g1[i][j];
                    }
#pragma unroll
                for (int i = 0; i < 4; ++i) D0[(32 + i) * HW + lane] += g0x[i];
#pragma unroll
                for (int j = 0; j < 4; ++j) Dl[lane * 4 + j] += gl[j];
            }
            __syncthreads();
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) loss_acc += __shfl_xor_sync(0xffffffffu, loss_acc, d);
    if (lane == 0) red_s[warp] = loss_acc;
    __syncthreads();
    float *part = p.part + (size_t)blockIdx.x * p.part_stride;
    if (tid == 0) part[0] = (red_s[0] + red_s[1]) + (red_s[2] + red_s[3]);
    if (p.want_grad) {
        for (int l = 0; l < L; ++l) {
            const int in_l = p.dims[l], out_l = p.dims[l + 1];
            const float *D = l == 0 ? D0 : (l == L - 1 ? Dl : D1);
            const int ldd = l == L - 1 ? 4 : HW;
            float *o = part + p.part_off[l];
            for (int e = tid; e < (in_l + 1) * out_l; e += FT) o[e] = D[(e / out_l) * ldd + e % out_l];
        }
    }
}

// sum of the per-CTA partials in a fixed order; seed; += into (or = over) the caller's padded d_ws / d_bs (the reference
// accumulates).  32 consecutive elements per block (one coalesced 128 B line per partial), 32 warps stride over the partials
// with all their loads in flight, fixed-order combine through shared memory.
__global__ void __launch_bounds__(1024) fused_f32_reduce_kernel(const float *__restrict__ part, int n_part, F32Params p, float *__restrict__ d_ws,
                                                                 float *__restrict__ d_bs, float *__restrict__ loss, float seed_value, int seed_is_loss,
                                                                 int overwrite)
{
    __shared__ float sloss;
    __shared__ float acc[31][33];
    // the loss sum (warp 31) and the gradient gather (warps 0-30) run side by side under one barrier
    const int el = threadIdx.x & 31, grp = threadIdx.x >> 5;
    const int n_el = p.part_stride - 1;
    const int e_glob = blockIdx.x * 32 + el;
    if (grp == 31) {
        float s = 0.0f;
#pragma unroll 8
        for (int i = el; i < n_part; i += 32) s += part[(size_t)i * p.part_stride];
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        if (el == 0) { sloss = s; if (blockIdx.x == 0 && loss) loss[0] = s; }
    } else if (d_ws) {
        float s = 0.0f;
        if (e_glob < n_el) {
            const float *src = part + 1 + e_glob;
#pragma unroll 8
            for (int i = grp; i < n_part; i += 31) s += src[(size_t)i * p.part_stride];
        }
        acc[grp][el] = s;
    }
    __syncthreads();
    if (!d_ws) return;
    const float scale = seed_is_loss ? sloss * seed_value : seed_value;
    if (grp != 0 || e_glob >= n_el) return;
    float s = 0.0f;
#pragma unroll
    for (int w2 = 0; w2 < 31; ++w2) s += acc[w2][el];
    int e = e_glob + 1, l = 0;
    while (l + 1 < p.L && e >= p.part_off[l + 1]) ++l;
    e -= p.part_off[l];
    const int out_l = p.dims[l + 1], k = e / out_l, j = e % out_l;
    float *dst = k < p.dims[l] ? d_ws + ((size_t)l * p.max_in + k) * p.max_out + j : d_bs + (size_t)l * p.max_out + j;
    *dst = overwrite ? scale * s : *dst + scale * s;
}

} // namespace

// LNB_ERR_UNSUPPORTED when the problem does not fit the fused exact kernel (the caller then runs the layerwise kernels).
// Rays and camera batches are encoded first (float64 sample positions and sin / cos like the reference host, encode.cu).
// overwrite != 0: d_ws / d_bs are written (=) instead of accumulated (+=), live entries only (the trainer's buffer).
int lnb_fused_f32_step(lnb_ctx *ctx, const lnb_mlp *mlp, const lnb_step_args *a, bool nerf, int overwrite,
                       const lnb_comp_args *cx)
{
    const int L = mlp->n_layers;
    auto unsupported = [&](const char *why) {
        ctx->err = std::string("fused fp32 path: ") + why;
        return LNB_ERR_UNSUPPORTED;
    };
    if (lnb_cx_extras(cx)) return unsupported("no compositing extras (background, acc, depth): the layerwise kernels have them");
    if (L < 2 || L > 3) return unsupported("needs 2 or 3 layers");
    if (mlp->dims[0] + 1 > K0) return unsupported("input width + 1 must be <= 36");
    for (int l = 1; l < L; ++l)
        if (mlp->dims[l] + 1 > HW) return unsupported("hidden width + 1 must be <= 32");
    if (mlp->dims[L] > 4) return unsupported("more than 4 output channels");
    if (a->inter || a->rgba || a->alpha || a->cumprod || a->weights || a->d_X || a->d_target || a->d_dists || a->d_color || a->d_inter)
        return unsupported("only loss, colour, d_ws and d_bs are produced");
    if (a->color && a->color_accumulate) return unsupported("colour accumulation");
    const int R = a->R, S = nerf ? a->S : 1;
    const long long N = a->n_rows > 0 ? a->n_rows : (long long)R * S;
    if (nerf && (S < 2 || S > FT || N != (long long)R * S)) return unsupported("needs 2 <= S <= 128 and n_rows == R*S");
    if (!nerf && (N != R || a->target_w > 4)) return unsupported("needs n_rows == R and a target of <= 4 columns");
    if (a->rows > N) return unsupported("rows > n_rows");
    if (a->want_grad && !a->target && N > 0) return unsupported("gradient without target");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;

    const bool cam = !a->X && !a->rays_o && a->cam;
    const bool rays = !a->X && (a->rays_o || cam);
    F32Params p{};
    p.target = a->target; p.ws = a->ws; p.bs = a->bs;
    p.color = nerf ? a->color : nullptr;
    p.N = N; p.R = R; p.S = S;
    p.rows_per_tile = nerf ? (FT / S) * S : FT;
    p.n_tiles = (int)((N + p.rows_per_tile - 1) / p.rows_per_tile);
    p.L = L;
    for (int l = 0; l <= L; ++l) p.dims[l] = mlp->dims[l];
    p.max_in = mlp->max_in; p.max_out = mlp->max_out;
    p.head = mlp->head; p.want_grad = a->want_grad; p.Wt = a->target_w > 0 ? a->target_w : 3;
    int off = 1;
    for (int l = 0; l < L; ++l) { p.part_off[l] = off; off += (mlp->dims[l] + 1) * mlp->dims[l + 1]; }
    p.part_stride = off;

    p.c_in_magic = (unsigned)((0x100000000ull + (unsigned)mlp->dims[0] - 1) / (unsigned)mlp->dims[0]);
    const size_t smem = sizeof(float) * ((size_t)FT * LD * L + FT * 4 + K0 * HW + (L == 3 ? 2 * HW * HW : 0) + 2 * HW * 4 + 3 * HW + 512);
    int grid = ctx->sm_count * 3;
    if (grid > p.n_tiles) grid = p.n_tiles;
    if (grid < 1) grid = 1;
    const int c_in = mlp->dims[0];
    LNB_TRY(lnb_arena_reserve(ctx, (size_t)grid * p.part_stride * sizeof(float) + (rays ? ((size_t)N * c_in + (size_t)R * S) * sizeof(float) + 1024 : 0) + 4096));
    p.part = (float *)lnb_arena_take(ctx, (size_t)grid * p.part_stride * sizeof(float));
    p.X = a->X; p.dists = a->dists;
    if (rays) {
        float *Xe = (float *)lnb_arena_take(ctx, (size_t)N * c_in * sizeof(float)), *de = (float *)lnb_arena_take(ctx, (size_t)R * S * sizeof(float));
        const int Ed = lnb_rays_dir_bands(c_in, a->pe_bands);
        if (cam) LNB_TRY(lnb_launch_camera_encode(ctx, a->cam, lnb_cx_views(cx), R, S, a->pe_bands, Ed, Xe, de, nullptr, 0));
        else LNB_TRY(lnb_launch_sample_encode(ctx, a->rays_o, a->rays_d, a->t, a->ray_dtype == LNB_RAY_F64, R, S, a->pe_bands, Ed, Xe, de));
        p.X = Xe; p.dists = de;
    }
    p.x_vec4 = (reinterpret_cast<uintptr_t>(p.X) & 15) == 0 && ((long long)p.rows_per_tile * c_in) % 4 == 0;
    float *loss = a->loss ? a->loss : (float *)lnb_arena_take(ctx, 16);
    if (N > 0) {
        LNB_CUDA(cudaFuncSetAttribute(fused_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        lnb_prof_begin(ctx, "fused_f32_kernel");
        fused_f32_kernel<<<grid, FT, smem, ctx->stream>>>(p);
        lnb_prof_end(ctx);
        LNB_CHECK_LAUNCH();
    } else {
        grid = 0;
    }
    const int n_el = p.part_stride - 1;
    const int blocks = a->want_grad ? (n_el + 31) / 32 : 1;
    fused_f32_reduce_kernel<<<blocks, 1024, 0, ctx->stream>>>(p.part, grid, p, a->want_grad ? a->d_ws : nullptr, a->want_grad ? a->d_bs : nullptr, loss,
                                                              a->seed_mode == LNB_SEED_LOSS ? 1.0f : a->seed, a->seed_mode == LNB_SEED_LOSS, overwrite);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}
