// kernels_f32.cu -- the exact (IEEE fp32, CUDA-core) layerwise kernels of libloma_nerf_b200.so.
//
// These implement the reference's path one stage at a time with every intermediate materialised,
// which is what the compat ABI needs (the reference hosts read intermediate_outputs, rgba, alpha,
// cumprod_alpha, weights_samples back) and what the fused tensor-core kernel (fused_tc.cu) is
// checked against on the device.  Reference: /root/reference/scripts/nerf.py:67-304,
// scripts/mlp_fit.py:39-147 and their reverse (loma_public/reverse_diff.py:576-951).
#include <stdint.h>

#include "camera.cuh"
#include "lnb_internal.h"

namespace {

__device__ __forceinline__ float sigmoidf_(float z) { return 1.0f / (1.0f + expf(0.0f - z)); }

// ------------------------------------------------------------------------------------------------
// Row GEMM with fused epilogue.  256 threads, thread tile 4x4, BM x BN block tile (128x32 or 64x64).
//   Thread (tx,ty): rows ty*4.., cols tx*4..
// ------------------------------------------------------------------------------------------------
template <int BM, int BN>
__global__ void __launch_bounds__(256) row_gemm_kernel(lnb_gemm_args g)
{
    // K slab of 40: the reference's layer widths (22..33 inputs, 16..30 hidden) fit one slab.  A is
    // kept row-major in shared memory (pitch BK+1): a warp stages one row segment per load
    // (coalesced, conflict-free) and reads 4 rows x 1 scalar per k (4 distinct banks + broadcast).
    constexpr int BK = 40;
    static_assert(BM * BN == 4096, "256 threads x 4x4");
    constexpr int TXN = BN / 4; // threads along n
    __shared__ float As[BM][BK + 1];
    __shared__ __align__(16) float Bs[BK][BN + 4];
    const int t = threadIdx.x;
    const int tx = t % TXN, ty = t / TXN;
    const long long row0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

    for (int k0 = 0; k0 < g.k_dim; k0 += BK) {
        const int kmax = g.k_dim - k0 < BK ? g.k_dim - k0 : BK;
        for (int e = t; e < BM * BK; e += 256) {
            const int i = e / BK, kk = e % BK;
            const long long r = row0 + i;
            float v = 0.0f;
            if (r < g.a_rows && kk < kmax) v = __ldg(g.A + r * g.lda + (k0 + kk));
            As[i][kk] = v;
        }
        for (int e = t; e < BK * BN; e += 256) {
            const int kk = e / BN, n = e % BN;
            float v = 0.0f;
            if (kk < kmax && n0 + n < g.n_dim)
                v = __ldg(g.B + (long long)(k0 + kk) * g.sbk + (long long)(n0 + n) * g.sbn);
            Bs[kk][n] = v;
        }
        __syncthreads();
#pragma unroll 4
        for (int kk = 0; kk < kmax; ++kk) {
            const float4 b = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
            const float av[4] = {As[ty * 4][kk], As[ty * 4 + 1][kk], As[ty * 4 + 2][kk], As[ty * 4 + 3][kk]};
            const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        long long r = row0 + ty * 4 + i;
        if (r >= g.rows) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int n = n0 + tx * 4 + j;
            if (n >= g.n_dim) continue;
            float v = acc[i][j];
            float *c = g.C + r * g.ldc + n;
            if (g.acc) v += *c;
            if (g.bias) v += __ldg(g.bias + n);
            if (g.act == ACT_RELU) v = v > 0.0f ? v : 0.0f;
            else if (g.act == ACT_SIGMOID) v = sigmoidf_(v);
            else if (g.act == ACT_NERF_HEAD) v = (n == 3) ? (v > 0.0f ? v : 0.0f) : sigmoidf_(v);
            if (g.mask && !(__ldg(g.mask + r * g.ldmask + n) > 0.0f)) v = 0.0f;
            *c = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// dW partials: contraction over rows.  Block = 256 threads as 16 (k) x 16 (j); thread tile TKxTJ.
// ------------------------------------------------------------------------------------------------
template <int TK, int TJ>
__global__ void __launch_bounds__(256)
dw_partials_kernel(const float *__restrict__ H, int ldh, const float *__restrict__ dZ, int ldz,
                   float *__restrict__ partial, int in_dim, int out_dim, long long rows,
                   long long rows_per_chunk)
{
    constexpr int SLAB = 32, KT = 16 * TK, JT = 16 * TJ;
    __shared__ float Hs[SLAB][KT + 1];
    __shared__ float Zs[SLAB][JT + 1];
    const int t = threadIdx.x, tj = t % 16, tk = t / 16;
    const int k0 = blockIdx.y * KT, j0 = blockIdx.z * JT;
    const long long r_begin = (long long)blockIdx.x * rows_per_chunk;
    long long r_end = r_begin + rows_per_chunk;
    if (r_end > rows) r_end = rows;
    float acc[TK][TJ];
#pragma unroll
    for (int a = 0; a < TK; ++a)
#pragma unroll
        for (int b = 0; b < TJ; ++b) acc[a][b] = 0.0f;
    for (long long r0 = r_begin; r0 < r_end; r0 += SLAB) {
        for (int e = t; e < SLAB * KT; e += 256) {
            int i = e / KT, k = e % KT;
            long long r = r0 + i;
            float v = 0.0f;
            if (r < r_end) {
                int kk = k0 + k;
                if (kk < in_dim) v = __ldg(H + r * ldh + kk);
                else if (kk == in_dim) v = 1.0f; // bias-gradient row
            }
            Hs[i][k] = v;
        }
        for (int e = t; e < SLAB * JT; e += 256) {
            int i = e / JT, j = e % JT;
            long long r = r0 + i;
            float v = 0.0f;
            if (r < r_end && j0 + j < out_dim) v = __ldg(dZ + r * ldz + j0 + j);
            Zs[i][j] = v;
        }
        __syncthreads();
#pragma unroll 8
        for (int i = 0; i < SLAB; ++i) {
            float hv[TK], zv[TJ];
#pragma unroll
            for (int a = 0; a < TK; ++a) hv[a] = Hs[i][tk + 16 * a];
#pragma unroll
            for (int b = 0; b < TJ; ++b) zv[b] = Zs[i][tj + 16 * b];
#pragma unroll
            for (int a = 0; a < TK; ++a)
#pragma unroll
                for (int b = 0; b < TJ; ++b) acc[a][b] = fmaf(hv[a], zv[b], acc[a][b]);
        }
        __syncthreads();
    }
    float *out = partial + (size_t)blockIdx.x * (size_t)(in_dim + 1) * out_dim;
#pragma unroll
    for (int a = 0; a < TK; ++a) {
        int k = k0 + tk + 16 * a;
        if (k > in_dim) continue;
#pragma unroll
        for (int b = 0; b < TJ; ++b) {
            int j = j0 + tj + 16 * b;
            if (j < out_dim) out[(size_t)k * out_dim + j] = acc[a][b];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Wide layers (e.g. the paper-size 256-wide MLP): classic register-blocked fp32 GEMMs.  128 x 128
// block tile, K slab of 16, 256 threads, 8 x 8 outputs per thread as 2 x 2 groups of 4 x 4 (so the
// shared-memory reads are float4: the A reads broadcast, the B reads are contiguous), the next slab
// prefetched into registers while the current one is multiplied (one barrier per slab).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sgemm128_kernel(lnb_gemm_args g)
{
    constexpr int BM = 128, BN = 128, BK = 16;
    __shared__ __align__(16) float As[2][BK][BM + 4];   // k-major: As[k][row]
    __shared__ __align__(16) float Bs[2][BK][BN + 4];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const long long row0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int ar = t >> 2, ak = (t & 3) * 4;            // A loader: rows ar, ar + 64; columns ak .. ak + 3 of the slab
    const bool b_n_fast = g.sbn == 1;                   // B loader walks the contiguous direction of B
    float4 pa[2];
    float pb[8];
    auto load = [&](int k0) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const long long r = row0 + ar + 64 * h;
            pa[h] = r < g.a_rows ? __ldg(reinterpret_cast<const float4 *>(g.A + r * g.lda + k0 + ak)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int e = t + 256 * i;
            const int kk = b_n_fast ? e >> 7 : e & 15, n = b_n_fast ? e & 127 : e >> 4;
            pb[i] = n0 + n < g.n_dim ? __ldg(g.B + (long long)(k0 + kk) * g.sbk + (long long)(n0 + n) * g.sbn) : 0.0f;
        }
    };
    auto store = [&](int buf) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            As[buf][ak + 0][ar + 64 * h] = pa[h].x; As[buf][ak + 1][ar + 64 * h] = pa[h].y;
            As[buf][ak + 2][ar + 64 * h] = pa[h].z; As[buf][ak + 3][ar + 64 * h] = pa[h].w;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int e = t + 256 * i;
            const int kk = b_n_fast ? e >> 7 : e & 15, n = b_n_fast ? e & 127 : e >> 4;
            Bs[buf][kk][n] = pb[i];
        }
    };
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
    load(0);
    store(0);
    __syncthreads();
    const int n_slabs = g.k_dim / BK;
    for (int sl = 0; sl < n_slabs; ++sl) {
        const int buf = sl & 1;
        if (sl + 1 < n_slabs) load((sl + 1) * BK);
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[buf][kk][ty * 4]), a1 = *reinterpret_cast<const float4 *>(&As[buf][kk][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[buf][kk][tx * 4]), b1 = *reinterpret_cast<const float4 *>(&Bs[buf][kk][64 + tx * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (sl + 1 < n_slabs) store(buf ^ 1);
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const long long r = row0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + i - 4);
        if (r >= g.rows) continue;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + j - 4);
            if (n >= g.n_dim) continue;
            float v = acc[i][j];
            float *c = g.C + r * g.ldc + n;
            if (g.acc) v += *c;
            if (g.bias) v += __ldg(g.bias + n);
            if (g.act == ACT_RELU) v = v > 0.0f ? v : 0.0f;
            else if (g.act == ACT_SIGMOID) v = sigmoidf_(v);
            else if (g.act == ACT_NERF_HEAD) v = (n == 3) ? (v > 0.0f ? v : 0.0f) : sigmoidf_(v);
            if (g.mask && !(__ldg(g.mask + r * g.ldmask + n) > 0.0f)) v = 0.0f;
            *c = v;
        }
    }
}

// dW partials of a wide layer: partial[z][k][j] = sum over the chunk's rows of H[i][k] dZ[i][j] for a 128 x 128 (k, j)
// tile, and (k-tile 0 only) the bias row partial[z][in_dim][j] = sum_i dZ[i][j].  Same register blocking.
__global__ void __launch_bounds__(256)
dw128_kernel(const float *__restrict__ H, int ldh, const float *__restrict__ dZ, int ldz, float *__restrict__ partial, int in_dim,
             int out_dim, long long rows, long long rows_per_chunk)
{
    constexpr int SL = 16;
    __shared__ __align__(16) float Hs[2][SL][128 + 4];
    __shared__ __align__(16) float Zs[2][SL][128 + 4];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int k0 = blockIdx.y * 128, j0 = blockIdx.z * 128;
    const long long r_begin = (long long)blockIdx.x * rows_per_chunk;
    long long r_end = r_begin + rows_per_chunk;
    if (r_end > rows) r_end = rows;
    const int li = t >> 5, lc = (t & 31) * 4;           // loader: slab rows li, li + 8; columns lc .. lc + 3
    float4 ph[2], pz[2];
    auto load = [&](long long r0) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const long long r = r0 + li + 8 * h;
            const bool live = r < r_end;
            ph[h] = (live && k0 + lc < in_dim) ? __ldg(reinterpret_cast<const float4 *>(H + r * ldh + k0 + lc)) : make_float4(0.f, 0.f, 0.f, 0.f);
            pz[h] = (live && j0 + lc < out_dim) ? __ldg(reinterpret_cast<const float4 *>(dZ + r * ldz + j0 + lc)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto store = [&](int buf) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            *reinterpret_cast<float4 *>(&Hs[buf][li + 8 * h][lc]) = ph[h];
            *reinterpret_cast<float4 *>(&Zs[buf][li + 8 * h][lc]) = pz[h];
        }
    };
    float acc[8][8], bsum[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        bsum[i] = 0.0f;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
    }
    const bool do_bias = blockIdx.y == 0 && ty == 0;
    if (r_begin < r_end) {
        load(r_begin);
        store(0);
    }
    __syncthreads();
    int buf = 0;
    for (long long r0 = r_begin; r0 < r_end; r0 += SL, buf ^= 1) {
        const bool more = r0 + SL < r_end;
        if (more) load(r0 + SL);
#pragma unroll
        for (int i = 0; i < SL; ++i) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&Hs[buf][i][ty * 4]), a1 = *reinterpret_cast<const float4 *>(&Hs[buf][i][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Zs[buf][i][tx * 4]), b1 = *reinterpret_cast<const float4 *>(&Zs[buf][i][64 + tx * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(av[a], bv[b], acc[a][b]);
            if (do_bias)
#pragma unroll
                for (int b = 0; b < 8; ++b) bsum[b] += bv[b];
        }
        if (more) store(buf ^ 1);
        __syncthreads();
    }
    float *out = partial + (size_t)blockIdx.x * (size_t)(in_dim + 1) * out_dim;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        const int k = k0 + (a < 4 ? ty * 4 + a : 64 + ty * 4 + a - 4);
        if (k >= in_dim) continue;
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int j = j0 + (b < 4 ? tx * 4 + b : 64 + tx * 4 + b - 4);
            if (j < out_dim) out[(size_t)k * out_dim + j] = acc[a][b];
        }
    }
    if (do_bias)
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const int j = j0 + (b < 4 ? tx * 4 + b : 64 + tx * 4 + b - 4);
            if (j < out_dim) out[(size_t)in_dim * out_dim + j] = bsum[b];
        }
}

// Fast path for narrow layers (in_dim + 1 <= KP <= 64, out_dim <= 32): one warp per row, lane j
// owns output column j and keeps the whole column dW[0..in_dim][j] (+ the bias row) in registers;
// the row of H is staged in shared memory and read back as broadcast float4s.  8 warps stride
// over the block's rows and are combined through shared memory in warp order (deterministic).
template <int KP>
__global__ void __launch_bounds__(256)
dw_rows_kernel(const float *__restrict__ H, int ldh, const float *__restrict__ dZ, int ldz,
               float *__restrict__ partial, int in_dim, int out_dim, long long rows,
               long long rows_per_chunk)
{
    __shared__ __align__(16) float hs[8][2][KP];
    __shared__ float accs[KP][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int e = threadIdx.x; e < KP * 33; e += 256) (&accs[0][0])[e] = 0.0f;
    const long long r_begin = (long long)blockIdx.x * rows_per_chunk;
    long long r_end = r_begin + rows_per_chunk;
    if (r_end > rows) r_end = rows;
    float acc[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) acc[k] = 0.0f;
    constexpr int NH = (KP + 31) / 32; // H elements per lane per row
    // two rows per iteration (r and r + 8), the next pair's loads issued before this pair's math
    auto load_row = [&](long long r, float (&h)[NH], float &dz) {
#pragma unroll
        for (int q = 0; q < NH; ++q) {
            const int k = lane + 32 * q;
            h[q] = (r < r_end && k < in_dim) ? __ldg(H + r * ldh + k) : ((r < r_end && k == in_dim) ? 1.0f : 0.0f);
        }
        dz = (r < r_end && lane < out_dim) ? __ldg(dZ + r * ldz + lane) : 0.0f;
    };
    float ha[NH], hb[NH], dza, dzb;
    long long r = r_begin + warp;
    load_row(r, ha, dza);
    load_row(r + 8, hb, dzb);
    for (; r < r_end; r += 16) {
#pragma unroll
        for (int q = 0; q < NH; ++q) {
            const int k = lane + 32 * q;
            if (k < KP) { hs[warp][0][k] = ha[q]; hs[warp][1][k] = hb[q]; }
        }
        const float za = dza, zb = dzb;
        load_row(r + 16, ha, dza);
        load_row(r + 24, hb, dzb);
        __syncwarp();
#pragma unroll
        for (int k4 = 0; k4 < KP / 4; ++k4) {
            const float4 h0 = *reinterpret_cast<const float4 *>(&hs[warp][0][k4 * 4]);
            const float4 h1 = *reinterpret_cast<const float4 *>(&hs[warp][1][k4 * 4]);
            acc[k4 * 4] = fmaf(h1.x, zb, fmaf(h0.x, za, acc[k4 * 4]));
            acc[k4 * 4 + 1] = fmaf(h1.y, zb, fmaf(h0.y, za, acc[k4 * 4 + 1]));
            acc[k4 * 4 + 2] = fmaf(h1.z, zb, fmaf(h0.z, za, acc[k4 * 4 + 2]));
            acc[k4 * 4 + 3] = fmaf(h1.w, zb, fmaf(h0.w, za, acc[k4 * 4 + 3]));
        }
        __syncwarp();
    }
    __syncthreads();
    for (int w = 0; w < 8; ++w) { // warps add in a fixed order: the result is deterministic
        if (warp == w) {
#pragma unroll
            for (int k = 0; k < KP; ++k) accs[k][lane] += acc[k];
        }
        __syncthreads();
    }
    float *out = partial + (size_t)blockIdx.x * (size_t)(in_dim + 1) * out_dim;
    for (int e = threadIdx.x; e < (in_dim + 1) * out_dim; e += 256) out[e] = accs[e / out_dim][e % out_dim];
}

__global__ void dw_reduce_kernel(const float *__restrict__ partial, int n_chunks, int in_dim,
                                 int out_dim, float *__restrict__ d_w, int ldw,
                                 float *__restrict__ d_b, float seed_value,
                                 const float *__restrict__ seed_dev)
{
    // one warp per output element: lanes stride over chunks, fixed-order shuffle tree
    const int lane = threadIdx.x & 31;
    const long long e = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long n = (long long)(in_dim + 1) * out_dim;
    if (e >= n) return;
    float s = 0.0f;
    for (int z = lane; z < n_chunks; z += 32) s += __ldg(partial + (size_t)z * n + e);
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if (lane == 0) {
        float scale = seed_value * (seed_dev ? __ldg(seed_dev) : 1.0f);
        int k = (int)(e / out_dim), j = (int)(e % out_dim);
        if (k < in_dim) d_w[(size_t)k * ldw + j] += scale * s;
        else if (d_b) d_b[j] += scale * s;
    }
}

// ------------------------------------------------------------------------------------------------
// Compositing.  One warp per ray; samples are visited in chunks of 32 (lane = sample in chunk) so
// loads are coalesced; transmittance is a warp-shuffle product scan with a carried prefix.
// Reference semantics (scripts/nerf.py:176-288, SURVEY.md 8 a5):
//   alpha = 1 - expf(-sigma*dist); q = (1-alpha)+1e-10f; C_s = prod_{k<=s} q_k; T_0 = 1, T_s = C_s
//   w = alpha*T; color += sum_s w*rgb
// ------------------------------------------------------------------------------------------------
constexpr int COMP_WARPS = 8;
constexpr int COMP_MAX_CHUNKS = 64; // S <= 2048

__device__ __forceinline__ float warp_incl_prod(float p, int lane)
{
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        float o = __shfl_up_sync(0xffffffffu, p, d);
        if (lane >= d) p *= o;
    }
    return p;
}

// The compositing extras (lnb_composite) as the EXT instantiations of the kernels below take them (by value): the
// background, the acc / depth outputs and the depth source of sample s of ray r (sample_depth)
struct CompK {
    int background;
    float bg0, bg1, bg2;
    float *acc, *depth;
    const void *t;
    int t_f64, cam_mode;
    CamDev cam;
};
template <bool VIEWS>
__device__ __forceinline__ float sample_depth(const CompK &k, int ray, int s, int S)
{
    if (VIEWS) {   // views mode: camera mode's depth under the ray's jitter key g = view * P + q and seed'
        CamDev c = k.cam;
        if (c.seed_dev) c.seed = *c.seed_dev;
        return (float)cam_t_f64(c, (long long)__ldg(c.view + ray) * c.P + __ldg(c.pixels + ray), s, S);
    }
    if (k.cam_mode) return (float)cam_t_f64(k.cam, cam_pixel(k.cam, ray), s, S);
    const size_t i = (size_t)ray * S + s;
    return k.t_f64 ? (float)__ldg(reinterpret_cast<const double *>(k.t) + i) : __ldg(reinterpret_cast<const float *>(k.t) + i);
}

// EXT: with the extras of `k` (acc = sum w, depth = sum w t, colour += (1 - acc) bg before the caller's colour is added)
template <bool EXT, bool VIEWS = false>   // VIEWS: the depths of a views batch (a separate instantiation)
__global__ void __launch_bounds__(COMP_WARPS * 32)
composite_fwd_kernel(const float *__restrict__ head, int ldh, const float *__restrict__ dists,
                     const float *__restrict__ target, int R, int S, float *__restrict__ rgba,
                     float *__restrict__ alpha, float *__restrict__ cumprod,
                     float *__restrict__ weights, float *__restrict__ color, int color_accumulate,
                     float *__restrict__ ray_sse, const CompK k)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ray = blockIdx.x * COMP_WARPS + warp;
    if (ray >= R) return;
    float carry = 1.0f, c0 = 0.0f, c1 = 0.0f, c2 = 0.0f, c3 = 0.0f, c4 = 0.0f;   // c3, c4: acc, depth (EXT)
    for (int s0 = 0; s0 < S; s0 += 32) {
        const int s = s0 + lane;
        const bool valid = s < S;
        const size_t i = (size_t)ray * S + s;
        float r = 0.f, gch = 0.f, b = 0.f, sig = 0.f, dist = 0.f;
        if (valid) {
            const float *h = head + i * ldh;
            r = __ldg(h); gch = __ldg(h + 1); b = __ldg(h + 2); sig = __ldg(h + 3);
            dist = __ldg(dists + i);
        }
        float a = 1.0f - expf((0.0f - sig) * dist);
        float q = (1.0f - a) + 1e-10f;
        float p = warp_incl_prod(valid ? q : 1.0f, lane) * carry;
        carry = __shfl_sync(0xffffffffu, p, 31);
        float T = (s == 0) ? 1.0f : p;
        float w = a * T;
        if (valid) {
            if (rgba) *reinterpret_cast<float4 *>(rgba + i * 4) = make_float4(r, gch, b, sig);
            if (alpha) alpha[i] = a;
            if (cumprod) cumprod[i] = T;
            if (weights) weights[i] = w;
            c0 = fmaf(w, r, c0); c1 = fmaf(w, gch, c1); c2 = fmaf(w, b, c2);
            if (EXT) {
                c3 += w;
                if (k.depth) c4 = fmaf(w, sample_depth<VIEWS>(k, ray, s, S), c4);
            }
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        c0 += __shfl_xor_sync(0xffffffffu, c0, d);
        c1 += __shfl_xor_sync(0xffffffffu, c1, d);
        c2 += __shfl_xor_sync(0xffffffffu, c2, d);
        if (EXT) {
            c3 += __shfl_xor_sync(0xffffffffu, c3, d);
            c4 += __shfl_xor_sync(0xffffffffu, c4, d);
        }
    }
    if (lane == 0) {
        float *c = color + (size_t)ray * 3;
        if (EXT) {
            if (k.acc) k.acc[ray] = c3;
            if (k.depth) k.depth[ray] = c4;
            if (k.background) {
                const float tr = 1.0f - c3;   // the light that reaches the background
                c0 = fmaf(tr, k.bg0, c0); c1 = fmaf(tr, k.bg1, c1); c2 = fmaf(tr, k.bg2, c2);
            }
        }
        if (color_accumulate) { c0 += c[0]; c1 += c[1]; c2 += c[2]; }
        c[0] = c0; c[1] = c1; c[2] = c2;
        float sse = 0.0f;
        if (target) {
            const float *tg = target + (size_t)ray * 3;
            float d0 = c0 - tg[0], d1 = c1 - tg[1], d2 = c2 - tg[2];
            sse = d0 * d0 + d1 * d1 + d2 * d2;
        }
        if (ray_sse) ray_sse[ray] = sse;
    }
}

// Backward, unit seed (SURVEY.md Appendix B; the reverse sweep multiplies, never divides by q):
//   dcol = 2 (color - target); d_rgb_s = w_s dcol; d_w_s = <rgb_s, dcol>
//   d_alpha_s = d_w_s T_s - dq_s;  dT_s = d_w_s alpha_s (s >= 1), dT_0 = 0
//   G_s = dT_s + q_{s+1} G_{s+1}  (G_S = 0);  dq_s = Cpre_{s-1} G_s, Cpre_{-1} = 1
//   e = expf(-sigma dist); d_sigma = d_alpha e dist; d_dist = d_alpha e sigma
// EXT with a background: d_w_s = <rgb_s - bg, dcol> (the background term's adjoint; bg itself gets none)
template <bool EXT>
__global__ void __launch_bounds__(COMP_WARPS * 32)
composite_bwd_kernel(const float *__restrict__ head, int ldh, const float *__restrict__ dists,
                     const float *__restrict__ target, const float *__restrict__ color, int R,
                     int S, float *__restrict__ dZ, int ldz, int out_dim,
                     float *__restrict__ d_dists_u, float *__restrict__ d_color_u, const CompK k)
{
    __shared__ float carry_in[COMP_WARPS][COMP_MAX_CHUNKS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ray = blockIdx.x * COMP_WARPS + warp;
    if (ray >= R) return;
    const int n_chunks = (S + 31) / 32;
    // pass 1: prefix product entering each chunk
    float carry = 1.0f;
    for (int c = 0; c < n_chunks; ++c) {
        const int s = c * 32 + lane;
        const size_t i = (size_t)ray * S + s;
        float q = 1.0f;
        if (s < S) {
            float sig = __ldg(head + i * ldh + 3), dist = __ldg(dists + i);
            float a = 1.0f - expf((0.0f - sig) * dist);
            q = (1.0f - a) + 1e-10f;
        }
        if (lane == 0) carry_in[warp][c] = carry;
        float p = warp_incl_prod(q, lane) * carry;
        carry = __shfl_sync(0xffffffffu, p, 31);
    }
    __syncwarp();
    float dc0, dc1, dc2;
    {
        const float *cl = color + (size_t)ray * 3, *tg = target + (size_t)ray * 3;
        dc0 = 2.0f * (cl[0] - tg[0]); dc1 = 2.0f * (cl[1] - tg[1]); dc2 = 2.0f * (cl[2] - tg[2]);
        if (lane == 0 && d_color_u) {
            d_color_u[(size_t)ray * 3 + 0] = dc0;
            d_color_u[(size_t)ray * 3 + 1] = dc1;
            d_color_u[(size_t)ray * 3 + 2] = dc2;
        }
    }
    // pass 2: chunks in reverse
    float G_next = 0.0f; // G of the first sample of the following chunk
    float q_next = 0.0f; // q of the first sample of the following chunk
    for (int c = n_chunks - 1; c >= 0; --c) {
        const int s = c * 32 + lane;
        const bool valid = s < S;
        const size_t i = (size_t)ray * S + s;
        float r = 0.f, gch = 0.f, b = 0.f, sig = 0.f, dist = 0.f;
        if (valid) {
            const float *h = head + i * ldh;
            r = __ldg(h); gch = __ldg(h + 1); b = __ldg(h + 2); sig = __ldg(h + 3);
            dist = __ldg(dists + i);
        }
        const float e = expf((0.0f - sig) * dist);
        const float a = 1.0f - e;
        const float q = valid ? (1.0f - a) + 1e-10f : 1.0f;
        const float cin = carry_in[warp][c];
        const float Cpre = warp_incl_prod(q, lane) * cin; // true inclusive product
        const float T = (s == 0) ? 1.0f : Cpre;
        const float w = a * T;
        const float d_w = (EXT && k.background) ? (r - k.bg0) * dc0 + (gch - k.bg1) * dc1 + (b - k.bg2) * dc2
                                                : r * dc0 + gch * dc1 + b * dc2;
        const float dT = (s == 0 || !valid) ? 0.0f : d_w * a;
        // affine suffix scan: G_s = A_s + B_s * G_next
        float qn = __shfl_down_sync(0xffffffffu, q, 1);
        if (lane == 31) qn = q_next;
        float A = dT, B = (valid && s + 1 < S) ? qn : 0.0f;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            float A2 = __shfl_down_sync(0xffffffffu, A, d);
            float B2 = __shfl_down_sync(0xffffffffu, B, d);
            if (lane + d < 32) { A = fmaf(B, A2, A); B = B * B2; }
        }
        const float G = fmaf(B, G_next, A);
        float Cm1 = __shfl_up_sync(0xffffffffu, Cpre, 1);
        if (lane == 0) Cm1 = cin;
        const float dq = Cm1 * G;
        const float d_alpha = d_w * T - dq;
        if (valid) {
            float *z = dZ + i * ldz;
            z[0] = (w * dc0) * (r * (1.0f - r));
            z[1] = (w * dc1) * (gch * (1.0f - gch));
            z[2] = (w * dc2) * (b * (1.0f - b));
            z[3] = (sig > 0.0f) ? d_alpha * e * dist : 0.0f;
            for (int j = 4; j < out_dim; ++j) z[j] = 0.0f;
            if (d_dists_u) d_dists_u[i] = d_alpha * e * sig;
        }
        G_next = __shfl_sync(0xffffffffu, G, 0);
        q_next = __shfl_sync(0xffffffffu, q, 0);
    }
}

// ------------------------------------------------------------------------------------------------
__global__ void sum_kernel(const float *__restrict__ v, long long n, float *__restrict__ out)
{
    __shared__ float sm[32];
    float s = 0.0f;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) s += v[i];
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x < 32) {
        s = (threadIdx.x < (blockDim.x >> 5)) ? sm[threadIdx.x] : 0.0f;
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        if (threadIdx.x == 0) out[0] = s;
    }
}

__global__ void fit_loss_kernel(const float *__restrict__ pred, int ldp,
                                const float *__restrict__ target, int R, int Wt,
                                float *__restrict__ ray_sse)
{
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    float s = 0.0f;
    for (int c = 0; c < Wt; ++c) {
        float d = pred[(size_t)r * ldp + c] - target[(size_t)r * Wt + c];
        s = fmaf(d, d, s);
    }
    ray_sse[r] = s;
}

__global__ void fit_head_bwd_kernel(const float *__restrict__ pred, int ldp,
                                    const float *__restrict__ target, int R, int Wt, int rows,
                                    int out_dim, float *__restrict__ dZ, int ldz,
                                    float *__restrict__ d_color_u)
{
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)rows * out_dim) return;
    int i = (int)(e / out_dim), j = (int)(e % out_dim);
    float v = 0.0f;
    if (i < R && j < Wt) {
        float y = pred[(size_t)i * ldp + j];
        float dc = 2.0f * (y - target[(size_t)i * Wt + j]);
        if (d_color_u) d_color_u[(size_t)i * Wt + j] = dc;
        v = dc * (y * (1.0f - y));
    }
    dZ[(size_t)i * ldz + j] = v;
}

__global__ void fill_kernel(float *p, size_t n, float v)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

__global__ void axpy2d_kernel(float *__restrict__ dst, long long ldd, const float *__restrict__ src,
                              long long lds, long long rows, int cols, float sign,
                              float seed_value, const float *__restrict__ seed_dev)
{
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rows * cols) return;
    long long i = e / cols;
    int j = (int)(e % cols);
    float scale = sign * seed_value * (seed_dev ? __ldg(seed_dev) : 1.0f);
    dst[i * ldd + j] += scale * src[i * lds + j];
}

} // namespace

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
int lnb_launch_row_gemm(lnb_ctx *ctx, const lnb_gemm_args &g)
{
    if (g.rows <= 0 || g.n_dim <= 0) return LNB_OK;
    if (g.n_dim >= 64 && g.k_dim >= 64 && g.k_dim % 16 == 0 && g.lda % 4 == 0 && ((uintptr_t)g.A & 15) == 0 && g.rows >= 128) {
        dim3 grid((unsigned)((g.rows + 127) / 128), (unsigned)((g.n_dim + 127) / 128));
        sgemm128_kernel<<<grid, 256, 0, ctx->stream>>>(g);
        LNB_CHECK_LAUNCH();
        return LNB_OK;
    }
    if (g.n_dim <= 32) {
        dim3 grid((unsigned)((g.rows + 127) / 128), (unsigned)((g.n_dim + 31) / 32));
        row_gemm_kernel<128, 32><<<grid, 256, 0, ctx->stream>>>(g);
    } else {
        dim3 grid((unsigned)((g.rows + 63) / 64), (unsigned)((g.n_dim + 63) / 64));
        row_gemm_kernel<64, 64><<<grid, 256, 0, ctx->stream>>>(g);
    }
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_dw_partials(lnb_ctx *ctx, const float *H, int ldh, const float *dZ, int ldz,
                           float *partial, int in_dim, int out_dim, int rows, int n_chunks)
{
    if (rows <= 0 || n_chunks <= 0) return LNB_OK;
    long long rpc = ((long long)rows + n_chunks - 1) / n_chunks;
    rpc = (rpc + 31) / 32 * 32;
    if (out_dim <= 32 && in_dim + 1 <= 64) {
        const int kp = (in_dim + 1 + 15) / 16 * 16;
#define LNB_DWR(KPV) dw_rows_kernel<KPV><<<(unsigned)n_chunks, 256, 0, ctx->stream>>>(H, ldh, dZ, ldz, partial, in_dim, out_dim, rows, rpc)
        if (kp == 16) LNB_DWR(16);
        else if (kp == 32) LNB_DWR(32);
        else if (kp == 48) LNB_DWR(48);
        else LNB_DWR(64);
#undef LNB_DWR
        LNB_CHECK_LAUNCH();
        return LNB_OK;
    }
    if (in_dim >= 64 && out_dim >= 64 && in_dim % 4 == 0 && out_dim % 4 == 0 && ldh % 4 == 0 && ldz % 4 == 0 && ((uintptr_t)H & 15) == 0 &&
        ((uintptr_t)dZ & 15) == 0) {
        rpc = (rpc + 15) / 16 * 16;
        dim3 grid((unsigned)n_chunks, (unsigned)((in_dim + 127) / 128), (unsigned)((out_dim + 127) / 128));
        dw128_kernel<<<grid, 256, 0, ctx->stream>>>(H, ldh, dZ, ldz, partial, in_dim, out_dim, rows, rpc);
        LNB_CHECK_LAUNCH();
        return LNB_OK;
    }
    const int tj = out_dim <= 32 ? 2 : 4;
    const int tk = (in_dim + 1) <= 32 ? 2 : ((in_dim + 1) <= 48 ? 3 : 4);
    dim3 grid((unsigned)n_chunks, (unsigned)((in_dim + 1 + 16 * tk - 1) / (16 * tk)),
              (unsigned)((out_dim + 16 * tj - 1) / (16 * tj)));
#define LNB_DW(TK, TJ)                                                                          \
    dw_partials_kernel<TK, TJ><<<grid, 256, 0, ctx->stream>>>(H, ldh, dZ, ldz, partial, in_dim,  \
                                                              out_dim, rows, rpc)
    if (tk == 2 && tj == 2) LNB_DW(2, 2);
    else if (tk == 3 && tj == 2) LNB_DW(3, 2);
    else if (tk == 4 && tj == 2) LNB_DW(4, 2);
    else if (tk == 2 && tj == 4) LNB_DW(2, 4);
    else if (tk == 3 && tj == 4) LNB_DW(3, 4);
    else LNB_DW(4, 4);
#undef LNB_DW
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_dw_reduce(lnb_ctx *ctx, const float *partial, int n_chunks, int in_dim,
                         int out_dim, float *d_w, int ldw, float *d_b, float seed_value,
                         const float *seed_dev)
{
    long long n = (long long)(in_dim + 1) * out_dim;
    unsigned blocks = (unsigned)((n * 32 + 255) / 256);
    dw_reduce_kernel<<<blocks, 256, 0, ctx->stream>>>(partial, n_chunks, in_dim, out_dim, d_w, ldw,
                                                      d_b, seed_value, seed_dev);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

static CompK comp_k(const lnb_comp_args *cx)
{
    CompK k{};
    if (!cx) return k;
    k.background = cx->background;
    k.bg0 = cx->bg[0]; k.bg1 = cx->bg[1]; k.bg2 = cx->bg[2];
    k.acc = cx->acc; k.depth = cx->depth;
    k.t = cx->t; k.t_f64 = cx->t_f64;
    if (cx->cam) { k.cam_mode = 1; k.cam = make_cam_dev(*cx->cam, cx->views); }
    return k;
}

int lnb_launch_composite_fwd(lnb_ctx *ctx, const float *head, int ldh, const float *dists,
                             const float *target, int R, int S, float *rgba, float *alpha,
                             float *cumprod, float *weights, float *color, int color_accumulate,
                             float *ray_sse, const lnb_comp_args *cx)
{
    if (R <= 0) return LNB_OK;
    auto kern = lnb_cx_extras(cx) ? (cx->views ? composite_fwd_kernel<true, true> : composite_fwd_kernel<true>) : composite_fwd_kernel<false>;
    kern<<<(R + COMP_WARPS - 1) / COMP_WARPS, COMP_WARPS * 32, 0, ctx->stream>>>(
        head, ldh, dists, target, R, S, rgba, alpha, cumprod, weights, color, color_accumulate,
        ray_sse, comp_k(cx));
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_composite_bwd(lnb_ctx *ctx, const float *head, int ldh, const float *dists,
                             const float *target, const float *color, int R, int S, float *dZ_head,
                             int ldz, int out_dim, float *d_dists_u, float *d_color_u, const lnb_comp_args *cx)
{
    if (R <= 0) return LNB_OK;
    LNB_ARG(S <= 32 * COMP_MAX_CHUNKS, "samples per ray > 2048");
    auto kern = (cx && cx->background) ? composite_bwd_kernel<true> : composite_bwd_kernel<false>;
    kern<<<(R + COMP_WARPS - 1) / COMP_WARPS, COMP_WARPS * 32, 0, ctx->stream>>>(
        head, ldh, dists, target, color, R, S, dZ_head, ldz, out_dim, d_dists_u, d_color_u, comp_k(cx));
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_sum(lnb_ctx *ctx, const float *v, long long n, float *out)
{
    sum_kernel<<<1, 1024, 0, ctx->stream>>>(v, n, out);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_fit_loss(lnb_ctx *ctx, const float *pred, int ldp, const float *target, int R,
                        int Wt, float *ray_sse)
{
    if (R <= 0) return LNB_OK;
    fit_loss_kernel<<<(R + 255) / 256, 256, 0, ctx->stream>>>(pred, ldp, target, R, Wt, ray_sse);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_fit_head_bwd(lnb_ctx *ctx, const float *pred, int ldp, const float *target, int R,
                            int Wt, int rows, int out_dim, float *dZ, int ldz, float *d_color_u)
{
    long long n = (long long)rows * out_dim;
    if (n <= 0) return LNB_OK;
    fit_head_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(
        pred, ldp, target, R, Wt, rows, out_dim, dZ, ldz, d_color_u);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_fill(lnb_ctx *ctx, float *p, size_t n, float v)
{
    if (n == 0) return LNB_OK;
    fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(p, n, v);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_axpy2d(lnb_ctx *ctx, float *dst, long long ldd, const float *src, long long lds,
                      long long rows, int cols, float sign, float seed_value,
                      const float *seed_dev)
{
    long long n = rows * cols;
    if (n <= 0) return LNB_OK;
    axpy2d_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(
        dst, ldd, src, lds, rows, cols, sign, seed_value, seed_dev);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}
