// sample_pdf.cu -- hierarchical sampling on the device: fine depths drawn by inverse transform from the piecewise-constant
// PDF a coarse pass's compositing weights define along each ray (lnb_sample_pdf, include/loma_nerf_b200.h).
// Every operation is float64 and explicitly rounded (__d*_rn: no FMA contraction), the cumulative sum runs in order, so a
// row equals the header's numpy statement of the rule bit for bit.
#include <math_constants.h>

#include "camera.cuh"
#include "lnb_internal.h"

namespace {

constexpr int SAMPLE_PDF_MAX = 4096;   // S + n_fine: also lnb_uniform's counter space per ray

// One CTA per ray.  Shared memory: key[P], the row's S + n_fine output values padded with +inf to the power of two P,
// then cdf[S - 1].  key[0, S) holds the coarse depths (the bins are formed from them), key[S, S + n_fine) the samples.
__global__ void __launch_bounds__(512) sample_pdf_kernel(const double *__restrict__ t, const float *__restrict__ w, int S,
                                                         int n_fine, int P, int stratified, unsigned long long seed,
                                                         long long ray0, double *__restrict__ out)
{
    extern __shared__ double sm[];
    double *key = sm, *cdf = sm + P;
    const long long r = blockIdx.x;
    const int M = S + n_fine, nb = S - 1, tid = threadIdx.x, nt = blockDim.x;
    for (int k = tid; k < S; k += nt) key[k] = t[r * S + k];
    for (int k = M + tid; k < P; k += nt) key[k] = CUDART_INF;
    for (int j = tid; j < S - 2; j += nt) cdf[j + 1] = __dadd_rn((double)w[r * S + j + 1], 1e-5);   // v_j
    __syncthreads();
    if (tid == 0) {   // c_{j+1} = c_j + v_j in order: a parallel scan would reorder the additions
        double c = 0.0;
        cdf[0] = 0.0;
#pragma unroll 4
        for (int j = 1; j < nb; ++j) { c = __dadd_rn(c, cdf[j]); cdf[j] = c; }
    }
    __syncthreads();
    const double total = cdf[nb - 1];
    __syncthreads();
    for (int k = tid; k < nb; k += nt) cdf[k] = __ddiv_rn(cdf[k], total);   // cdf_0 = 0, cdf_{S-2} = 1 exactly
    __syncthreads();
    const double step = n_fine > 1 ? __ddiv_rn(1.0, (double)(n_fine - 1)) : 0.0;
    for (int i = tid; i < n_fine; i += nt) {
        double u;
        if (stratified)
            u = __ddiv_rn(__dadd_rn((double)i, (double)lnb_uniform_bits(seed, ray0 + r, i) * (1.0 / 16777216.0)), (double)n_fine);
        else   // np.linspace(0, 1, n_fine): i * (1 / (n - 1)), the last value exactly 1
            u = (n_fine > 1 && i == n_fine - 1) ? 1.0 : __dmul_rn((double)i, step);
        int lo = 0, hi = nb;   // ind = #{k : cdf_k <= u}, searchsorted(side="right")
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (cdf[mid] <= u) lo = mid + 1; else hi = mid;
        }
        const int below = lo - 1 > 0 ? lo - 1 : 0, above = lo < nb - 1 ? lo : nb - 1;
        const double mb = __dmul_rn(0.5, __dadd_rn(key[below], key[below + 1]));
        const double ma = __dmul_rn(0.5, __dadd_rn(key[above], key[above + 1]));
        double d = __dsub_rn(cdf[above], cdf[below]);
        if (d < 1e-5) d = 1.0;
        const double tau = __ddiv_rn(__dsub_rn(u, cdf[below]), d);
        key[S + i] = __dadd_rn(mb, __dmul_rn(tau, __dsub_rn(ma, mb)));
    }
    __syncthreads();
    // bitonic sort of key[0, P) ascending: the x_i need not be monotone (interpolation may overshoot by an ulp), nor the t_k
    for (int k = 2; k <= P; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < P / 2; i += nt) {
                const int a = 2 * i - (i & (j - 1)), b = a + j;
                const double x = key[a], y = key[b];
                if ((x > y) == ((a & k) == 0)) { key[a] = y; key[b] = x; }
            }
            __syncthreads();
        }
    for (int k = tid; k < M; k += nt) out[r * M + k] = key[k];
}

} // namespace

extern "C" int lnb_sample_pdf(lnb_ctx *ctx, const double *t, const float *w, int R, int S, int n_fine, int stratified,
                              unsigned long long seed, long long ray0, double *out)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(R == 0 || (t && w && out), "sample_pdf: t, weights and out are required");
    LNB_ARG(R >= 0 && S >= 3 && n_fine >= 1 && (long long)S + n_fine <= SAMPLE_PDF_MAX,
            "sample_pdf: needs R >= 0, S >= 3, n_fine >= 1 and S + n_fine <= 4096");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    if (R == 0) return LNB_OK;
    int P = 2;
    while (P < S + n_fine) P <<= 1;
    const int threads = P / 2 < 32 ? 32 : (P / 2 > 512 ? 512 : P / 2);
    const size_t smem = (size_t)(P + S - 1) * sizeof(double);
    if (smem > 48 * 1024)
        LNB_CUDA(cudaFuncSetAttribute(sample_pdf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sample_pdf_kernel<<<(unsigned)R, threads, smem, ctx->stream>>>(t, w, S, n_fine, P, stratified != 0, seed, ray0, out);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}
