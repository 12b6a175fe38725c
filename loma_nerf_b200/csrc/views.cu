// views.cu -- the per-step batch of a device-resident scene (lnb_views_draw, include/loma_nerf_b200.h): which view and pixel
// each ray looks through, and its target colour, drawn on the device from a counter the draw itself advances, so that a
// captured graph of (draw + step) trains on a new batch at every replay.
#include "lnb_internal.h"

namespace {

// z(k, i) = mix(seed + 0x9E3779B97F4A7C15 * (k * 2^32 + i + 1)), mix the SplitMix64 finaliser (as lnb_uniform's)
__host__ __device__ inline unsigned long long draw_z(unsigned long long seed, unsigned long long k, unsigned long long i)
{
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * ((k << 32) + i + 1ull);
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

constexpr unsigned long long PICK_VIEW = 0xFFFFFFFFull, PICK_SEED = 0xFFFFFFFEull;

// One thread per ray.  Every block reads k = counter[0] first; the last block to take a ticket (counter[1]) writes k + 1 and
// resets the ticket, so no block can see the advanced counter.  No griddepcontrol.launch_dependents: a dependent launched
// with programmatic serialization (the fused train kernel, which builds its first tile's inputs before it waits) starts only
// when this grid has completed and its batch is visible.
__global__ void views_draw_kernel(const float *__restrict__ images, int n_views, long long P, int R, int one_view,
                                  unsigned long long seed, unsigned long long *counter, int *__restrict__ view,
                                  int *__restrict__ pixels, float *__restrict__ target, unsigned long long *step_seed)
{
    __shared__ unsigned long long k_s;
    if (threadIdx.x == 0) k_s = *(volatile unsigned long long *)counter;
    __syncthreads();
    const unsigned long long k = k_s;
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < R) {
        long long v, q;
        if (one_view) {
            v = (long long)__umul64hi(draw_z(seed, k, PICK_VIEW), (unsigned long long)n_views);
            q = (long long)__umul64hi(draw_z(seed, k, (unsigned long long)r), (unsigned long long)P);
        } else {
            const long long g = (long long)__umul64hi(draw_z(seed, k, (unsigned long long)r), (unsigned long long)n_views * (unsigned long long)P);
            v = g / P;
            q = g - v * P;
        }
        view[r] = (int)v;
        pixels[r] = (int)q;
        const float *src = images + ((size_t)v * (size_t)P + (size_t)q) * 3;
        target[(size_t)r * 3] = src[0];
        target[(size_t)r * 3 + 1] = src[1];
        target[(size_t)r * 3 + 2] = src[2];
    }
    if (r == 0 && step_seed) *step_seed = draw_z(seed, k, PICK_SEED);
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(counter + 1, 1ull) == (unsigned long long)gridDim.x - 1) {
            counter[0] = k + 1;
            counter[1] = 0;
        }
    }
}

} // namespace

extern "C" unsigned long long lnb_views_pick(unsigned long long seed, unsigned long long k, unsigned long long i, unsigned long long n)
{
    return (unsigned long long)(((unsigned __int128)draw_z(seed, k, i) * n) >> 64);
}

extern "C" int lnb_views_draw(lnb_ctx *ctx, const float *images, int n_views, long long P, int R, int one_view,
                              unsigned long long seed, unsigned long long *counter, int *view, int *pixels, float *target,
                              unsigned long long *step_seed)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(n_views >= 1 && P >= 1 && P < (1ll << 31) && R >= 0 && (long long)R < (long long)PICK_SEED, "views_draw: sizes");
    LNB_ARG(images && counter && (R == 0 || (view && pixels && target)), "views_draw: null pointer");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    const int blocks = R > 0 ? (R + 255) / 256 : 1;   // an empty batch still advances the counter and writes the seed
    views_draw_kernel<<<blocks, 256, 0, ctx->stream>>>(images, n_views, P, R, one_view, seed, counter, view, pixels, target, step_seed);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}
