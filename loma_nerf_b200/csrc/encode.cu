// encode.cu -- sample generation and positional encoding on the device.
// Reference: /root/reference/pos_encoding.py:4-70 (float64 sin/cos of 2^i x, cast to float32,
// feature index = slot*F + coord) and train_nerf.py:289-311 (pts = o + d t, dists, last = 1e8).
// The exact variants here compute in float64 like the reference; the fused tensor-core path has
// its own fp32 prologue (fused_tc.cu) with the error bound stated in DESIGN.md.
#include <cuda_bf16.h>

#include "camera.cuh"
#include "lnb_internal.h"

namespace {

__global__ void pos_encoding_kernel(const double *__restrict__ x, long long n, int F, int E,
                                    float *__restrict__ out)
{
    // one thread per (point, coord): writes 1 + 2E features with stride F
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * F) return;
    long long p = e / F;
    int f = (int)(e % F);
    const int C = F * (1 + 2 * E);
    double v = x[e];
    float *o = out + p * C;
    o[f] = (float)v;
    double freq = 1.0;
    for (int i = 0; i < E; ++i) {
        double s, c;
        sincos(freq * v, &s, &c);
        o[(2 * i + 1) * F + f] = (float)s;
        o[(2 * i + 2) * F + f] = (float)c;
        freq *= 2.0;
    }
}

// slot 0 = v and slots 2i+1 / 2i+2 = sin / cos(2^i v), i < E, of one coordinate f: feature 3 * slot + f of the row at o.
// fp32 features: float64 sin / cos, rounded once (pos_encoding.py:38-70).
__device__ __forceinline__ void encode_coord(double v, int E, int f, float *o)
{
    o[f] = (float)v;
    double freq = 1.0;
    for (int i = 0; i < E; ++i) {
        double sn, cs;
        sincos(freq * v, &sn, &cs);
        o[(2 * i + 1) * 3 + f] = (float)sn;
        o[(2 * i + 2) * 3 + f] = (float)cs;
        freq *= 2.0;
    }
}
// the wide tensor-core path's bf16 operand: the float value rounded once more
__device__ __forceinline__ void encode_coord(double v, int E, int f, __nv_bfloat16 *o)
{
    o[f] = __float2bfloat16_rn((float)v);
    double freq = 1.0;
    for (int i = 0; i < E; ++i) {
        // the argument is formed in double and rounded once (error <= 2^-24 * |arg|, far below the bf16 step of
        // the result); fp32 sincosf with full range reduction instead of the double one: B200's fp64 rate is low
        float sn, cs;
        sincosf((float)(freq * v), &sn, &cs);
        o[(2 * i + 1) * 3 + f] = __float2bfloat16_rn(sn);
        o[(2 * i + 2) * 3 + f] = __float2bfloat16_rn(cs);
        freq *= 2.0;
    }
}

// coordinate f of the unit view direction d / |d|, |d| = sqrt((d0^2 + d1^2) + d2^2) in float64 with every operation
// rounded (no FMA contraction): what numpy computes elementwise
__device__ __forceinline__ double unit_coord(const double (&d)[3], int f)
{
    const double n2 = __dadd_rn(__dadd_rn(__dmul_rn(d[0], d[0]), __dmul_rn(d[1], d[1])), __dmul_rn(d[2], d[2]));
    return __ddiv_rn(d[f], __dsqrt_rn(n2));
}

// one thread per (sample, coordinate).  Ed >= 0 appends the view direction's encoding PE(u, Ed) after PE(x, E).
// CAM: 0 rays mode, 1 camera mode, 2 views mode (a pose per ray; a ray with an out-of-range index gets NaN features and dists)
template <typename T, int CAM>
__global__ void sample_encode_kernel(const T *__restrict__ o, const T *__restrict__ d,
                                     const T *__restrict__ t, const CamDev cam, int R, int S, int E, int Ed,
                                     float *__restrict__ X, float *__restrict__ dists, __nv_bfloat16 *__restrict__ Xb, int ldb)
{
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)R * S * 3) return;
    long long smp = e / 3;
    int f = (int)(e % 3);
    int r = (int)(smp / S), s = (int)(smp % S);
    const int P = 3 * (1 + 2 * E), C = P + (Ed >= 0 ? 3 * (1 + 2 * Ed) : 0);
    double tt, tnext = 0.0, v, dd[3];
    if (CAM == 2) {   // views mode: camera mode's ray of pixels[r] under its own pose, jitter keyed by g
        CamDev cr;
        long long q, g;
        const bool ok = views_ray(cam, r, cr, q, g);
        double oo[3];
        cam_ray_f64(cr, q, oo, dd);
        tt = cam_t_f64(cr, g, s, S);
        if (s + 1 < S) tnext = cam_t_f64(cr, g, s + 1, S);
        if (!ok) tt = tnext = __longlong_as_double(0x7ff8000000000000ll);
        v = oo[f] + dd[f] * tt;
    } else if (CAM) {   // rays and depths from the pose (camera.cuh): float64 values in get_rays' / linspace's operation order
        const long long q = cam_pixel(cam, r);
        double oo[3];
        cam_ray_f64(cam, q, oo, dd);
        tt = cam_t_f64(cam, q, s, S);
        if (s + 1 < S) tnext = cam_t_f64(cam, q, s + 1, S);
        v = oo[f] + dd[f] * tt;
    } else {
        tt = (double)t[smp];
        if (s + 1 < S) tnext = (double)t[smp + 1];
        v = (double)o[r * 3 + f] + (double)d[r * 3 + f] * tt;
        if (Ed >= 0)
            for (int k = 0; k < 3; ++k) dd[k] = (double)d[r * 3 + k];
    }
    if (Xb) {
        __nv_bfloat16 *x = Xb + smp * ldb;
        encode_coord(v, E, f, x);
        if (Ed >= 0) encode_coord(unit_coord(dd, f), Ed, f, x + P);
        if (f == 0)
            for (int c = C; c < ldb; ++c) x[c] = __float2bfloat16_rn(0.0f);
    } else {
        float *x = X + smp * C;
        encode_coord(v, E, f, x);
        if (Ed >= 0) encode_coord(unit_coord(dd, f), Ed, f, x + P);
    }
    if (f == 0 && dists) dists[smp] = (s + 1 < S || (CAM == 2 && tt != tt)) ? (float)(tnext - tt) : (float)1e8;
}

} // namespace

int lnb_launch_pos_encoding(lnb_ctx *ctx, const double *x, long long n, int F, int E, float *out)
{
    long long tot = n * F;
    if (tot <= 0) return LNB_OK;
    pos_encoding_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(x, n, F, E, out);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

int lnb_launch_sample_encode(lnb_ctx *ctx, const void *o, const void *d, const void *t, int f64,
                             int R, int S, int E, int Ed, float *X, float *dists)
{
    return lnb_launch_sample_encode_bf16(ctx, o, d, t, f64, R, S, E, Ed, X, dists, nullptr, 0);
}

// the same, writing either fp32 features X [N][C] or (Xb != NULL) bf16 rows Xb [N][ldb], zero beyond C
// (C = 3+6E, plus 3+6Ed with directions)
int lnb_launch_sample_encode_bf16(lnb_ctx *ctx, const void *o, const void *d, const void *t, int f64,
                                  int R, int S, int E, int Ed, float *X, float *dists, void *Xb, int ldb)
{
    long long tot = (long long)R * S * 3;
    if (tot <= 0) return LNB_OK;
    const unsigned blocks = (unsigned)((tot + 255) / 256);
    if (f64)
        sample_encode_kernel<double, 0><<<blocks, 256, 0, ctx->stream>>>((const double *)o, (const double *)d, (const double *)t, CamDev{}, R, S, E, Ed, X, dists, (__nv_bfloat16 *)Xb, ldb);
    else
        sample_encode_kernel<float, 0><<<blocks, 256, 0, ctx->stream>>>((const float *)o, (const float *)d, (const float *)t, CamDev{}, R, S, E, Ed, X, dists, (__nv_bfloat16 *)Xb, ldb);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

// camera mode: the same outputs with rays and depths generated from the pose (lnb_camera); views mode with views != NULL
int lnb_launch_camera_encode(lnb_ctx *ctx, const lnb_camera *cam, const lnb_views *views, int R, int S, int E, int Ed, float *X,
                             float *dists, void *Xb, int ldb)
{
    long long tot = (long long)R * S * 3;
    if (tot <= 0) return LNB_OK;
    const unsigned blocks = (unsigned)((tot + 255) / 256);
    if (views)
        sample_encode_kernel<double, 2><<<blocks, 256, 0, ctx->stream>>>(nullptr, nullptr, nullptr, make_cam_dev(*cam, views), R, S, E, Ed, X, dists, (__nv_bfloat16 *)Xb, ldb);
    else
        sample_encode_kernel<double, 1><<<blocks, 256, 0, ctx->stream>>>(nullptr, nullptr, nullptr, make_cam_dev(*cam), R, S, E, Ed, X, dists, (__nv_bfloat16 *)Xb, ldb);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

namespace {
// the rays and depths themselves (tests, and hosts that want them): o, d [R][3], t [R][S] float64
__global__ void camera_rays_kernel(const CamDev cam, int R, int S, double *__restrict__ o, double *__restrict__ d, double *__restrict__ t)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)R * S) return;
    const int r = (int)(e / S), s = (int)(e % S);
    const long long q = cam_pixel(cam, r);
    if (t) t[e] = cam_t_f64(cam, q, s, S);
    if (s == 0) {
        double oo[3], dd[3];
        cam_ray_f64(cam, q, oo, dd);
        for (int k = 0; k < 3; ++k) { if (o) o[r * 3 + k] = oo[k]; if (d) d[r * 3 + k] = dd[k]; }
    }
}
// views mode's rays and depths (lnb_views_rays); NaN for a ray with an out-of-range index
__global__ void views_rays_kernel(const CamDev cam, int R, int S, double *__restrict__ o, double *__restrict__ d, double *__restrict__ t)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)R * S) return;
    const int r = (int)(e / S), s = (int)(e % S);
    CamDev cr;
    long long q, g;
    const bool ok = views_ray(cam, r, cr, q, g);
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (t) t[e] = ok ? cam_t_f64(cr, g, s, S) : nan;
    if (s == 0) {
        double oo[3], dd[3];
        cam_ray_f64(cr, q, oo, dd);
        for (int k = 0; k < 3; ++k) { if (o) o[r * 3 + k] = ok ? oo[k] : nan; if (d) d[r * 3 + k] = ok ? dd[k] : nan; }
    }
}
__global__ void color_to_u8_kernel(const float *__restrict__ rgb, long long n, unsigned char *__restrict__ out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (unsigned char)__float2int_rn(255.0f * fminf(fmaxf(rgb[i], 0.0f), 1.0f));
}
} // namespace

extern "C" int lnb_camera_rays(lnb_ctx *ctx, const lnb_camera *cam, int R, int S, double *rays_o, double *rays_d, double *t)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(cam && R >= 0 && S >= 1, "camera_rays arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    const long long tot = (long long)R * S;
    if (tot <= 0) return LNB_OK;
    camera_rays_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(make_cam_dev(*cam), R, S, rays_o, rays_d, t);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

extern "C" int lnb_views_rays(lnb_ctx *ctx, const lnb_views *views, int R, int S, double *rays_o, double *rays_d, double *t)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(views && R >= 0 && S >= 1, "views_rays arguments");
    LNB_TRY(lnb_views_check(ctx, views, R, S));
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    const long long tot = (long long)R * S;
    if (tot <= 0) return LNB_OK;
    views_rays_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(make_cam_dev(views_camera(*views), views), R, S, rays_o, rays_d, t);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

extern "C" int lnb_color_to_u8(lnb_ctx *ctx, const float *rgb, long long n, unsigned char *out)
{
    if (!ctx) return LNB_ERR_ARG;
    LNB_ARG(rgb && out && n >= 0, "color_to_u8 arguments");
    if (cudaSetDevice(ctx->device) != cudaSuccess) return LNB_ERR_CUDA;
    if (n == 0) return LNB_OK;
    color_to_u8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(rgb, n, out);
    LNB_CHECK_LAUNCH();
    return LNB_OK;
}

extern "C" double lnb_uniform(unsigned long long seed, long long pixel, int s)
{
    return (double)lnb_uniform_bits(seed, pixel, s) * (1.0 / 16777216.0);
}
