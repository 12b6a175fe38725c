// camera.cuh -- device-side ray generation and sample depths (lnb_camera, include/loma_nerf_b200.h): get_rays
// (/root/reference/train_nerf.py:23-62) and the sample construction (train_nerf.py:289-311) without any per-ray or
// per-sample input.  Two forms: float64 like numpy forms the values (exact path, encode.cu) and float32 (tensor-core
// path, fused_tc.cu).  Shared by the translation units that generate rays.
#pragma once
#include "lnb_internal.h"

// kernel-parameter copy of an lnb_camera (passed by value)
struct CamDev {
    double c2w[12];
    double fx, fy, cx, cy, step, near, far;   // step = 1 / (width - 1): numpy linspace(0, 1, width) = arange * step, last = 1
    long long first_pixel;
    const int *pixels;
    unsigned long long seed;
    int width, height, stratified;
    // views mode (lnb_views; poses == NULL: camera mode): pixels is the views' pixel list
    const double *poses;
    const int *view;
    const unsigned long long *seed_dev;
    long long P;
    int n_views;
};

inline CamDev make_cam_dev(const lnb_camera &c)
{
    CamDev d{};
    for (int i = 0; i < 12; ++i) d.c2w[i] = c.c2w[i];
    d.fx = c.fx; d.fy = c.fy; d.cx = c.cx; d.cy = c.cy;
    d.step = c.width > 1 ? 1.0 / (double)(c.width - 1) : 0.0;
    d.near = c.near; d.far = c.far;
    d.first_pixel = c.first_pixel; d.pixels = c.pixels; d.seed = c.seed;
    d.width = c.width; d.height = c.height; d.stratified = c.stratified;
    return d;
}

// The camera fields a views batch shares with camera mode (c2w unused, pixels = the views' pixel list)
inline lnb_camera views_camera(const lnb_views &v)
{
    lnb_camera c{};
    c.fx = v.fx; c.fy = v.fy; c.cx = v.cx; c.cy = v.cy;
    c.width = v.width; c.height = v.height;
    c.pixels = v.pixels;
    c.near = v.near; c.far = v.far;
    c.stratified = v.stratified; c.seed = v.seed;
    return c;
}
inline CamDev make_cam_dev(const lnb_camera &c, const lnb_views *v)
{
    CamDev d = make_cam_dev(c);
    if (v) {
        d.poses = v->poses; d.view = v->view; d.seed_dev = v->seed_dev;
        d.P = (long long)v->width * v->height; d.n_views = v->n_views;
    }
    return d;
}

// SplitMix64 finaliser over (seed, pixel, sample): 24 uniform bits
__host__ __device__ inline unsigned lnb_uniform_bits(unsigned long long seed, long long pixel, int s)
{
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * ((unsigned long long)pixel * 4096ull + (unsigned long long)s + 1ull);
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
    z ^= z >> 27; z *= 0x94D049BB133111EBull;
    z ^= z >> 31;
    return (unsigned)(z >> 40);
}

__device__ __forceinline__ long long cam_pixel(const CamDev &c, long long ray) { return c.pixels ? (long long)__ldg(c.pixels + ray) : c.first_pixel + ray; }

// Views mode: camera mode's camera of ray r (its pose in c2w, its jitter seed seed') in cr, with its pixel q and jitter key
// g = view[r] * P + q.  false when view[r] or pixels[r] is out of range (c2w is then the table's first pose: nothing outside
// the table is read; the caller makes the ray NaN).
__device__ __forceinline__ bool views_ray(const CamDev &c, long long r, CamDev &cr, long long &q, long long &g)
{
    const int v = __ldg(c.view + r), p = __ldg(c.pixels + r);
    const bool ok = v >= 0 && v < c.n_views && p >= 0 && p < c.P;
    const double *m = c.poses + 12 * (long long)(ok ? v : 0);
    cr = c;
#pragma unroll
    for (int i = 0; i < 12; ++i) cr.c2w[i] = __ldg(m + i);
    if (c.seed_dev) cr.seed = *c.seed_dev;
    q = p;
    g = (long long)v * c.P + p;
    return ok;
}

// float64: the operation order of get_rays (linspace value, (i - cx) / fx, dirs @ R^T as a plain k-sum)
__device__ __forceinline__ void cam_ray_f64(const CamDev &c, long long q, double o[3], double d[3])
{
    const int col = (int)(q % c.width), row = (int)(q / c.width);
    const double i = col == c.width - 1 ? 1.0 : col * c.step, j = row == c.width - 1 ? 1.0 : row * c.step;
    const double dx = (i - c.cx) / c.fx, dy = -(j - c.cy) / c.fy, dz = -1.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        d[k] = __dadd_rn(__dadd_rn(__dmul_rn(dx, c.c2w[4 * k]), __dmul_rn(dy, c.c2w[4 * k + 1])), __dmul_rn(dz, c.c2w[4 * k + 2]));
        o[k] = c.c2w[4 * k + 3];
    }
}
// depth of sample s of an S-sample ray: numpy linspace(near, far, S) = near + s * ((far - near) / (S - 1)), last = far
__device__ __forceinline__ double cam_t_f64(const CamDev &c, long long q, int s, int S)
{
    // explicit roundings (no FMA contraction): numpy's linspace is arange * step + start, two rounded operations
    if (!c.stratified) return (s == S - 1 && S > 1) ? c.far : __dadd_rn(__dmul_rn((double)s, (c.far - c.near) / (double)(S > 1 ? S - 1 : 1)), c.near);
    const double u = (double)lnb_uniform_bits(c.seed, q, s) * (1.0 / 16777216.0);
    return __dadd_rn(c.near, __ddiv_rn(__dmul_rn((double)s + u, c.far - c.near), (double)S));
}
