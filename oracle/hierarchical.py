"""oracle/hierarchical.py -- float64 restatement of hierarchical sampling (lnb_sample_pdf, include/loma_nerf_b200.h).

The NeRF paper's sample_pdf draws fine depths by inverse transform from the piecewise-constant PDF a coarse pass's
compositing weights define along each ray.  sample_pdf_f64 states the library's rule in numpy, one float64 operation per
numpy operation (each rounded, no fused multiply-add), so the device's rows equal it bit for bit.  coarse_fine_f64 runs
the whole coarse-to-fine evaluation of one batch in float64.
"""
import numpy as np

from oracle import oracle as O
from oracle import viewdirs as V

_M64 = (1 << 64) - 1


def uniform(seed, q, s):
    """lnb_uniform(seed, q, s): the SplitMix64 finaliser over (seed, q, s), 24 bits in [0, 1)."""
    z = (int(seed) + 0x9E3779B97F4A7C15 * ((int(q) * 4096 + int(s) + 1) & _M64)) & _M64
    z ^= z >> 30
    z = (z * 0xBF58476D1CE4E5B9) & _M64
    z ^= z >> 27
    z = (z * 0x94D049BB133111EB) & _M64
    z ^= z >> 31
    return float(z >> 40) * (1.0 / 16777216.0)


def sample_positions(R, n_fine, stratified=False, seed=0, ray0=0):
    """u [R][n_fine]: np.linspace(0, 1, n_fine) for every ray, or (i + lnb_uniform(seed, ray0 + r, i)) / n_fine."""
    if not stratified:
        return np.broadcast_to(np.linspace(0.0, 1.0, n_fine), (R, n_fine)).copy()
    xi = np.array([[uniform(seed, ray0 + r, i) for i in range(n_fine)] for r in range(R)], np.float64).reshape(R, n_fine)
    return (np.arange(n_fine, dtype=np.float64)[None, :] + xi) / np.float64(n_fine)


def sample_pdf_f64(t, w, n_fine, stratified=False, seed=0, ray0=0, u=None):
    """The rule of lnb_sample_pdf: t [R][S] float64, w [R][S] float32 -> [R][S + n_fine] float64.  u [R][n_fine]
    overrides the sample positions (tests of the inverse transform itself)."""
    t = np.asarray(t, np.float64)
    w = np.asarray(w, np.float32)
    R, S = t.shape
    if u is None:
        u = sample_positions(R, n_fine, stratified, seed, ray0)
    mids = 0.5 * (t[:, 1:] + t[:, :-1])                          # m_k, k < S-1
    v = w[:, 1:-1].astype(np.float64) + 1e-5                     # v_j, j < S-2
    c = np.zeros((R, S - 1), np.float64)
    for j in range(S - 2):                                       # summed in order, as the kernel does
        c[:, j + 1] = c[:, j] + v[:, j]
    cdf = c / c[:, -1:]
    out = np.empty((R, S + u.shape[1]), np.float64)
    for r in range(R):
        ind = np.searchsorted(cdf[r], u[r], side="right")
        below = np.maximum(ind - 1, 0)
        above = np.minimum(ind, S - 2)
        d = cdf[r, above] - cdf[r, below]
        d = np.where(d < 1e-5, 1.0, d)
        tau = (u[r] - cdf[r, below]) / d
        x = mids[r, below] + tau * (mids[r, above] - mids[r, below])
        out[r] = np.sort(np.concatenate([t[r], x]))
    return out


def coarse_fine_f64(rays_o, rays_d, t, coarse, fine, target, E, n_fine, E_d=None, stratified=False, seed=0, ray0=0, g=None):
    """The coarse-to-fine evaluation of one batch: nerf_f64 of the coarse net at t, sample_pdf_f64 of its weights
    (rounded to float32, as the device hands them over), then the fine net at the S + n_fine sorted depths.
    coarse / fine: (dims, ws, bs).  Returns (coarse result, t_fine, fine result)."""
    R, S = np.shape(t)
    X, dists = V.features(rays_o, rays_d, t, E, E_d)
    rc = O.nerf_f64(X, coarse[1], coarse[2], coarse[0], target, dists, R, S, g=g)
    t_fine = sample_pdf_f64(t, rc["weights"].astype(np.float32), n_fine, stratified, seed, ray0)
    Xf, dists_f = V.features(rays_o, rays_d, t_fine, E, E_d)
    rf = O.nerf_f64(Xf, fine[1], fine[2], fine[0], target, dists_f, R, S + n_fine, g=g)
    return rc, t_fine, rf
