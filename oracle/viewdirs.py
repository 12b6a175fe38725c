"""oracle/viewdirs.py -- float64 restatement of the view-direction input of rays and camera mode.

A net whose input width is dims[0] = (3 + 6E) + (3 + 6E_d) takes, per sample, [ PE(x, E) | PE(u, E_d) ] with
x = o + d t and u = d / |d| the unit direction of the sample's ray (include/loma_nerf_b200.h, lnb_step_args.pe_bands).
|d| = sqrt((d0^2 + d1^2) + d2^2): numpy's elementwise operations, each rounded, in that order.  PE is
oracle.positional_encoding (float64 math, float32 result).  The reference has no direction input; this is the
library's own convention, stated here so that the tests can rebuild the features on the host.
"""
import numpy as np

from oracle import oracle as O


def unit_directions(rays_d):
    """u = d / |d| per ray, float64 [R][3]."""
    d = np.asarray(rays_d, np.float64)
    n = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
    return d / n[:, None]


def view_encoding(rays_d, E_d, S):
    """PE(u, E_d) of every ray, repeated for its S samples: [R*S][3 + 6E_d] float32."""
    return np.repeat(O.positional_encoding(unit_directions(rays_d), E_d), S, axis=0)


def features(rays_o, rays_d, t, E, E_d=None):
    """X [R*S][(3 + 6E) (+ 3 + 6E_d)] and dists [R][S], as rays mode builds them (t is (S,) or (R, S))."""
    pts, dists = O.sample_points(rays_o, rays_d, t)
    R, S = pts.shape[0], pts.shape[1]
    X = O.positional_encoding(pts, E).reshape(R * S, -1)
    if E_d is not None:
        X = np.concatenate([X, view_encoding(rays_d, E_d, S)], axis=1)
    return X, dists


def make_nerf_case(seed, R, S, E=5, E_dir=None, width=30, n_layers=3, stratified=True, sigma_bias_shift=1.0):
    """oracle.make_nerf_case, with E_dir: the features [PE(x, E) | PE(u, E_dir)] and a net of that input width (its
    weights drawn like oracle.make_nerf_case draws them).  E_dir=None returns oracle.make_nerf_case's case itself."""
    case = O.make_nerf_case(seed, R, S, E=E, width=width, n_layers=n_layers, stratified=stratified,
                            sigma_bias_shift=sigma_bias_shift)
    if E_dir is None:
        return case
    X = np.concatenate([case["X"], view_encoding(case["rays_d"], E_dir, S)], axis=1)
    dims = O.mlp_dims(X.shape[1], width, n_layers, 4)
    ws, bs = O.init_mlp(np.random.default_rng(seed + 1), dims, sigma_bias_shift)
    return dict(case, X=X, ws=ws, bs=bs, dims=np.array(dims, np.int32), E_dir=E_dir)
