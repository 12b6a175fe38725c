"""oracle/oracle.py -- Python face of the parity checker.

TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this module; the product package
(loma_nerf_b200) never does.

Three checkers, strongest first:

* ``RefLib``   -- the REAL reference: the loma programs scripts/nerf.py and
  scripts/mlp_fit.py compiled by the reference's own compiler (oracle/build_ref.py
  -> oracle/_ref/*.so), driven with contiguous numpy arrays + row-pointer tables
  (the same ragged float**/float*** ABI the reference hosts use,
  /root/reference/mlp_utils.py:33-118) from a big-stack thread (the grad function
  keeps >=16 MB of tape on the stack, SURVEY.md 8b).
* ``COracle``  -- oracle/nerf_oracle.c, the plain-C fp32 restatement (flat buffers).
* ``nerf_f64`` / ``mlp_fit_f64`` -- float64 numpy restatement of the closed form
  (SURVEY.md Appendix B) for shapes too large for the serial C code.

Pinning status: see the header of nerf_oracle.c and tests/test_oracle.py.
"""
import ctypes
import os
import subprocess
import threading
from ctypes import POINTER, c_float, c_int

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF_DIR = os.path.join(HERE, "_ref")
BUILD_DIR = os.path.join(HERE, "_build")

c_float_p = POINTER(c_float)
c_float_pp = POINTER(c_float_p)
c_float_ppp = POINTER(c_float_pp)
c_int_p = POINTER(c_int)
c_int_pp = POINTER(c_int_p)


# ------------------------------------------------------------------------------------------------
# shapes and synthetic inputs shared by the tests, golden generator and bench
# ------------------------------------------------------------------------------------------------
def mlp_dims(c_in, width, n_layers, c_out):
    """[in, W, ..., W, out] as get_sample_mlp builds them (mlp_utils.py:177-204)."""
    return [c_in] + [width] * (n_layers - 1) + [c_out]


def init_mlp(rng, dims, sigma_bias_shift=0.0):
    """He-normal weights [in][out], N(0,0.5) biases (mlp_utils.py:166-204), padded like
    pad_array (mlp_utils.py:272-313) to (L,max_in,max_out) / (L,max_out) float32."""
    L = len(dims) - 1
    max_in, max_out = max(dims[:-1]), max(dims[1:])
    ws = np.zeros((L, max_in, max_out), np.float32)
    bs = np.zeros((L, max_out), np.float32)
    for l in range(L):
        i, o = dims[l], dims[l + 1]
        ws[l, :i, :o] = rng.normal(0.0, (2.0 / i) ** 0.5, size=(i, o)).astype(np.float32)
        bs[l, :o] = rng.normal(0.0, 0.5, size=o).astype(np.float32)
    if sigma_bias_shift and dims[-1] == 4:
        bs[L - 1, 3] += np.float32(sigma_bias_shift)
    return ws, bs


def positional_encoding(x, num_functions):
    """pos_encoding.py:4-70 for any leading shape: float64 math, float32 result, feature index
    = slot*F + coord with slot 0 identity, 2i+1 sin(2^i x), 2i+2 cos(2^i x)."""
    x = np.asarray(x, np.float64)
    parts = [x]
    for i in range(num_functions):
        parts.append(np.sin((2.0 ** i) * x))
        parts.append(np.cos((2.0 ** i) * x))
    out = np.stack(parts, axis=-2)  # (..., slots, F)
    return out.reshape(*x.shape[:-1], -1).astype(np.float32)


def sample_points(rays_o, rays_d, t_vals):
    """train_nerf.py:289-311. t_vals is (S,) (the reference's shared linspace) or (R,S)
    (stratified). Returns pts (R,S,3) float64 and dists (R,S) float32 with last = 1e8."""
    rays_o = np.asarray(rays_o, np.float64)
    rays_d = np.asarray(rays_d, np.float64)
    t = np.asarray(t_vals, np.float64)
    if t.ndim == 1:
        t = np.broadcast_to(t[None, :], (rays_o.shape[0], t.shape[0]))
    pts = rays_o[:, None, :] + rays_d[:, None, :] * t[:, :, None]
    dists = np.concatenate([t[:, 1:] - t[:, :-1], np.full_like(t[:, :1], 1e8)], axis=1)
    return pts, dists.astype(np.float32)


def synthetic_rays(rng, n_rays, n_views=1):
    """Blender-lego-like rays as get_rays makes them (train_nerf.py:23-62): camera on a radius-4
    sphere looking at the origin, pinhole focal = 0.5/tan(0.5*0.6911) in normalised [0,1] pixel
    coordinates, directions ((i-.5)/f, -(j-.5)/f, -1) @ R^T, NOT normalised.  float64."""
    focal = 0.5 / np.tan(0.5 * 0.6911)
    o_all, d_all = [], []
    per = [n_rays // n_views + (1 if v < n_rays % n_views else 0) for v in range(n_views)]
    for v in range(n_views):
        th = rng.uniform(0, 2 * np.pi)
        ph = rng.uniform(np.deg2rad(10), np.deg2rad(60))
        cam = 4.0 * np.array([np.cos(th) * np.cos(ph), np.sin(th) * np.cos(ph), np.sin(ph)])
        fwd = -cam / np.linalg.norm(cam)
        right = np.cross(fwd, np.array([0.0, 0.0, 1.0]))
        right /= np.linalg.norm(right)
        up = np.cross(right, fwd)
        Rm = np.stack([right, up, -fwd], axis=1)  # camera looks down -z
        i = rng.uniform(0, 1, per[v])
        j = rng.uniform(0, 1, per[v])
        dirs = np.stack([(i - 0.5) / focal, -(j - 0.5) / focal, -np.ones_like(i)], -1)
        d_all.append(dirs @ Rm.T)
        o_all.append(np.broadcast_to(cam, (per[v], 3)).copy())
    return np.concatenate(o_all), np.concatenate(d_all)


def stratified_t(rng, n_rays, n_samples, near=2.0, far=6.0):
    """SURVEY.md 8d: t_s = near + (s+u)(far-near)/S, u ~ U[0,1) per (ray, sample)."""
    u = rng.uniform(0, 1, (n_rays, n_samples))
    return near + (np.arange(n_samples)[None, :] + u) * (far - near) / n_samples


def make_nerf_case(seed, R, S, E=5, width=30, n_layers=3, stratified=True, sigma_bias_shift=1.0):
    """One synthetic nerf problem in the reference's compat layout (pre-encoded features)."""
    rng = np.random.default_rng(seed)
    o, d = synthetic_rays(rng, R)
    t = stratified_t(rng, R, S) if stratified else np.linspace(2.0, 6.0, S)
    pts, dists = sample_points(o, d, t)
    X = positional_encoding(pts, E).reshape(R * S, -1)
    dims = mlp_dims(X.shape[1], width, n_layers, 4)
    ws, bs = init_mlp(np.random.default_rng(seed + 1), dims, sigma_bias_shift)
    target = rng.uniform(0, 1, (R, 3)).astype(np.float32)
    tt = np.broadcast_to(t, (R, S)) if np.ndim(t) == 1 else t
    return dict(X=X, ws=ws, bs=bs, dims=np.array(dims, np.int32), target=target, dists=dists,
                R=R, S=S, rays_o=o, rays_d=d, t=np.ascontiguousarray(tt, dtype=np.float64), E=E)


def make_fit_case(seed, N, E=5, width=16, n_layers=3):
    """One synthetic 2-D image-fit problem (fit_img.py:379-421 shapes)."""
    rng = np.random.default_rng(seed)
    xy = rng.uniform(0, 1, (N, 2))
    X = positional_encoding(xy, E)
    dims = mlp_dims(X.shape[1], width, n_layers, 3)
    ws, bs = init_mlp(np.random.default_rng(seed + 1), dims)
    target = (0.5 + 0.4 * np.sin(6 * xy[:, :1] + np.array([0.0, 1.0, 2.0])) * np.cos(4 * xy[:, 1:])
              + 0.05 * rng.normal(size=(N, 3))).clip(0, 1).astype(np.float32)
    return dict(X=X, ws=ws, bs=bs, dims=np.array(dims, np.int32), target=target, xy=xy, E=E)


# ------------------------------------------------------------------------------------------------
# float64 numpy restatement (SURVEY.md Appendix B)
# ------------------------------------------------------------------------------------------------
def head_f64(Z, head):
    """The head's activation of the last layer's pre-activations Z: sigmoid, and for nerf ReLU on sigma."""
    Y = 1.0 / (1.0 + np.exp(-Z))
    if head == "nerf":
        Y[:, 3] = np.maximum(Z[:, 3], 0.0)
    return Y


def head_adjoint_f64(Y, dY, head):
    """Adjoint of the head's pre-activations from that of its outputs Y."""
    dZ = dY * Y * (1.0 - Y)
    if head == "nerf":
        dZ[:, 3] = dY[:, 3] * (Y[:, 3] > 0)
    return dZ


def _mlp_f64(X, ws, bs, dims, head):
    L = len(dims) - 1
    H = [np.asarray(X, np.float64)]
    for l in range(L):
        Z = H[-1] @ ws[l, :dims[l], :dims[l + 1]].astype(np.float64) + bs[l, :dims[l + 1]]
        H.append(np.maximum(Z, 0.0) if l < L - 1 else head_f64(Z, head))
    return H  # H[0]=X, H[l+1] = post-activation output of layer l


def _mlp_back_f64(H, dY, ws, bs, dims, head):
    """dY = adjoint of the head's post-activation output. Returns d_ws, d_bs, d_X, [dZ_l]."""
    L = len(dims) - 1
    d_ws = np.zeros(ws.shape, np.float64)
    d_bs = np.zeros(bs.shape, np.float64)
    dZs = [None] * L
    dH = dY
    for l in range(L - 1, -1, -1):
        dZ = dH * (H[l + 1] > 0) if l < L - 1 else head_adjoint_f64(H[l + 1], dH, head)
        dZs[l] = dZ
        d_ws[l, :dims[l], :dims[l + 1]] = H[l].T @ dZ
        d_bs[l, :dims[l + 1]] = dZ.sum(0)
        dH = dZ @ ws[l, :dims[l], :dims[l + 1]].astype(np.float64).T
    return d_ws, d_bs, dH, dZs


def composite_f64(rgba, dists, target, R, S, g=None):
    """Compositing and SSE loss of the head outputs rgba [R*S][4] (scripts/nerf.py:176-302) and, when g is not None, the
    adjoints: dY (of rgba, seeded with g; g='loss' seeds with the loss), d_dists, d_acc, d_target."""
    out = np.asarray(rgba, np.float64).reshape(R, S, 4)
    rgb, sigma = out[..., :3], out[..., 3]
    dist = np.asarray(dists, np.float64).reshape(R, S)
    e = np.exp(-sigma * dist)
    alpha = 1.0 - e
    q = (1.0 - alpha) + np.float64(np.float32(1e-10))
    C = np.cumprod(q, axis=1)
    T = C.copy()
    T[:, 0] = 1.0
    w = alpha * T
    color = (w[..., None] * rgb).sum(1)
    loss = ((color - target) ** 2).sum()
    res = dict(loss=loss, color=color, rgba=out, alpha=alpha, cumprod=T, weights=w)
    if g is None:
        return res
    g = loss if isinstance(g, str) else float(g)
    d_color = 2.0 * g * (color - target)
    d_rgb = w[..., None] * d_color[:, None, :]
    d_w = (rgb * d_color[:, None, :]).sum(-1)
    d_alpha = d_w * T
    dC = d_w * alpha
    dC[:, 0] = 0.0
    dq = np.zeros_like(q)
    for s in range(S - 1, 0, -1):
        dq[:, s] = C[:, s - 1] * dC[:, s]
        dC[:, s - 1] += q[:, s] * dC[:, s]
    dq[:, 0] = dC[:, 0]
    d_alpha = d_alpha - dq
    d_sigma = d_alpha * e * dist
    d_dists = d_alpha * e * sigma
    dY = np.concatenate([d_rgb, d_sigma[..., None]], -1).reshape(R * S, 4)
    res.update(dY=dY, d_target=-d_color, d_dists=d_dists, d_acc=d_color, g=g)
    return res


def fit_loss_f64(pred, target, g=None):
    """SSE of the first target.shape[0] rows / target.shape[1] channels of pred (scripts/mlp_fit.py:140-145) and, when g is
    not None, its adjoint dY (of pred, seeded with g; g='loss' seeds with the loss)."""
    R, Wt = target.shape
    diff = pred[:R, :Wt] - target
    loss = (diff ** 2).sum()
    res = dict(loss=loss, pred=pred)
    if g is None:
        return res
    g = loss if isinstance(g, str) else float(g)
    dY = np.zeros_like(pred)
    dY[:R, :Wt] = 2.0 * g * diff
    res.update(dY=dY, d_target=-dY[:R, :Wt], g=g)
    return res


def nerf_f64(X, ws, bs, dims, target, dists, R, S, g=None):
    """Forward (+ backward when g is not None; g='loss' seeds with the loss as the reference host
    does, train_nerf.py:477). Returns a dict of float64 arrays."""
    dims = [int(v) for v in dims]
    H = _mlp_f64(X, ws, bs, dims, "nerf")
    res = composite_f64(H[-1], dists, target, R, S, g)
    res["inter"] = [h for h in H[1:]]
    if g is None:
        return res
    d_ws, d_bs, d_X, dZs = _mlp_back_f64(H, res.pop("dY"), ws, bs, dims, "nerf")
    res.update(d_ws=d_ws, d_bs=d_bs, d_X=d_X, d_inter=dZs)
    return res


def mlp_fit_f64(X, ws, bs, dims, target, g=None):
    dims = [int(v) for v in dims]
    H = _mlp_f64(X, ws, bs, dims, "sigmoid")
    res = fit_loss_f64(H[-1], target, g)
    res["inter"] = [h for h in H[1:]]
    if g is None:
        return res
    d_ws, d_bs, d_X, dZs = _mlp_back_f64(H, res.pop("dY"), ws, bs, dims, "sigmoid")
    res.update(d_ws=d_ws, d_bs=d_bs, d_X=d_X, d_inter=dZs)
    return res


# ------------------------------------------------------------------------------------------------
# C restatement
# ------------------------------------------------------------------------------------------------
def build_c_oracle():
    so = os.path.join(BUILD_DIR, "liboracle.so")
    src = os.path.join(HERE, "nerf_oracle.c")
    if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.run(["make", "-C", HERE, "-s"], check=True)
    return so


def _fp(a):
    return a.ctypes.data_as(c_float_p)


def _ip(a):
    return a.ctypes.data_as(c_int_p)


class COracle:
    """ctypes face of oracle/nerf_oracle.c (flat buffers, fp32)."""

    def __init__(self):
        self.lib = ctypes.CDLL(build_c_oracle())
        L = self.lib
        L.oracle_nerf_forward.restype = c_float
        L.oracle_mlp_fit_forward.restype = c_float
        L.oracle_nerf_backward.restype = None
        L.oracle_mlp_fit_backward.restype = None
        L.oracle_mult_a_b.restype = None
        L.oracle_pos_encoding.restype = None
        L.oracle_sample_points.restype = None

    @staticmethod
    def _prep(X, ws, bs, dims):
        X = np.ascontiguousarray(X, np.float32)
        ws = np.ascontiguousarray(ws, np.float32)
        bs = np.ascontiguousarray(bs, np.float32)
        dims = np.ascontiguousarray(dims, np.int32)
        return X, ws, bs, dims, len(dims) - 1, ws.shape[1], ws.shape[2]

    def nerf_forward(self, X, ws, bs, dims, target, dists, R, S, rows=None):
        X, ws, bs, dims, L, mi, mo = self._prep(X, ws, bs, dims)
        N = X.shape[0]
        rows = N if rows is None else max(rows, N)
        ld = mo
        target = np.ascontiguousarray(target, np.float32)
        dists = np.ascontiguousarray(dists, np.float32)
        inter = np.zeros((L, rows, ld), np.float32)
        rgba = np.zeros((R, S, 4), np.float32)
        alpha = np.zeros((R, S), np.float32)
        cum = np.zeros((R, S), np.float32)
        wgt = np.zeros((R, S), np.float32)
        acc = np.zeros((R, 3), np.float32)
        loss = self.lib.oracle_nerf_forward(
            _fp(X), c_int(N), c_int(X.shape[1]), _fp(ws), _fp(bs), c_int(L), _ip(dims), c_int(mi),
            c_int(mo), _fp(target), c_int(R), c_int(S), _fp(dists), c_int(rows), c_int(ld),
            _fp(inter), _fp(rgba), _fp(alpha), _fp(cum), _fp(wgt), _fp(acc))
        return dict(loss=np.float32(loss), inter=inter, rgba=rgba, alpha=alpha, cumprod=cum,
                    weights=wgt, color=acc)

    def nerf_backward(self, X, ws, bs, dims, target, dists, R, S, g, rows=None):
        X, ws, bs, dims, L, mi, mo = self._prep(X, ws, bs, dims)
        N = X.shape[0]
        rows = N if rows is None else max(rows, N)
        ld = mo
        target = np.ascontiguousarray(target, np.float32)
        dists = np.ascontiguousarray(dists, np.float32)
        d_X = np.zeros_like(X)
        d_ws = np.zeros_like(ws)
        d_bs = np.zeros_like(bs)
        d_t = np.zeros_like(target)
        d_d = np.zeros_like(dists)
        d_acc = np.zeros((R, 3), np.float32)
        d_inter = np.zeros((L, rows, ld), np.float32)
        self.lib.oracle_nerf_backward(
            _fp(X), c_int(N), c_int(X.shape[1]), _fp(ws), _fp(bs), c_int(L), _ip(dims), c_int(mi),
            c_int(mo), _fp(target), c_int(R), c_int(S), _fp(dists), c_int(rows), c_int(ld),
            c_float(g), _fp(d_X), _fp(d_ws), _fp(d_bs), _fp(d_t), _fp(d_d), _fp(d_acc),
            _fp(d_inter))
        return dict(d_X=d_X, d_ws=d_ws, d_bs=d_bs, d_target=d_t, d_dists=d_d, d_acc=d_acc,
                    d_inter=d_inter)

    def mlp_fit_forward(self, X, ws, bs, dims, target, rows=None):
        X, ws, bs, dims, L, mi, mo = self._prep(X, ws, bs, dims)
        N = X.shape[0]
        rows = N if rows is None else max(rows, N)
        target = np.ascontiguousarray(target, np.float32)
        inter = np.zeros((L, rows, mo), np.float32)
        loss = self.lib.oracle_mlp_fit_forward(
            _fp(X), c_int(N), c_int(X.shape[1]), _fp(ws), _fp(bs), c_int(L), _ip(dims), c_int(mi),
            c_int(mo), _fp(target), c_int(target.shape[0]), c_int(target.shape[1]), c_int(rows),
            c_int(mo), _fp(inter))
        return dict(loss=np.float32(loss), inter=inter)

    def mlp_fit_backward(self, X, ws, bs, dims, target, g, rows=None):
        X, ws, bs, dims, L, mi, mo = self._prep(X, ws, bs, dims)
        N = X.shape[0]
        rows = N if rows is None else max(rows, N)
        target = np.ascontiguousarray(target, np.float32)
        d_X = np.zeros_like(X)
        d_ws = np.zeros_like(ws)
        d_bs = np.zeros_like(bs)
        d_t = np.zeros_like(target)
        d_inter = np.zeros((L, rows, mo), np.float32)
        self.lib.oracle_mlp_fit_backward(
            _fp(X), c_int(N), c_int(X.shape[1]), _fp(ws), _fp(bs), c_int(L), _ip(dims), c_int(mi),
            c_int(mo), _fp(target), c_int(target.shape[0]), c_int(target.shape[1]), c_int(rows),
            c_int(mo), c_float(g), _fp(d_X), _fp(d_ws), _fp(d_bs), _fp(d_t), _fp(d_inter))
        return dict(d_X=d_X, d_ws=d_ws, d_bs=d_bs, d_target=d_t, d_inter=d_inter)

    def mult_a_b(self, a, b):
        a = np.ascontiguousarray(a, np.float32)
        b = np.ascontiguousarray(b, np.float32)
        c = np.zeros((a.shape[0], b.shape[1]), np.float32)
        self.lib.oracle_mult_a_b(_fp(a), c_int(a.shape[0]), c_int(a.shape[1]), _fp(b),
                                 c_int(b.shape[0]), c_int(b.shape[1]), _fp(c))
        return c

    def pos_encoding(self, x, E):
        x = np.ascontiguousarray(x, np.float64)
        F = x.shape[-1]
        n = x.size // F
        out = np.zeros((n, F * (1 + 2 * E)), np.float32)
        self.lib.oracle_pos_encoding(x.ctypes.data_as(POINTER(ctypes.c_double)),
                                     ctypes.c_long(n), c_int(F), c_int(E), _fp(out))
        return out.reshape(*x.shape[:-1], -1)


# ------------------------------------------------------------------------------------------------
# the real reference (.so built by build_ref.py), ragged ABI
# ------------------------------------------------------------------------------------------------
def rows2(a, ptr_t=c_float_p):
    """float**/int** view of a contiguous 2-D array: a table of row pointers (zero-copy)."""
    assert a.flags.c_contiguous and a.ndim == 2
    n, stride, base = a.shape[0], a.strides[0], a.ctypes.data
    tab = (ptr_t * n)()
    for i in range(n):
        tab[i] = ctypes.cast(base + i * stride, ptr_t)
    return tab


def rows3(a):
    """float*** view of a contiguous 3-D float32 array. Returns (table, keepalive)."""
    assert a.flags.c_contiguous and a.ndim == 3
    inner = [rows2(a[i]) for i in range(a.shape[0])]
    tab = (c_float_pp * a.shape[0])()
    for i, t in enumerate(inner):
        tab[i] = ctypes.cast(t, c_float_pp)
    return tab, inner


def run_big_stack(fn, stack_bytes=1 << 30):
    """The reference's grad functions keep their AD tapes on the stack (16 MB stock, 1.9 GB for
    the paper-size variant): run in a thread with a big stack."""
    box = {}

    def tgt():
        try:
            box["r"] = fn()
        except BaseException as e:  # noqa: BLE001
            box["e"] = e

    old = threading.stack_size(stack_bytes)
    try:
        th = threading.Thread(target=tgt)
        th.start()
        th.join()
    finally:
        threading.stack_size(old)
    if "e" in box:
        raise box["e"]
    return box["r"]


NERF_ARGTYPES = [c_float_pp, c_int, c_int, c_float_ppp, c_float_pp, c_float_pp, c_int, c_int, c_int,
                 c_int_pp, c_int_pp, c_int_pp, c_float_ppp, c_float_ppp, c_int, c_float_pp,
                 c_float_pp, c_float_pp, c_float_pp, c_float_pp]
FIT_ARGTYPES = [c_float_pp, c_int, c_int, c_float_pp, c_float_ppp, c_float_pp, c_float_pp, c_int,
                c_int, c_int, c_int_pp, c_int_pp, c_int_pp, c_float_ppp]


def grad_argtypes(argtypes):
    """reverse_diff.py:504-517: every In arg is followed by its adjoint (int -> int*), then
    the trailing float _dreturn."""
    out = []
    for t in argtypes:
        out.append(t)
        out.append(c_int_p if t is c_int else t)
    return out + [c_float]


def set_compat_argtypes(lib):
    """The argtypes/restype compiler.compile sets (loma_public/compiler.py:262-276)."""
    if hasattr(lib, "nerf_evaluate_and_march"):
        lib.nerf_evaluate_and_march.argtypes = NERF_ARGTYPES
        lib.nerf_evaluate_and_march.restype = c_float
        lib.grad_nerf_evaluate_and_march.argtypes = grad_argtypes(NERF_ARGTYPES)
        lib.grad_nerf_evaluate_and_march.restype = None
    if hasattr(lib, "mlp_fit"):
        lib.mlp_fit.argtypes = FIT_ARGTYPES
        lib.mlp_fit.restype = c_float
        lib.grad_mlp_fit.argtypes = grad_argtypes(FIT_ARGTYPES)
        lib.grad_mlp_fit.restype = None
        lib.mult_a_b.argtypes = [c_float_pp, c_int, c_int, c_float_pp, c_int, c_int, c_float_pp]
        lib.mult_a_b.restype = None
    return lib


class CompatCaller:
    """Drives any library exporting the reference's five symbols (the real reference in
    oracle/_ref, or the product libloma_nerf_b200.so) through the ragged ABI exactly as the
    reference hosts do (train_nerf.py:325-478, fit_img.py:468-532), but with zero-copy
    row-pointer tables instead of mlp_utils.convert_ndim_array_to_ndim_ctypes."""

    def __init__(self, lib, big_stack=True, scratch_rows=256, scratch_cols=None,
                 stack_bytes=1 << 30):
        self.lib = set_compat_argtypes(lib)
        self.big_stack = big_stack
        self.stack_bytes = stack_bytes
        self.scratch_rows = scratch_rows
        self.scratch_cols = scratch_cols

    def _call(self, fn):
        return run_big_stack(fn, self.stack_bytes) if self.big_stack else fn()

    def _shapes(self, dims, rows):
        L = len(dims) - 1
        wsh = np.array([[dims[l], dims[l + 1]] for l in range(L)], np.int32)
        bsh = np.array([[dims[l + 1], 1] for l in range(L)], np.int32)
        ish = np.array([[rows, dims[l + 1]] for l in range(L)], np.int32)
        return wsh, bsh, ish

    def nerf(self, X, ws, bs, dims, target, dists, R, S, g=None, rows=None):
        """One forward call (and one grad call when g is given; g='loss' passes the forward's
        return value as _dreturn like train_nerf.py:477). N = R*S must fit the library."""
        X = np.ascontiguousarray(X, np.float32)
        ws = np.ascontiguousarray(ws, np.float32)
        bs = np.ascontiguousarray(bs, np.float32)
        target = np.ascontiguousarray(target, np.float32)
        dists = np.ascontiguousarray(dists, np.float32)
        dims = [int(v) for v in dims]
        L, N = len(dims) - 1, X.shape[0]
        rows = max(N, self.scratch_rows) if rows is None else rows
        cols = self.scratch_cols or max(max(dims[1:]), 1)
        wsh, bsh, ish = self._shapes(dims, rows)
        inter = np.zeros((L, rows, cols), np.float32)
        rgba = np.zeros((R, S, 4), np.float32)
        alpha = np.zeros((R, S), np.float32)
        cum = np.zeros((R, S), np.float32)
        wgt = np.zeros((R, S), np.float32)
        acc = np.zeros((R, 3), np.float32)
        keep = []

        def t3(a):
            t, k = rows3(a)
            keep.append(k)
            return t

        fargs = [rows2(X), N, X.shape[1], t3(ws), rows2(bs), rows2(target), R, 3, L,
                 rows2(wsh, c_int_p), rows2(bsh, c_int_p), rows2(ish, c_int_p), t3(inter),
                 t3(rgba), S, rows2(dists), rows2(alpha), rows2(cum), rows2(wgt), rows2(acc)]
        loss = self._call(lambda: self.lib.nerf_evaluate_and_march(*fargs))
        res = dict(loss=np.float32(loss), inter=inter, rgba=rgba, alpha=alpha, cumprod=cum,
                   weights=wgt, color=acc)
        if g is None:
            return res
        g = float(loss) if isinstance(g, str) else float(g)
        z = lambda a: np.zeros_like(a)  # noqa: E731
        p_inter, p_rgba, p_alpha, p_cum, p_wgt, p_acc = (z(inter), z(rgba), z(alpha), z(cum),
                                                         z(wgt), z(acc))
        d = dict(d_X=z(X), d_ws=z(ws), d_bs=z(bs), d_target=z(target), d_inter=z(inter),
                 d_rgba=z(rgba), d_dists=z(dists), d_alpha=z(alpha), d_cumprod=z(cum),
                 d_weights=z(wgt), d_acc=z(acc))
        di = [c_int(0) for _ in range(7)]
        dwsh, dbsh, dish = z(wsh), z(bsh), z(ish)
        gargs = [rows2(X), rows2(d["d_X"]), N, ctypes.byref(di[0]), X.shape[1],
                 ctypes.byref(di[1]), t3(ws), t3(d["d_ws"]), rows2(bs), rows2(d["d_bs"]),
                 rows2(target), rows2(d["d_target"]), R, ctypes.byref(di[2]), 3,
                 ctypes.byref(di[3]), L, ctypes.byref(di[4]),
                 rows2(wsh, c_int_p), rows2(dwsh, c_int_p), rows2(bsh, c_int_p),
                 rows2(dbsh, c_int_p), rows2(ish, c_int_p), rows2(dish, c_int_p),
                 t3(p_inter), t3(d["d_inter"]), t3(p_rgba), t3(d["d_rgba"]), S,
                 ctypes.byref(di[5]), rows2(dists), rows2(d["d_dists"]), rows2(p_alpha),
                 rows2(d["d_alpha"]), rows2(p_cum), rows2(d["d_cumprod"]), rows2(p_wgt),
                 rows2(d["d_weights"]), rows2(p_acc), rows2(d["d_acc"]), g]
        self._call(lambda: self.lib.grad_nerf_evaluate_and_march(*gargs))
        res.update(d)
        res.update(g=g, primal_after_grad=dict(inter=p_inter, rgba=p_rgba, alpha=p_alpha,
                                               cumprod=p_cum, weights=p_wgt, color=p_acc))
        return res

    def mlp_fit(self, X, ws, bs, dims, target, g=None, rows=None):
        X = np.ascontiguousarray(X, np.float32)
        ws = np.ascontiguousarray(ws, np.float32)
        bs = np.ascontiguousarray(bs, np.float32)
        target = np.ascontiguousarray(target, np.float32)
        dims = [int(v) for v in dims]
        L, N = len(dims) - 1, X.shape[0]
        rows = max(N, self.scratch_rows) if rows is None else rows
        cols = self.scratch_cols or max(rows, max(dims[1:]))
        wsh, bsh, ish = self._shapes(dims, N)  # fit_img.py traces the true chunk shape
        inter = np.zeros((L, rows, cols), np.float32)
        out = np.zeros((target.shape[0], 3), np.float32)
        keep = []

        def t3(a):
            t, k = rows3(a)
            keep.append(k)
            return t

        fargs = [rows2(X), N, X.shape[1], rows2(out), t3(ws), rows2(bs), rows2(target),
                 target.shape[0], target.shape[1], L, rows2(wsh, c_int_p), rows2(bsh, c_int_p),
                 rows2(ish, c_int_p), t3(inter)]
        loss = self._call(lambda: self.lib.mlp_fit(*fargs))
        res = dict(loss=np.float32(loss), inter=inter)
        if g is None:
            return res
        g = float(loss) if isinstance(g, str) else float(g)
        z = lambda a: np.zeros_like(a)  # noqa: E731
        p_inter = z(inter)
        d = dict(d_X=z(X), d_out=z(out), d_ws=z(ws), d_bs=z(bs), d_target=z(target),
                 d_inter=z(inter))
        di = [c_int(0) for _ in range(5)]
        dwsh, dbsh, dish = z(wsh), z(bsh), z(ish)
        gargs = [rows2(X), rows2(d["d_X"]), N, ctypes.byref(di[0]), X.shape[1],
                 ctypes.byref(di[1]), rows2(out), rows2(d["d_out"]), t3(ws), t3(d["d_ws"]),
                 rows2(bs), rows2(d["d_bs"]), rows2(target), rows2(d["d_target"]),
                 target.shape[0], ctypes.byref(di[2]), target.shape[1], ctypes.byref(di[3]), L,
                 ctypes.byref(di[4]), rows2(wsh, c_int_p), rows2(dwsh, c_int_p),
                 rows2(bsh, c_int_p), rows2(dbsh, c_int_p), rows2(ish, c_int_p),
                 rows2(dish, c_int_p), t3(p_inter), t3(d["d_inter"]), g]
        self._call(lambda: self.lib.grad_mlp_fit(*gargs))
        res.update(d)
        res.update(g=g, primal_after_grad=dict(inter=p_inter))
        return res

    def mult_a_b(self, a, b):
        a = np.ascontiguousarray(a, np.float32)
        b = np.ascontiguousarray(b, np.float32)
        c = np.zeros((a.shape[0], b.shape[1]), np.float32)
        self.lib.mult_a_b(rows2(a), a.shape[0], a.shape[1], rows2(b), b.shape[0], b.shape[1],
                          rows2(c))
        return c


def have_ref(name="nerf"):
    return os.path.exists(os.path.join(REF_DIR, name + ".so"))


def load_ref(name="nerf"):
    """CompatCaller over the real reference library oracle/_ref/<name>.so."""
    path = os.path.join(REF_DIR, name + ".so")
    if not os.path.exists(path):
        raise FileNotFoundError(path + " (run `python oracle/build_ref.py` where /root/reference exists)")
    lib = ctypes.CDLL(path)
    if name == "nerf_big":
        return CompatCaller(lib, scratch_rows=192, scratch_cols=256, stack_bytes=3 << 30)
    return CompatCaller(lib)


def ref_nerf_chunked(ref, case, g=None, rays_per_call=None):
    """Evaluate a batch larger than the reference's static capacity (<=256 samples per call,
    train_nerf.py:193-196) by looping over ray chunks and summing loss and gradients in float64
    (the loss is a plain sum over rays, nerf.py:297-302, so this is exact up to fp32 order)."""
    R, S = case["R"], case["S"]
    rpc = rays_per_call or max(1, 256 // S)
    tot = dict(loss=0.0, d_ws=np.zeros(case["ws"].shape), d_bs=np.zeros(case["bs"].shape))
    colors, dX, dD, dT = [], [], [], []
    for r0 in range(0, R, rpc):
        r1 = min(R, r0 + rpc)
        sl = slice(r0 * S, r1 * S)
        out = ref.nerf(case["X"][sl], case["ws"], case["bs"], case["dims"], case["target"][r0:r1],
                       case["dists"][r0:r1], r1 - r0, S, g=g)
        tot["loss"] += float(out["loss"])
        colors.append(out["color"])
        if g is not None:
            tot["d_ws"] += out["d_ws"]
            tot["d_bs"] += out["d_bs"]
            dX.append(out["d_X"]); dD.append(out["d_dists"]); dT.append(out["d_target"])
    tot["color"] = np.concatenate(colors)
    if g is not None:
        tot["d_X"] = np.concatenate(dX)
        tot["d_dists"] = np.concatenate(dD)
        tot["d_target"] = np.concatenate(dT)
    return tot
