"""Float64 models of the compositing extras (lnb_composite in include/loma_nerf_b200.h): opacity and depth maps and
compositing onto a background colour.  TEST INFRASTRUCTURE ONLY, beside the untouched oracle/ it builds on.

  acc_r   = sum_s w_s,  depth_r = sum_s w_s t_s,  color_r = sum_s w_s rgb_s + (1 - acc_r) bg
  backward: d_w_s = <rgb_s - bg, dcol_r>; everything after d_w_s as in oracle.composite_f64.

With bg=None the colour, loss and adjoints are oracle.composite_f64's own (it is called), so the reference's compositing
cannot drift from this model."""
import numpy as np

from oracle import oracle as O
from oracle import tc_model as M


def composite_f64(rgba, dists, target, R, S, g=None, bg=None, t=None):
    """oracle.composite_f64 plus acc [R], depth [R] (when t [R][S] is given) and the background term (bg: 3 floats)."""
    if bg is None:
        res = O.composite_f64(rgba, dists, target, R, S, g)
        w = res["weights"]
    else:
        bg = np.asarray(bg, np.float64).reshape(3)
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
        acc = w.sum(1)
        color = (w[..., None] * rgb).sum(1) + (1.0 - acc)[:, None] * bg[None, :]
        loss = ((color - target) ** 2).sum()
        res = dict(loss=loss, color=color, rgba=out, alpha=alpha, cumprod=T, weights=w)
        if g is not None:
            g = loss if isinstance(g, str) else float(g)
            d_color = 2.0 * g * (color - target)
            d_rgb = w[..., None] * d_color[:, None, :]
            d_w = ((rgb - bg[None, None, :]) * d_color[:, None, :]).sum(-1)
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
    res["acc"] = w.sum(1)
    if t is not None:
        res["depth"] = (w * np.asarray(t, np.float64).reshape(R, S)).sum(1)
    return res


def nerf_f64(X, ws, bs, dims, target, dists, R, S, g=None, bg=None, t=None):
    """oracle.nerf_f64 with the extras of composite_f64."""
    dims = [int(v) for v in dims]
    H = O._mlp_f64(X, ws, bs, dims, "nerf")
    res = composite_f64(H[-1], dists, target, R, S, g, bg, t)
    res["inter"] = [h for h in H[1:]]
    if g is None:
        return res
    d_ws, d_bs, d_X, dZs = O._mlp_back_f64(H, res.pop("dY"), ws, bs, dims, "nerf")
    res.update(d_ws=d_ws, d_bs=d_bs, d_X=d_X, d_inter=dZs)
    return res


def nerf_tc_model(X, ws, bs, dims, target, dists, R, S, g=None, variant="fused", rays=None, bg=None, t=None, _exact=False):
    """oracle.tc_model.nerf_tc_model (the tensor-core kernels' bf16 roundings) with the extras of composite_f64."""
    rb, rf = (M._ident, M._ident) if _exact else (M.bf16, M.f32)
    dims = [int(v) for v in dims]
    A0 = M.rays_features(*rays) if rays is not None else X
    W, A, hz, Y = M._forward(A0, ws, bs, dims, variant, rb, rf, "nerf")
    res = composite_f64(Y, dists, target, R, S, None if g is None else 1.0, bg, t)
    res.update(A_l=A, hz=hz)
    if g is None:
        return res
    return M._backward(res, W, A, O.head_adjoint_f64(Y, res.pop("dY"), "nerf"), ws, bs, dims, g, rb, rf)
