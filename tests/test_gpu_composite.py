"""Compositing extras on the GPU (lnb_composite, include/loma_nerf_b200.h): opacity and depth maps and compositing onto a
background colour, on the exact path (layerwise fp32 kernels), the fused tensor-core kernels' extras instantiations, the
wide path, the trainer and the frame renderer.  Checked against the float64 models of tests/composite_model.py."""
import ctypes

import numpy as np
import pytest

import composite_model as CM
from conftest import grad_errs, rel_err
from oracle import oracle as O
from test_gpu_tc_model import BOUNDS, over

pytestmark = pytest.mark.gpu

EXACT_TOL = 1e-5
BG = (1.0, 0.5, 0.25)
# acc and depth on the tensor-core paths: a ray's last sample has dist 1e8, so its alpha = 1 - exp(-1e8 sigma) turns the
# bf16-level error of a near-zero sigma into a weight error the colour damps (sigmoid rgb < 1, shared with the other
# samples) and the plain sum of weights does not.  Measured on one B200: 7.5e-4 at C2 (fused); the bound is 3x that.
MAPS_TOL = 2.5e-3


@pytest.fixture(scope="module")
def env():
    import torch
    from loma_nerf_b200 import api
    assert torch.cuda.is_available()
    c = api.Context(0)
    yield torch, api, c
    c.close()


def _cv(torch, a, dt=None):
    return torch.as_tensor(np.ascontiguousarray(a)).to(dt or torch.float32).cuda().contiguous()


def _np(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)


def _scene(theta=35.0):
    from loma_nerf_b200 import render
    focal = 0.5 / np.tan(0.5 * 0.6911)
    K = np.array([[focal, 0, 0.5], [0, focal, 0.5], [0, 0, 1]], np.float64)
    return K, render.pose_spherical(theta, -30.0, 4.0)


def _features(o, d, t, E):
    """X [R*S][3 + 6E] and dists as the exact encoder forms them from float64 (or float32-valued) rays."""
    pts, dists = O.sample_points(np.asarray(o, np.float64), np.asarray(d, np.float64), np.asarray(t, np.float64))
    return O.positional_encoding(pts, E).reshape(-1, 3 + 6 * E), dists


def _batch(env, mode, case, stratified=True):
    """The inputs of one step in `mode` and the features / dists / depths the oracle sees for them."""
    torch, api, ctx = env
    R, S, E = case["R"], case["S"], case["E"]
    if mode == "features":
        return dict(X=_cv(torch, case["X"]), dists=_cv(torch, case["dists"])), case["X"], case["dists"], None
    if mode in ("rays64", "rays32"):
        dt = np.float64 if mode == "rays64" else np.float32
        o, d, t = (np.ascontiguousarray(case[k], dt) for k in ("rays_o", "rays_d", "t"))
        tdt = torch.float64 if mode == "rays64" else torch.float32
        X, dists = _features(o, d, t, E)
        return dict(rays=tuple(_cv(torch, a, tdt) for a in (o, d, t))), X, dists, t.astype(np.float64)
    K, pose = _scene()
    W = 40
    pix = np.random.default_rng(R + S).choice(W * W, R, replace=False).astype(np.int32)
    cam = api.make_camera(pose, K, W, pixels=torch.as_tensor(pix).cuda(), stratified=stratified, seed=17)
    o, d, t = (_np(v) for v in ctx.camera_rays(cam, R, S))
    X, dists = _features(o, d, t, E)
    return dict(camera=cam), X, dists, t


def _step(env, dims, ws, bs, b, case, **kw):
    torch, api, ctx = env
    R, S, E = case["R"], case["S"], case["E"]
    if "X" in b:
        return ctx.nerf_step(dims, b["X"], ws, bs, b["dists"], R=R, S=S, **kw)
    if "rays" in b:
        return ctx.nerf_step_rays(dims, *b["rays"], E, ws, bs, **kw)
    return ctx.nerf_step_camera(dims, b["camera"], R, S, E, ws, bs, **kw)


# ---------------------------------------------------------------------------------------------------------------------
# exact path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["f32", "f32_layerwise"])
@pytest.mark.parametrize("mode,accumulate", [("features", False), ("features", True), ("rays64", False), ("rays32", False),
                                             ("cam-strat", False), ("cam-lin", False)])
def test_exact_path_against_the_f64_model(env, path, mode, accumulate):
    torch, api, ctx = env
    case = O.make_nerf_case(900, 37, 19, E=4, width=30, n_layers=3)
    b, X, dists, t = _batch(env, mode, case, stratified=mode != "cam-lin")
    dims = [int(v) for v in case["dims"]]
    ws, bs, tg = _cv(torch, case["ws"]), _cv(torch, case["bs"]), _cv(torch, case["target"])
    R = case["R"]
    c0 = np.random.default_rng(3).uniform(0, 0.2, (R, 3)).astype(np.float32)
    outs = ("color", "loss", "acc") + (("depth",) if mode != "features" else ())
    out = dict(color=_cv(torch, c0)) if accumulate else None
    if mode == "features":
        out = dict(out or {}, d_X=torch.zeros((R * case["S"], dims[0]), device="cuda"), d_dists=torch.zeros((R, case["S"]), device="cuda"))
        outs += ("d_X", "d_dists")
    fn = ctx.nerf_step if mode == "features" else None
    kw = dict(target=tg, grad=True, seed=1.0, outputs=outs, out=out, path=path, background=BG)
    if fn is not None:
        o = ctx.nerf_step(dims, b["X"], ws, bs, b["dists"], R=R, S=case["S"], color_accumulate=accumulate, **kw)
    else:   # (colour accumulation is a features-mode argument of Context.nerf_step)
        o = _step(env, dims, ws, bs, b, case, **kw)
    ctx.synchronize()
    o = {k: _np(v) for k, v in o.items()}
    tgt = case["target"].astype(np.float64) - (c0 if accumulate else 0.0)   # colour += c0: the model sees the shifted target
    f = CM.nerf_f64(X, case["ws"], case["bs"], dims, tgt, dists, R, case["S"], 1.0, bg=BG, t=t)
    want_color = f["color"] + (c0 if accumulate else 0.0)
    errs = dict(loss=rel_err(o["loss"][0], f["loss"]), color=rel_err(o["color"], want_color), acc=rel_err(o["acc"], f["acc"]),
                d_ws=rel_err(o["d_ws"], f["d_ws"]), d_bs=rel_err(o["d_bs"], f["d_bs"]))
    if "depth" in o:
        errs["depth"] = rel_err(o["depth"], f["depth"])
    if mode == "features":
        errs.update(d_X=rel_err(o["d_X"], f["d_X"]), d_dists=rel_err(o["d_dists"], f["d_dists"]))
    assert max(errs.values()) <= EXACT_TOL, errs


@pytest.mark.parametrize("mode", ["features", "rays64", "cam-lin"])
def test_exact_acc_and_depth_are_the_sums_of_the_same_calls_weights(env, mode):
    torch, api, ctx = env
    case = O.make_nerf_case(901, 70, 40, E=3, width=20, n_layers=3)
    b, X, dists, t = _batch(env, mode, case, stratified=False)
    dims = [int(v) for v in case["dims"]]
    outs = ("color", "weights", "acc") + (("depth",) if mode != "features" else ())
    o = _step(env, dims, _cv(torch, case["ws"]), _cv(torch, case["bs"]), b, case, outputs=outs, path="f32", background=BG)
    ctx.synchronize()
    w = _np(o["weights"]).astype(np.float64)
    np.testing.assert_allclose(_np(o["acc"]), w.sum(1), rtol=2e-6, atol=1e-6)
    if mode != "features":
        np.testing.assert_allclose(_np(o["depth"]), (w * t).sum(1), rtol=2e-6, atol=1e-5)


# ---------------------------------------------------------------------------------------------------------------------
# tensor-core paths
# ---------------------------------------------------------------------------------------------------------------------
TC_CASES = [  # (id, R, S, E, width, layers, mode): C2-like shapes, tail tiles, 16 / 32 / 64 columns
    ("c2-feat", 4097, 64, 5, 30, 3, "features"),
    ("w15-feat-S30", 1001, 30, 5, 15, 3, "features"),
    ("w62-feat-S100", 301, 100, 3, 62, 2, "features"),
    ("w30-rays-E2", 777, 64, 2, 30, 3, "rays64"),
    ("w20-rays32-E2-L4", 501, 40, 2, 20, 4, "rays32"),
]


@pytest.mark.parametrize("grad", [True, False], ids=["train", "render"])
@pytest.mark.parametrize("c", TC_CASES, ids=lambda c: c[0])
def test_fused_tc_extras_against_the_bf16_model(env, c, grad):
    torch, api, ctx = env
    cid, R, S, E, width, layers, mode = c
    case = O.make_nerf_case(910 + R, R, S, E=E, width=width, n_layers=layers)
    b, X, dists, t = _batch(env, mode, case)
    dims = [int(v) for v in case["dims"]]
    outs = ("color", "loss", "acc") + (("depth",) if mode != "features" else ())
    box = {}

    def call():
        box["o"] = _step(env, dims, _cv(torch, case["ws"]), _cv(torch, case["bs"]), b, case, target=_cv(torch, case["target"]),
                         grad=grad, outputs=outs, path="tc", background=BG)
    prof = ctx.profile_dominant(call)
    ctx.synchronize()
    assert prof is not None and prof["kernel"].startswith("fused_mg_kernel" if grad else "fused_v1_kernel"), prof
    assert prof["kernel"].endswith("+extras"), prof
    o = {k: _np(v) for k, v in box["o"].items()}
    rays = None
    if mode != "features":
        rays = (np.asarray(case["rays_o"], np.float64), np.asarray(case["rays_d"], np.float64), t, E)
        if mode == "rays32":
            rays = tuple(np.asarray(np.asarray(v, np.float32), np.float64) for v in rays[:3]) + (E,)
    m = CM.nerf_tc_model(case["X"], case["ws"], case["bs"], dims, case["target"], dists, R, S, 1.0 if grad else None,
                         "fused", rays=rays, bg=BG, t=t)
    errs = dict(loss=rel_err(o["loss"][0], m["loss"]), color=rel_err(o["color"], m["color"]), acc=rel_err(o["acc"], m["acc"]))
    if "depth" in o:
        errs["depth"] = rel_err(o["depth"], m["depth"])
    if grad:
        errs.update(grad_errs(o, m))
    bounds = dict(BOUNDS["fused"], acc=MAPS_TOL, depth=MAPS_TOL)
    r = {k: v / (bounds[k] if k in ("acc", "depth") else bounds["out"] if k in ("loss", "color") else
                 bounds["l2"] if k.endswith("_l2") else bounds["grad"]) for k, v in errs.items()}
    assert max(r.values()) <= 1.0, (cid, errs)


@pytest.mark.parametrize("stratified", [False, True])
def test_fused_render_with_view_directions_in_camera_mode(env, stratified):
    """Camera mode with view directions: the extras render against the plain render of the same call (colour) and the
    exact path (acc, depth): the two tensor-core kernels share the MLP, so colour = plain + (1 - acc) bg to fp32."""
    torch, api, ctx = env
    E, Ed, S, R = 5, 2, 64, 3001
    rng = np.random.default_rng(920)
    dims = O.mlp_dims(api.rays_input_width(E, Ed), 30, 3, 4)
    ws, bs = (_cv(torch, a) for a in O.init_mlp(rng, dims, 1.0))
    K, pose = _scene(60.0)
    cam = api.make_camera(pose, K, 64, first_pixel=500, stratified=stratified, seed=5)
    kw = dict(path="tc", dir_bands=Ed)
    plain = ctx.nerf_step_camera(dims, cam, R, S, E, ws, bs, outputs=("color",), **kw)["color"]
    box = {}
    prof = ctx.profile_dominant(lambda: box.update(o=ctx.nerf_step_camera(dims, cam, R, S, E, ws, bs, outputs=("color", "acc", "depth"),
                                                                          background=BG, **kw)))
    exact = ctx.nerf_step_camera(dims, cam, R, S, E, ws, bs, outputs=("acc", "depth"), path="f32", dir_bands=Ed)
    ctx.synchronize()
    assert prof is not None and prof["kernel"] == "fused_v1_kernel<rays>+extras", prof
    o = {k: _np(v).astype(np.float64) for k, v in box["o"].items()}
    want = _np(plain).astype(np.float64) + (1.0 - o["acc"])[:, None] * np.asarray(BG)[None, :]
    assert np.abs(o["color"] - want).max() <= 2e-6
    assert rel_err(o["acc"], _np(exact["acc"])) <= 3e-2 and rel_err(o["depth"], _np(exact["depth"])) <= 3e-2


@pytest.mark.parametrize("mode", ["features", "rays64"])
def test_wide_path_extras_against_the_bf16_model(env, mode):
    torch, api, ctx = env
    case = O.make_nerf_case(930, 96, 192, E=2 if mode == "rays64" else 5, width=128, n_layers=3)
    b, X, dists, t = _batch(env, mode, case)
    dims = [int(v) for v in case["dims"]]
    outs = ("color", "loss", "acc") + (("depth",) if mode != "features" else ())
    box = {}
    prof = ctx.profile_dominant(lambda: box.update(o=_step(env, dims, _cv(torch, case["ws"]), _cv(torch, case["bs"]), b, case,
                                                           target=_cv(torch, case["target"]), grad=True, outputs=outs, path="tc",
                                                           background=BG)))
    ctx.synchronize()
    assert prof is not None and prof["kernel"].startswith("chain_tc_kernel"), prof
    o = {k: _np(v) for k, v in box["o"].items()}
    rays = (case["rays_o"], case["rays_d"], t, case["E"]) if mode != "features" else None
    m = CM.nerf_tc_model(case["X"], case["ws"], case["bs"], dims, case["target"], dists, case["R"], case["S"], 1.0, "wide",
                         rays=rays, bg=BG, t=t)
    errs = dict(loss=rel_err(o["loss"][0], m["loss"]), color=rel_err(o["color"], m["color"]), acc=rel_err(o["acc"], m["acc"]),
                **grad_errs(o, m))
    if "depth" in o:
        errs["depth"] = rel_err(o["depth"], m["depth"])
    bounds = dict(BOUNDS["wide"], acc=MAPS_TOL, depth=MAPS_TOL)
    r = {k: v / (bounds[k] if k in ("acc", "depth") else bounds["out"] if k in ("loss", "color") else
                 bounds["l2"] if k.endswith("_l2") else bounds["grad"]) for k, v in errs.items()}
    assert max(r.values()) <= 1.0, errs


@pytest.mark.parametrize("path,width,grad", [("f32", 30, True), ("f32_layerwise", 30, True), ("tc", 30, True), ("tc", 30, False),
                                             ("tc", 128, True)])
def test_zero_background_is_the_plain_step(env, path, width, grad):
    torch, api, ctx = env
    case = O.make_nerf_case(940, 203, 64, E=5, width=width, n_layers=3)
    dims = [int(v) for v in case["dims"]]
    a = dict(X=_cv(torch, case["X"]), ws=_cv(torch, case["ws"]), bs=_cv(torch, case["bs"]), dists=_cv(torch, case["dists"]),
             target=_cv(torch, case["target"]))
    kw = dict(grad=grad, outputs=("color", "loss"))
    # the exact path runs a step with extras on the layerwise kernels: it equals the plain step there
    plain = ctx.nerf_step(dims, a["X"], a["ws"], a["bs"], a["dists"], a["target"], path="f32_layerwise" if path == "f32" else path, **kw)
    zero = ctx.nerf_step(dims, a["X"], a["ws"], a["bs"], a["dists"], a["target"], background=(0.0, 0.0, 0.0), path=path, **kw)
    ctx.synchronize()
    for k in ("color", "loss"):
        assert np.array_equal(_np(plain[k]), _np(zero[k])), k
    if grad and path.startswith("f32"):
        for k in ("d_ws", "d_bs"):
            assert np.array_equal(_np(plain[k]), _np(zero[k])), k


def test_host_variant_equals_the_device_variant(env):
    torch, api, ctx = env
    case = O.make_nerf_case(950, 55, 21, E=3, width=20, n_layers=3)
    dims = [int(v) for v in case["dims"]]
    outs = ("color", "loss", "acc", "depth")
    kw = dict(target=case["target"], grad=True, outputs=outs, path="f32", background=BG)
    host = ctx.nerf_step_rays(dims, case["rays_o"], case["rays_d"], case["t"], 3, case["ws"], case["bs"], **kw)
    kw["target"] = _cv(torch, case["target"])
    r = [_cv(torch, case[k], torch.float64) for k in ("rays_o", "rays_d", "t")]
    devr = ctx.nerf_step_rays(dims, *r, 3, _cv(torch, case["ws"]), _cv(torch, case["bs"]), **kw)
    ctx.synchronize()
    for k in outs + ("d_ws", "d_bs"):
        assert np.array_equal(np.asarray(host[k]), _np(devr[k])), k


def test_argument_checks(env):
    torch, api, ctx = env
    from loma_nerf_b200 import _lib as L
    case = O.make_nerf_case(960, 8, 16, E=2, width=16, n_layers=2)
    dims = [int(v) for v in case["dims"]]
    X, ws, bs, dists = (_cv(torch, case[k]) for k in ("X", "ws", "bs", "dists"))
    with pytest.raises(ValueError):     # before anything launches
        ctx.nerf_step(dims, X, ws, bs, dists, outputs=("color", "depth"))
    mlp = api.make_mlp(dims, case["ws"].shape, L.HEAD_NERF)
    color, depth = torch.zeros((8, 3), device="cuda"), torch.zeros(8, device="cuda")
    a = L.LnbStepArgs()
    a.R, a.S, a.n_rows, a.rows, a.target_w = 8, 16, 128, 128, 3
    a.X, a.ws, a.bs, a.dists, a.color = X.data_ptr(), ws.data_ptr(), bs.data_ptr(), dists.data_ptr(), color.data_ptr()
    a.path = L.PATH_F32

    def rc(background, bg, depth_ptr=None):
        c = L.LnbComposite()
        c.background = background
        for i in range(3):
            c.bg[i] = bg[i]
        c.depth = depth_ptr
        return ctx.lib.lnb_nerf_step_composite(ctx.h, ctypes.byref(mlp), ctypes.byref(a), ctypes.byref(c))
    assert rc(0, (0, 0, 0), depth.data_ptr()) == L.LNB_ERR_ARG          # depth in features mode
    assert rc(2, (1, 1, 1)) == L.LNB_ERR_ARG                             # background not 0 or 1
    assert rc(1, (1, float("nan"), 1)) == L.LNB_ERR_ARG                  # non-finite colour
    assert rc(1, (1, 1, 1)) == L.LNB_OK
    ctx.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# trainer
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("route,width,path", [("fused", 30, "tc"), ("wide", 128, "tc"), ("exact", 30, "f32")])
def test_trainer_grad_with_background(env, route, width, path):
    torch, api, ctx = env
    case = O.make_nerf_case(970, 1025, 64, E=5, width=width, n_layers=3)
    dims = [int(v) for v in case["dims"]]
    tr = api.Trainer(ctx, dims, case["ws"], case["bs"], background=BG)
    try:
        tr.grad(X=_cv(torch, case["X"]), dists=_cv(torch, case["dists"]), target=_cv(torch, case["target"]), path=path)
        ctx.order_torch_after()
        g = _np(tr.grad_buffer())
    finally:
        tr.close()
    nw = case["ws"].size
    o = dict(d_ws=g[:nw].reshape(case["ws"].shape), d_bs=g[nw:-1].reshape(case["bs"].shape), loss=g[-1:])
    args = (case["X"], case["ws"], case["bs"], dims, case["target"], case["dists"], case["R"], case["S"], 1.0)
    if route == "exact":
        f = CM.nerf_f64(*args, bg=BG)
        errs = dict(loss=rel_err(o["loss"][0], f["loss"]), d_ws=rel_err(o["d_ws"], f["d_ws"]), d_bs=rel_err(o["d_bs"], f["d_bs"]))
        assert max(errs.values()) <= EXACT_TOL, errs
        return
    m = CM.nerf_tc_model(*args, "fused" if route == "fused" else "wide", bg=BG)
    errs = dict(loss=rel_err(o["loss"][0], m["loss"]), **grad_errs(o, m))
    assert max(over(errs, BOUNDS["fused" if route == "fused" else "wide"]).values()) <= 1.0, errs


@pytest.mark.parametrize("path", ["tc", "f32"])
def test_trainer_without_background_is_unchanged(env, path):
    torch, api, ctx = env
    case = O.make_nerf_case(980, 512, 64, E=5, width=30, n_layers=3)
    dims = [int(v) for v in case["dims"]]
    batch = dict(X=_cv(torch, case["X"]), dists=_cv(torch, case["dists"]), target=_cv(torch, case["target"]), path=path)
    a, b = api.Trainer(ctx, dims, case["ws"], case["bs"]), api.Trainer(ctx, dims, case["ws"], case["bs"])
    try:
        b.set_background((1.0, 1.0, 1.0))
        b.set_background(None)
        wa, wb = (torch.zeros((512, 64), device="cuda") for _ in range(2))
        a.step_weights(wa, **batch)
        b.step_weights(wb, **batch)
        (pa, qa, la), (pb, qb, lb) = a.read(), b.read()
        assert np.array_equal(_np(wa), _np(wb)) and la == lb
        if path == "f32":
            assert np.array_equal(pa, pb) and np.array_equal(qa, qb)
        else:      # the tensor-core weight gradients' last bits follow the MMA completion order (LNB_PATH_TC)
            np.testing.assert_allclose(pb, pa, rtol=0, atol=1e-6)
        # and a background changes the step
        b.set_background((1.0, 1.0, 1.0))
        b.step_weights(wb, **batch)
        a.step_weights(wa, **batch)
        assert a.read()[2] != b.read()[2]
    finally:
        a.close()
        b.close()


def test_coarse_fine_white_background_graph_equals_eager(env):
    torch, api, ctx = env
    E, S, n_fine, R, W = 5, 32, 32, 64, 48
    rng = np.random.default_rng(990)
    dims = O.mlp_dims(33, 30, 3, 4)
    (wc, bc), (wf, bf) = O.init_mlp(rng, dims, 1.0), O.init_mlp(rng, dims, 1.0)
    target = _cv(torch, rng.uniform(0, 1, (R, 3)).astype(np.float32))
    K, pose = _scene(50.0)
    pix = torch.as_tensor(rng.choice(W * W, R, replace=False).astype(np.int32)).cuda()
    cams = [api.make_camera(pose, K, W, pixels=pix, stratified=True, seed=991 + i) for i in range(4)]
    white = (1.0, 1.0, 1.0)
    pairs = [(api.Trainer(ctx, dims, wc, bc, background=white), api.Trainer(ctx, dims, wf, bf, background=white)) for _ in range(2)]
    eager, graphed = (api.CoarseFine(c, f, n_fine) for c, f in pairs)
    kw = dict(S=S, pe_bands=E, target=target, path="f32")
    try:
        for cf in (eager, graphed):
            cf.step(camera=cams[0], **kw)
        for cam in cams[1:]:
            eager.step(camera=cam, **kw)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            ctx.set_stream(torch.cuda.current_stream())
            for cam in cams[1:]:
                graphed.step(camera=cam, **kw)
        ctx.set_stream(torch.cuda.current_stream())
        g.replay()
        torch.cuda.synchronize()
        for (ce, fe), (cg, fg) in [pairs]:
            for a, b in ((ce, cg), (fe, fg)):
                (wa, ba, la), (wb, bb, lb) = a.read(), b.read()
                assert np.array_equal(wa, wb) and np.array_equal(ba, bb) and la == lb
    finally:
        for c, f in pairs:
            c.close()
            f.close()


# ---------------------------------------------------------------------------------------------------------------------
# frame renderer
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["tc", "f32"])
@pytest.mark.parametrize("fine", [False, True], ids=["plain", "fine"])
def test_render_frame_device_maps(env, path, fine):
    torch, api, ctx = env
    from loma_nerf_b200 import render
    E, S, n_fine, W, chunk = 5, 32, 32, 40, 611
    rng = np.random.default_rng(995)
    dims = O.mlp_dims(33, 30, 3, 4)
    (wc, bc), (wf, bf) = O.init_mlp(rng, dims, 1.0), O.init_mlp(rng, dims, 1.0)
    wc_d, bc_d, wf_d, bf_d = (_cv(torch, a) for a in (wc, bc, wf, bf))
    K, pose = _scene(75.0)
    n = W * W
    acc, depth = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    img = render.render_frame_device(ctx, dims, wc_d, bc_d, W, W, K, pose, S, E, path=path, rays_per_call=chunk,
                                     fine=(dims, wf_d, bf_d, n_fine) if fine else None, background=(1, 1, 1), acc=acc, depth=depth)
    ctx.order_torch_after()
    img, acc, depth = _np(img), _np(acc).astype(np.float64), _np(depth).astype(np.float64)
    # the per-ray oracle: the rays and depths the camera generates (the fine pass: the depths the pipeline sampled)
    cam = api.make_camera(pose, K, W, W)
    o, d, t = (_np(v) for v in ctx.camera_rays(cam, n, S))
    if fine:
        w = ctx.nerf_step_camera(dims, cam, n, S, E, wc_d, bc_d, outputs=("weights",), path=path)["weights"]
        t = np.concatenate([_np(ctx.sample_pdf(_cv(torch, t[r0:r0 + chunk], torch.float64), w[r0:r0 + chunk], n_fine, ray0=r0))
                            for r0 in range(0, n, chunk)])
        net = (wf, bf)
    else:
        net = (wc, bc)
    X, dists = _features(o, d, t, E)
    m = CM.nerf_tc_model(X, net[0], net[1], dims, np.zeros((n, 3)), dists, n, t.shape[1], None, "fused", bg=(1, 1, 1), t=t,
                         _exact=path == "f32")
    # tc: the model rounds where the kernels do, but camera mode's fp32 rays and MUFU sin / cos can flip a bf16 rounding
    tol = 1e-5 if path == "f32" else 1e-2
    errs = (rel_err(acc, m["acc"]), rel_err(depth, m["depth"]))
    assert max(errs) <= tol, errs
    want = np.rint(255 * np.clip(m["color"], 0, 1)).reshape(W, W, 3)
    assert np.abs(img.astype(np.int64) - want).max() <= (1 if path == "f32" else 3)


def test_render_frame_device_without_extras_runs_the_plain_kernel(env):
    torch, api, ctx = env
    from loma_nerf_b200 import render
    rng = np.random.default_rng(996)
    dims = O.mlp_dims(33, 30, 3, 4)
    ws, bs = (_cv(torch, a) for a in O.init_mlp(rng, dims, 1.0))
    K, pose = _scene(20.0)
    box = {}
    prof = ctx.profile_dominant(lambda: box.update(img=render.render_frame_device(ctx, dims, ws, bs, 32, 32, K, pose, 32, 5)))
    plain = _np(box["img"])
    white = _np(render.render_frame_device(ctx, dims, ws, bs, 32, 32, K, pose, 32, 5, background=(1, 1, 1)))
    ctx.synchronize()
    assert prof is not None and prof["kernel"] == "fused_v1_kernel<rays>", prof     # the plain render kernel
    assert (white.astype(np.int64) >= plain.astype(np.int64) - 1).all()   # white only adds light
