"""View directions in rays and camera mode (include/loma_nerf_b200.h, lnb_step_args.pe_bands): a net of input width
(3 + 6E) + (3 + 6E_d) takes [PE(x, E) | PE(u, E_d)], u the unit direction of the sample's ray, built on the device on
every path.  Checked against the float64 restatement fed with the host-built features (oracle/viewdirs.py)."""
import numpy as np
import pytest

from conftest import grad_errs, rel_err
from oracle import oracle as O
from oracle import viewdirs as V

pytestmark = pytest.mark.gpu

TC_TOL, TC_LAYER_TOL, TC_L2_TOL = 3e-2, 6e-2, 3e-2     # the tensor-core bounds against the float64 restatement
WIDE_TOL = 6e-2
# Rays mode on the fused kernels against the same kernel in features mode fed with lnb_sample_encode_dirs' features: the
# two A_0 differ only where the fp32 encoding (MUFU sin / cos with angle doubling, u from rsqrtf) and the float64 one
# round to different bf16 values.  Measured on one B200 (max over the cases below): see FEATURES_TOL's log lines.
FEATURES_TOL = 1e-2


@pytest.fixture(scope="module")
def env():
    import torch
    from loma_nerf_b200 import api
    assert torch.cuda.is_available()
    c = api.Context(0)
    yield torch, api, c
    c.close()


def _scene(theta=35.0):
    from loma_nerf_b200 import render
    focal = 0.5 / np.tan(0.5 * 0.6911)
    K = np.array([[focal, 0, 0.5], [0, focal, 0.5], [0, 0, 1]], np.float64)
    return K, render.pose_spherical(theta, -30.0, 4.0)


def _cv(torch, a, dt=None):
    dt = dt or torch.float32
    return torch.as_tensor(np.ascontiguousarray(a)).to(dt).cuda().contiguous()


def _host(out):
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


def _errs(o, f):
    return dict(loss=rel_err(o["loss"][0], f["loss"]), color=rel_err(o["color"], f["color"]), **grad_errs(o, f))


def _check_tc(errs, tol=TC_TOL):
    assert max(errs["loss"], errs["color"], errs["d_ws"], errs["d_bs"]) <= tol, errs
    assert max(errs["d_ws_layer"], errs["d_bs_layer"]) <= TC_LAYER_TOL, errs
    assert max(errs["d_ws_l2"], errs["d_bs_l2"]) <= TC_L2_TOL, errs


def _camera_batch(env, W, R, S, seed, stratified):
    torch, api, ctx = env
    K, pose = _scene()
    pix = np.random.default_rng(seed).choice(W * W, R, replace=False).astype(np.int32)
    cam = api.make_camera(pose, K, W, pixels=torch.as_tensor(pix).cuda(), stratified=stratified, seed=seed)
    o, d, t = (v.cpu().numpy() for v in ctx.camera_rays(cam, R, S))
    return cam, o, d, t


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("E", [5, 10])
@pytest.mark.parametrize("E_d", [0, 1, 4])
def test_encoder_with_directions(env, E, E_d):
    torch, api, ctx = env
    case = O.make_nerf_case(40 + E, 97, 13, E=E)
    o, d, t = (_cv(torch, case[k], torch.float64) for k in ("rays_o", "rays_d", "t"))
    X, dists = ctx.sample_encode(o, d, t, E, dir_bands=E_d)
    Xp, dists_p = ctx.sample_encode(o, d, t, E)
    ctx.synchronize()
    X, dists, Xp, dists_p = (v.cpu().numpy() for v in (X, dists, Xp, dists_p))
    ref, ref_dists = V.features(case["rays_o"], case["rays_d"], case["t"], E, E_d)
    assert X.shape == ref.shape == (97 * 13, 6 + 6 * E + 6 * E_d)
    assert (np.abs(X.astype(np.float64) - ref) <= np.spacing(np.abs(ref))).all()      # within one float32 ulp
    assert np.array_equal(dists, ref_dists) and np.array_equal(dists, dists_p)
    assert np.array_equal(X[:, :3 + 6 * E], Xp)                                          # positions bit for bit


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("E,E_d", [(5, 4), (10, 4)])
def test_exact_path_rays_and_camera_mode(env, E, E_d):
    torch, api, ctx = env
    R, S = 64, 32
    case = V.make_nerf_case(50 + E, R, S, E=E, E_dir=E_d)
    dims = [int(v) for v in case["dims"]]
    ws, bs, target = (_cv(torch, case[k]) for k in ("ws", "bs", "target"))
    o, d, t = (_cv(torch, case[k], torch.float64) for k in ("rays_o", "rays_d", "t"))
    out = _host(ctx.nerf_step_rays(dims, o, d, t, E, ws, bs, target, grad=True, path="f32", dir_bands=E_d))
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], dims, case["target"], case["dists"], R, S, g=1.0)
    errs = _errs(out, f)
    assert max(errs["loss"], errs["color"], errs["d_ws"], errs["d_bs"]) <= 1e-5, errs
    for stratified in (False, True):
        cam, co, cd, ct = _camera_batch(env, 48, R, S, 60 + E, stratified)
        X, dists = V.features(co, cd, ct, E, E_d)
        f = O.nerf_f64(X, case["ws"], case["bs"], dims, case["target"], dists, R, S, g=1.0)
        out = _host(ctx.nerf_step_camera(dims, cam, R, S, E, ws, bs, target, grad=True, path="f32", dir_bands=E_d))
        errs = _errs(out, f)
        assert max(errs["loss"], errs["color"], errs["d_ws"], errs["d_bs"]) <= 1e-5, (stratified, errs)


def test_zero_direction_rows_change_nothing_and_still_get_gradients(env):
    torch, api, ctx = env
    E, E_d, R, S = 5, 4, 50, 24
    case = O.make_nerf_case(71, R, S, E=E)
    d33 = [int(v) for v in case["dims"]]
    d60 = [60] + d33[1:]
    ws60 = np.zeros((3, 60, 30), np.float32)
    ws60[:, :33, :] = case["ws"]
    o, d, t = (_cv(torch, case[k], torch.float64) for k in ("rays_o", "rays_d", "t"))
    bs, target = _cv(torch, case["bs"]), _cv(torch, case["target"])
    # the layerwise exact kernels: layer 0 is an ascending k-sum in both nets, the direction rows add +0 terms
    a = _host(ctx.nerf_step_rays(d33, o, d, t, E, _cv(torch, case["ws"]), bs, target, grad=True, path="f32_layerwise"))
    b = _host(ctx.nerf_step_rays(d60, o, d, t, E, _cv(torch, ws60), bs, target, grad=True, path="f32_layerwise", dir_bands=E_d))
    assert np.array_equal(a["loss"], b["loss"]) and np.array_equal(a["color"], b["color"])
    assert np.abs(b["d_ws"][0, 33:60, :]).max() > 0                                # the gradient reaches the rows
    # one sample per ray: the same point seen along two different directions
    rng = np.random.default_rng(72)
    pts = rng.uniform(-0.5, 0.5, (R, 3))
    dir_a, dir_b = rng.normal(size=(R, 3)), rng.normal(size=(R, 3))
    tt = np.full((R, 1), 3.0)
    ws_dir = ws60.copy()
    ws_dir[0, 33:60, :] = rng.normal(0, 0.5, (27, 30)).astype(np.float32)
    cols = []
    for w in (ws60, ws_dir):
        c = []
        for dv in (dir_a, dir_b):
            ro = pts - dv * tt
            res = ctx.nerf_step_rays(d60, _cv(torch, ro, torch.float64), _cv(torch, dv, torch.float64),
                                     _cv(torch, tt, torch.float64), E, _cv(torch, w), bs, None, grad=False,
                                     outputs=("color",), path="f32", dir_bands=E_d)
            c.append(res["color"].cpu().numpy())
        cols.append(c)
    assert np.abs(cols[0][0] - cols[0][1]).max() <= 1e-5          # direction rows zero: only the (equal) points count
    assert np.abs(cols[1][0] - cols[1][1]).max() > 1e-2            # non-zero: the colour depends on the direction


# ---------------------------------------------------------------------------------------------------------------------
FUSED = [  # hidden width, layers, S, ray source
    (15, 2, 7, "f64"),
    (15, 4, 128, "cam"),
    (30, 3, 64, "f32"),
    (30, 3, 128, "cam"),
    (30, 2, 64, "cam_strat"),
    (48, 4, 64, "f64"),
    (63, 2, 7, "cam_strat"),
    (63, 3, 128, "f32"),
]


def _rays_step(env, dims, src, rays, cam, R, S, E, E_d, ws, bs, target, grad, path="tc"):
    torch, api, ctx = env
    kw = dict(grad=grad, seed=1.0, outputs=("color", "loss"), path=path, dir_bands=E_d)
    if src.startswith("cam"):
        return ctx.nerf_step_camera(dims, cam, R, S, E, ws, bs, target, **kw)
    dt = torch.float64 if src == "f64" else torch.float32
    o, d, t = (_cv(torch, v, dt) for v in rays)
    return ctx.nerf_step_rays(dims, o, d, t, E, ws, bs, target, **kw)


@pytest.mark.parametrize("H,L,S,src", FUSED)
def test_fused_kernels_with_directions(env, H, L, S, src, monkeypatch):
    torch, api, ctx = env
    E, E_d = 5, 4
    R = max(8, 6000 // S)
    rng = np.random.default_rng(80 + H + L + S)
    dims = O.mlp_dims(60, H, L, 4)
    ws, bs = O.init_mlp(rng, dims, 1.0)
    target = rng.uniform(0, 1, (R, 3)).astype(np.float32)
    cam = None
    if src.startswith("cam"):
        cam, o, d, t = _camera_batch(env, 96, R, S, 81 + S, src == "cam_strat")
    else:
        case = O.make_nerf_case(82 + S, R, S, E=E)
        o, d, t = case["rays_o"], case["rays_d"], case["t"]
        if src == "f32":
            o, d, t = (v.astype(np.float32).astype(np.float64) for v in (o, d, t))
    X, dists = V.features(o, d, t, E, E_d)
    wsd, bsd, tgd = _cv(torch, ws), _cv(torch, bs), _cv(torch, target)
    f = O.nerf_f64(X, ws, bs, dims, target, dists, R, S, g=1.0)
    Xd, distsd = ctx.sample_encode(*(_cv(torch, v, torch.float64) for v in (o, d, t)), E, dir_bands=E_d)
    for grad, kernel in ((True, "fused_mg_kernel<rays>"), (False, "fused_v1_kernel<rays>")):
        res = {}
        prof = ctx.profile_dominant(lambda: res.update(_rays_step(env, dims, src, (o, d, t), cam, R, S, E, E_d, wsd, bsd, tgd, grad)))
        assert prof is not None and prof["kernel"] == kernel, prof
        got = _host(res)
        feat = _host(ctx.nerf_step(dims, Xd, wsd, bsd, distsd, tgd, R=R, S=S, grad=grad, seed=1.0, path="tc"))
        if grad:
            errs = _errs(got, f)
            _check_tc(errs)
            fe = _errs(got, feat)
        else:
            errs = dict(color=rel_err(got["color"], f["color"]))
            assert errs["color"] <= TC_TOL, errs
            fe = dict(color=rel_err(got["color"], feat["color"]))
        print("fused H=%d L=%d S=%d %s grad=%d vs f64 %s vs features %s" % (H, L, S, src, grad, errs, fe))
        assert max(fe.values()) <= FEATURES_TOL, fe
    if L == 3 and H == 30:   # the one-tile-per-CTA train kernel (LNB_TC_V1) takes the same stage
        monkeypatch.setenv("LNB_TC_V1", "1")
        res = {}
        prof = ctx.profile_dominant(lambda: res.update(_rays_step(env, dims, src, (o, d, t), cam, R, S, E, E_d, wsd, bsd, tgd, True)))
        assert prof is not None and prof["kernel"] == "fused_v1_kernel<rays>", prof
        _check_tc(_errs(_host(res), f))


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("width,L,R,S", [(30, 3, 64, 32), (256, 3, 300, 64), (256, 9, 8, 192)])
def test_ninety_inputs_run_on_the_wide_path(env, width, L, R, S):
    torch, api, ctx = env
    E, E_d = 10, 4
    rng = np.random.default_rng(90 + L)
    dims = O.mlp_dims(90, width, L, 4)
    ws, bs = O.init_mlp(rng, dims, 1.0)
    target = rng.uniform(0, 1, (R, 3)).astype(np.float32)
    wsd, bsd, tgd = _cv(torch, ws), _cv(torch, bs), _cv(torch, target)
    case = O.make_nerf_case(91 + L, R, S, E=E)
    cam, co, cd, ct = _camera_batch(env, 64, R, S, 92, False)
    for src, rays in (("f64", (case["rays_o"], case["rays_d"], case["t"])), ("cam", (co, cd, ct))):
        X, dists = V.features(*rays, E, E_d)
        f = O.nerf_f64(X, ws, bs, dims, target, dists, R, S, g=1.0)
        res = {}
        prof = ctx.profile_dominant(lambda: res.update(_rays_step(env, dims, src, rays, cam, R, S, E, E_d, wsd, bsd, tgd, True)))
        assert prof is None or not prof["kernel"].startswith("fused_"), prof
        got = _host(res)
        errs = _errs(got, f)
        Xd, distsd = ctx.sample_encode(*(_cv(torch, v, torch.float64) for v in rays), E, dir_bands=E_d)
        feat = _host(ctx.nerf_step(dims, Xd, wsd, bsd, distsd, tgd, R=R, S=S, grad=True, seed=1.0, path="tc"))
        fe = _errs(got, feat)
        print("wide width=%d L=%d %s vs f64 %s vs features %s" % (width, L, src, errs, fe))
        assert max(errs["loss"], errs["color"], errs["d_ws"], errs["d_bs"], errs["d_ws_l2"], errs["d_bs_l2"]) <= WIDE_TOL, errs
        assert max(fe["loss"], fe["color"], fe["d_ws"], fe["d_bs"]) <= FEATURES_TOL, fe


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W", [37, 64])
def test_device_frame_render_with_directions(env, W):
    torch, api, ctx = env
    from loma_nerf_b200 import render
    E, E_d, S = 5, 4, 24
    K, pose = _scene(theta=75.0)
    dims = O.mlp_dims(60, 30, 3, 4)
    ws, bs = O.init_mlp(np.random.default_rng(100 + W), dims, 1.0)
    ref = render.render_frame(ctx, dims, ws, bs, W, W, K, pose, S, E, path="f32", dir_bands=E_d)
    want = np.rint(255 * ref.clip(0, 1)).astype(np.int32)
    for path, tol in (("f32", 1), ("tc", 4)):
        img = render.render_frame_device(ctx, dims, _cv(torch, ws), _cv(torch, bs), W, W, K, pose, S, E, path=path,
                                         rays_per_call=W * 3 + 11, dir_bands=E_d)
        ctx.synchronize()
        assert np.abs(img.cpu().numpy().astype(np.int32) - want).max() <= tol, (W, path)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c_in,E,path", [(60, 5, "tc"), (90, 10, "tc"), (60, 5, "f32")])
def test_trainer_with_directions_on_host_and_device(env, c_in, E, path):
    torch, api, ctx = env
    E_d, W, S, R = 4, 64, 32, 256
    K, pose = _scene()
    dims = O.mlp_dims(c_in, 30, 3, 4)
    ws, bs = O.init_mlp(np.random.default_rng(110 + c_in), dims, 1.0)
    rng = np.random.default_rng(111)
    pix = rng.choice(W * W, R, replace=False).astype(np.int32)
    target = rng.uniform(0, 1, (R, 3)).astype(np.float32)
    tr_d, tr_h, tr_f = (api.Trainer(ctx, dims, ws, bs) for _ in range(3))
    for it in range(3):
        cam_d = api.make_camera(pose, K, W, pixels=torch.as_tensor(pix).cuda(), stratified=True, seed=120 + it)
        tr_d.step(camera=cam_d, S=S, pe_bands=E, dir_bands=E_d, target=_cv(torch, target), path=path)
        cam_h = api.make_camera(pose, K, W, pixels=pix, stratified=True, seed=120 + it)
        tr_h.step_host(camera=cam_h, S=S, pe_bands=E, dir_bands=E_d, target=target, path=path)
        o, d, t = (v.cpu().numpy() for v in ctx.camera_rays(cam_d, R, S))
        X, dists = V.features(o, d, t, E, E_d)
        tr_f.step(X=_cv(torch, X), dists=_cv(torch, dists), target=_cv(torch, target), path=path)
    (wd, bd, ld), (wh, bh, lh), (wf, bf, lf) = tr_d.read(), tr_h.read(), tr_f.read()
    for tr in (tr_d, tr_h, tr_f):
        tr.close()
    close = lambda a, b, tol: float(np.abs(a - b).max()) <= tol * float(np.abs(b).max())  # noqa: E731
    # device and host routes: the same arithmetic, summed in MMA completion order on the tensor cores
    assert close(wd, wh, 2e-5) and close(bd, bh, 2e-5) and abs(ld - lh) <= 1e-5 * abs(lh)
    # against a trainer fed the host-built features: the exact path to 1e-5; on the tensor-core paths the two inputs
    # differ by the fp32 vs float64 encoding before the bf16 rounding, and 3 Adam steps of lr 5e-4 move a weight <= 1.5e-3
    if path == "f32":
        assert close(wd, wf, 1e-5) and close(bd, bf, 1e-5) and abs(ld - lf) <= 1e-5 * abs(lf), (ld, lf)
    else:
        assert close(wd, wf, 4e-3) and close(bd, bf, 4e-3) and abs(ld - lf) <= TC_TOL * abs(lf), (ld, lf)


# ---------------------------------------------------------------------------------------------------------------------
def test_refusals(env, monkeypatch):
    torch, api, ctx = env
    E, R, S = 5, 8, 16
    case = O.make_nerf_case(130, R, S, E=E)
    o, d, t = (_cv(torch, case[k], torch.float64) for k in ("rays_o", "rays_d", "t"))

    def net(c_in):
        dims = O.mlp_dims(c_in, 30, 3, 4)
        ws, bs = O.init_mlp(np.random.default_rng(131), dims, 1.0)
        return dims, _cv(torch, ws), _cv(torch, bs)

    # Python: dir_bands must describe dims[0]; refused before anything is launched
    n0 = ctx.launches
    for c_in, E_d in ((60, None), (60, 3), (33, 0), (90, 4)):
        dims, ws, bs = net(c_in)
        with pytest.raises(ValueError):
            ctx.nerf_step_rays(dims, o, d, t, E, ws, bs, None, grad=False, path="f32", dir_bands=E_d)
    assert ctx.launches == n0
    # the library reads the form off dims[0] alone: an even width that is not 6 + 6E + 6E_d, an odd one != 3 + 6E
    monkeypatch.setattr(api, "check_rays_width", lambda *a, **k: None)
    for c_in in (34, 58, 62, 35, 31):
        dims, ws, bs = net(c_in)
        for path in ("f32", "tc"):
            with pytest.raises(api.LnbError):
                ctx.nerf_step_rays(dims, o, d, t, E, ws, bs, None, grad=False, path=path)
