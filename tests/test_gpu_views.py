"""Views mode (lnb_views): camera mode with a pose per ray, and the per-step draw of a device-resident scene
(lnb_views_draw), against restatements of their rules, camera mode, rays mode on host-built rays, and eager steps."""
import ctypes
import json
import os

import numpy as np
import pytest

from conftest import rel_err
from oracle import oracle as O
from test_views_host import pick, z_of

pytestmark = pytest.mark.gpu

F64_EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def env():
    import torch
    from loma_nerf_b200 import api
    assert torch.cuda.is_available()
    c = api.Context(0)
    yield torch, api, c
    c.close()


def _K():
    f = 0.5 / np.tan(0.5 * 0.6911)
    return np.array([[f, 0, 0.5], [0, f, 0.5], [0, 0, 1]], np.float64)


def _scene(api, ctx, n_views=5, W=24, H=None, seed=0):
    from loma_nerf_b200 import render
    H = W if H is None else H
    rng = np.random.default_rng(seed)
    poses = np.stack([render.pose_spherical(360.0 * v / n_views + 7.0, -30.0 + 3 * v, 4.0) for v in range(n_views)])
    images = rng.uniform(0, 1, (n_views, H, W, 3)).astype(np.float32)
    return api.Scene(ctx, poses, images, _K(), near=2.0, far=6.0), poses, images


def _set(torch, b, view, pixels):
    b.view.copy_(torch.as_tensor(np.asarray(view, np.int32)))
    b.pixels.copy_(torch.as_tensor(np.asarray(pixels, np.int32)))


def _np(x):
    return x.detach().cpu().numpy()


def _cv(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()


# ---------------------------------------------------------------------------------------------------------------------
# the draw
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_views,W,H,R,seed", [(1, 8, 8, 1, 0), (5, 24, 16, 300, 7), (3, 40, 40, 1000, 2 ** 64 - 1),
                                                (100, 16, 16, 4096, 99)])
@pytest.mark.parametrize("one_view", [False, True])
def test_draw_follows_the_rule_and_advances_the_counter(env, n_views, W, H, R, seed, one_view):
    torch, api, ctx = env
    sc, _, images = _scene(api, ctx, n_views, W, H, seed=n_views)
    P = W * H
    b = sc.batch(R, one_view=one_view, seed=seed)
    flat = images.reshape(n_views, P, 3)
    for k in range(3):
        b.draw()
        ctx.synchronize()
        assert _np(b.counter).tolist() == [k + 1, 0]
        if one_view:
            v = np.full(R, pick(seed, k, 2 ** 32 - 1, n_views))
            q = np.array([pick(seed, k, r, P) for r in range(R)])
        else:
            g = np.array([pick(seed, k, r, n_views * P) for r in range(R)])
            v, q = g // P, g % P
        assert np.array_equal(_np(b.view), v) and np.array_equal(_np(b.pixels), q)
        assert np.array_equal(_np(b.target).view(np.uint32), flat[v, q].view(np.uint32))
        assert int(_np(b.step_seed)[0]) & (2 ** 64 - 1) == z_of(seed, k, 2 ** 32 - 2)


# ---------------------------------------------------------------------------------------------------------------------
# rays and depths
# ---------------------------------------------------------------------------------------------------------------------
def test_views_rays_are_each_views_get_rays(env):
    torch, api, ctx = env
    from loma_nerf_b200 import render
    n_views, W, S, R = 5, 24, 30, 400
    sc, poses, _ = _scene(api, ctx, n_views, W)
    rng = np.random.default_rng(3)
    view, pix = rng.integers(0, n_views, R), rng.integers(0, W * W, R)
    b = sc.batch(R)
    _set(torch, b, view, pix)
    o, d, t = (_np(x) for x in ctx.views_rays(b, S))
    for v in range(n_views):
        o_ref, d_ref = render.get_rays(W, W, _K(), poses[v])
        m = view == v
        assert np.array_equal(o[m], o_ref[pix[m]])
        assert np.abs(d[m] - d_ref[pix[m]]).max() <= 4 * F64_EPS * np.abs(d_ref).max()
    assert np.array_equal(t, np.broadcast_to(np.linspace(2.0, 6.0, S), (R, S)))
    # stratified: u = lnb_uniform(seed', view * P + q, s), seed' the device seed when set, else views.seed
    bs = sc.batch(R, stratified=True)
    _set(torch, bs, view, pix)
    g = view.astype(np.int64) * (W * W) + pix
    for dev_seed in (True, False):
        if dev_seed:
            bs.step_seed.fill_(123456789)
            seed = 123456789
        else:
            bs.views.seed_dev, bs.views.seed = None, 4242
            seed = 4242
        t = _np(ctx.views_rays(bs, S)[2])
        u = np.array([[ctx.lib.lnb_uniform(seed, int(g[r]), s) for s in range(S)] for r in range(R)])
        assert np.array_equal(t, 2.0 + (np.arange(S)[None, :] + u) * (6.0 - 2.0) / S)


# ---------------------------------------------------------------------------------------------------------------------
# views = camera
# ---------------------------------------------------------------------------------------------------------------------
CASES = [  # (path, width, dir_bands, background)
    ("f32", 30, None, None), ("f32_layerwise", 30, None, None), ("f32_layerwise", 30, 2, (1.0, 1.0, 1.0)),
    ("tc", 30, None, None), ("tc", 30, 2, None), ("tc", 30, 2, (1.0, 0.5, 0.25)), ("tc", 30, None, (1.0, 1.0, 1.0)),
    ("tc", 256, None, None), ("tc", 256, None, (1.0, 1.0, 1.0)),
]


@pytest.mark.parametrize("path,width,dir_bands,background", CASES)
@pytest.mark.parametrize("grad", [False, True])
def test_views_on_one_view_are_camera_mode_bit_for_bit(env, path, width, dir_bands, background, grad):
    torch, api, ctx = env
    n_views, W, S, E, R = 4, 32, 32, 5, 512
    sc, poses, _ = _scene(api, ctx, n_views, W)
    dims = O.mlp_dims(api.rays_input_width(E, dir_bands), width, 3, 4)
    ws, bs = O.init_mlp(np.random.default_rng(11), dims, 1.0)
    rng = np.random.default_rng(12)
    pix = rng.integers(0, W * W, R).astype(np.int32)
    target = _cv(torch, rng.uniform(0, 1, (R, 3)))
    outs = ("color", "loss") + (("acc", "depth") if background is not None else ()) + (("weights",) if path == "f32_layerwise" else ())
    kw = dict(grad=grad, seed=1.0, outputs=outs, path=path, dir_bands=dir_bands, background=background)
    for v, stratified in ((0, True), (0, False), (3, False)):
        cam = api.make_camera(poses[v], _K(), W, pixels=torch.as_tensor(pix).cuda(), stratified=stratified, seed=555)
        b = sc.batch(R, stratified=stratified)
        _set(torch, b, np.full(R, v), pix)
        b.views.seed_dev, b.views.seed = None, 555
        a = ctx.nerf_step_camera(dims, cam, R, S, E, _cv(torch, ws), _cv(torch, bs), target, **kw)
        c = ctx.nerf_step_views(dims, b, S, E, _cv(torch, ws), _cv(torch, bs), target, **kw)
        ctx.synchronize()
        for k in outs:
            assert np.array_equal(_np(a[k]), _np(c[k])), (v, stratified, k)
        if grad:
            for k in ("d_ws", "d_bs"):
                if path.startswith("f32"):
                    assert np.array_equal(_np(a[k]), _np(c[k])), (v, stratified, k)
                else:   # the tensor cores sum weight gradients in MMA completion order: last bits may differ per launch
                    np.testing.assert_allclose(_np(c[k]), _np(a[k]), rtol=0, atol=1e-6 * max(1.0, np.abs(_np(a[k])).max()))


# ---------------------------------------------------------------------------------------------------------------------
# mixed views against rays mode on host-built float64 rays
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path,tol", [("f32", 1e-5), ("tc", 3e-2)])
@pytest.mark.parametrize("stratified", [False, True])
def test_mixed_views_equal_rays_mode_on_host_built_rays(env, path, tol, stratified):
    torch, api, ctx = env
    from loma_nerf_b200 import render
    n_views, W, S, E, R = 6, 32, 30, 5, 384
    sc, poses, _ = _scene(api, ctx, n_views, W)
    dims = O.mlp_dims(3 + 6 * E, 30, 3, 4)
    ws, bs = O.init_mlp(np.random.default_rng(21), dims, 1.0)
    b = sc.batch(R, stratified=stratified, seed=5)
    b.draw()
    ctx.synchronize()
    view, pix = _np(b.view), _np(b.pixels)
    assert len(set(view.tolist())) > 1
    o = np.zeros((R, 3)); d = np.zeros((R, 3))
    for v in range(n_views):
        ov, dv = render.get_rays(W, W, _K(), poses[v])
        m = view == v
        o[m], d[m] = ov[pix[m]], dv[pix[m]]
    if stratified:
        seed = int(_np(b.step_seed)[0]) & (2 ** 64 - 1)
        g = view.astype(np.int64) * (W * W) + pix
        u = np.array([[ctx.lib.lnb_uniform(seed, int(g[r]), s) for s in range(S)] for r in range(R)])
        t = 2.0 + (np.arange(S)[None, :] + u) * 4.0 / S
    else:
        t = np.broadcast_to(np.linspace(2.0, 6.0, S), (R, S)).copy()
    f64 = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float64)).cuda()  # noqa: E731
    kw = dict(grad=True, seed=1.0, outputs=("color", "loss"), path=path)
    a = ctx.nerf_step_rays(dims, f64(o), f64(d), f64(t), E, _cv(torch, ws), _cv(torch, bs), b.target, **kw)
    c = ctx.nerf_step_views(dims, b, S, E, _cv(torch, ws), _cv(torch, bs), **kw)
    ctx.synchronize()
    errs = {k: rel_err(_np(c[k]), _np(a[k])) for k in ("loss", "color", "d_ws", "d_bs")}
    assert max(errs.values()) <= tol, errs


@pytest.mark.parametrize("path", ["f32", "tc"])
@pytest.mark.parametrize("bad", ["view", "pixel", "negative"])
def test_an_out_of_range_index_makes_that_ray_and_the_loss_nan(env, path, bad):
    torch, api, ctx = env
    n_views, W, S, E, R = 3, 16, 32, 5, 64
    sc, _, _ = _scene(api, ctx, n_views, W)
    dims = O.mlp_dims(3 + 6 * E, 30, 3, 4)
    ws, bs = O.init_mlp(np.random.default_rng(31), dims, 1.0)
    b = sc.batch(R, seed=1)
    b.draw()
    kw = dict(grad=False, outputs=("color", "loss"), path=path)
    a = ctx.nerf_step_views(dims, b, S, E, _cv(torch, ws), _cv(torch, bs), **kw)
    ctx.synchronize()
    a = {k: _np(v).copy() for k, v in a.items()}
    if bad == "view":
        b.view[5] = n_views
    elif bad == "pixel":
        b.pixels[5] = W * W
    else:
        b.view[5] = -1
    c = ctx.nerf_step_views(dims, b, S, E, _cv(torch, ws), _cv(torch, bs), **kw)
    ctx.synchronize()
    col = _np(c["color"])
    assert np.isnan(_np(c["loss"])[0])
    assert np.isnan(col[5]).all()
    keep = np.arange(R) != 5
    assert np.array_equal(col[keep], a["color"][keep])


# ---------------------------------------------------------------------------------------------------------------------
# trainer
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("route,width,path", [("fused", 30, "tc"), ("wide", 256, "tc"), ("exact", 30, "f32")])
def test_trainer_views_equals_trainer_camera(env, route, width, path):
    torch, api, ctx = env
    n_views, W, S, E, R = 4, 32, 32, 5, 512
    sc, poses, _ = _scene(api, ctx, n_views, W)
    dims = O.mlp_dims(3 + 6 * E, width, 3, 4)
    ws, bs = O.init_mlp(np.random.default_rng(41), dims, 1.0)
    rng = np.random.default_rng(42)
    pix = rng.integers(0, W * W, R).astype(np.int32)
    b = sc.batch(R)
    _set(torch, b, np.full(R, 2), pix)
    b.target.copy_(_cv(torch, rng.uniform(0, 1, (R, 3))))
    cam = api.make_camera(poses[2], _K(), W, pixels=torch.as_tensor(pix).cuda())
    tv, tc = api.Trainer(ctx, dims, ws, bs), api.Trainer(ctx, dims, ws, bs)
    try:
        wv, wc = (torch.zeros((R, S), device="cuda") for _ in range(2))
        tv.step(views=b, S=S, pe_bands=E, path=path)
        tc.step(camera=cam, S=S, pe_bands=E, target=b.target, path=path)
        tv.step_weights(wv, views=b, S=S, pe_bands=E, path=path)
        tc.step_weights(wc, camera=cam, S=S, pe_bands=E, target=b.target, path=path)
        tv.grad(views=b, S=S, pe_bands=E, path=path)
        tc.grad(camera=cam, S=S, pe_bands=E, target=b.target, path=path)
        tv.apply()
        tc.apply()
        (pv, qv, lv), (pc, qc, lc) = tv.read(), tc.read()
        assert np.array_equal(_np(wv), _np(wc)) and lv == lc
        if path == "f32":
            assert np.array_equal(pv, pc) and np.array_equal(qv, qc)
        else:
            np.testing.assert_allclose(pv, pc, rtol=0, atol=1e-6)
            np.testing.assert_allclose(qv, qc, rtol=0, atol=1e-6)
    finally:
        tv.close()
        tc.close()


@pytest.mark.parametrize("path", ["f32", "tc"])
def test_graph_of_draw_and_step_equals_eager_steps(env, path):
    torch, api, ctx = env
    n_views, W, S, E, R = 8, 32, 32, 5, 1024
    sc, _, _ = _scene(api, ctx, n_views, W)
    dims = O.mlp_dims(3 + 6 * E, 30, 3, 4)
    ws, bs = O.init_mlp(np.random.default_rng(51), dims, 1.0)
    kw = dict(S=S, pe_bands=E, path=path)

    def eager():
        tr, b = api.Trainer(ctx, dims, ws, bs), sc.batch(R, stratified=True, seed=9)
        losses, draws = [], []
        for _ in range(8):
            b.draw()
            tr.step(views=b, **kw)
            ctx.synchronize()
            losses.append(tr.read()[2])
            draws.append(_np(b.pixels).copy())
        p = tr.read()
        tr.close()
        return p, losses, draws

    def graphed():
        tr, b = api.Trainer(ctx, dims, ws, bs), sc.batch(R, stratified=True, seed=9)
        loss_log = torch.zeros(8, device="cuda")
        step_i = torch.zeros(1, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            ctx.set_stream(torch.cuda.current_stream())
            for i in range(4):
                b.draw()
                tr.step(views=b, **kw)
                loss_log.index_copy_(0, step_i, tr.grad_buffer()[-1:])
                step_i.add_(1)
        ctx.set_stream(torch.cuda.current_stream())
        # capture launched nothing: the counter is still at 0 and the parameters are the initial ones
        assert _np(b.counter).tolist() == [0, 0]
        draws = []
        for _ in range(2):
            g.replay()
            torch.cuda.synchronize()
            draws.append(_np(b.pixels).copy())
        p = tr.read()
        assert _np(b.counter).tolist() == [8, 0]
        tr.close()
        return p, _np(loss_log).tolist(), draws

    (pe, qe, _), le, de = eager()
    (pg, qg, _), lg, dg = graphed()
    assert not np.array_equal(dg[0], dg[1])
    assert np.array_equal(dg[0], de[3]) and np.array_equal(dg[1], de[7])
    if path == "f32":
        assert np.array_equal(pe, pg) and np.array_equal(qe, qg) and le == lg
    else:
        np.testing.assert_allclose(pg, pe, rtol=0, atol=1e-5)
        np.testing.assert_allclose(lg, le, rtol=1e-4)
    os.environ["LNB_NO_PDL"] = "1"
    try:
        _, ln, _ = graphed()
    finally:
        del os.environ["LNB_NO_PDL"]
    if path == "f32":
        assert ln == lg
    else:
        np.testing.assert_allclose(ln, lg, rtol=1e-4)


# ---------------------------------------------------------------------------------------------------------------------
# refusals and the Blender loader
# ---------------------------------------------------------------------------------------------------------------------
def test_refusals(env):
    torch, api, ctx = env
    sc, _, _ = _scene(api, ctx, 2, 16)
    E, S, R = 5, 16, 32
    dims = O.mlp_dims(3 + 6 * E, 30, 3, 4)
    ws, bs = O.init_mlp(np.random.default_rng(61), dims, 1.0)
    b = sc.batch(R)
    b.draw()
    tr = api.Trainer(ctx, dims, ws, bs)
    try:
        with pytest.raises(api.LnbError, match="views batch"):
            tr.step_host(views=b, S=S, pe_bands=E, path="f32")
        with pytest.raises(api.LnbError, match="views batch"):
            tr.submit_host(views=b, S=S, pe_bands=E, path="f32")
        tr.set_views(None)
        a = tr.prepare(target=b.target, R=R, S=S, path="f32")
        with pytest.raises(api.LnbError, match="X \\(or rays, or a camera\\)"):
            tr.step(prepared=a)
        with pytest.raises(ValueError):
            tr.step(views=b, S=S, pe_bands=E + 1, path="f32")
        with pytest.raises(ValueError):
            ctx.nerf_step_views(dims, b, S, E, _cv(torch, ws), _cv(torch, bs), dir_bands=1)
    finally:
        tr.close()
    # LNB_ERR_ARG cases of lnb_views
    from loma_nerf_b200 import _lib as L
    mlp = api.make_mlp(dims, ws.shape, L.HEAD_NERF)
    w_, b_ = _cv(torch, ws), _cv(torch, bs)
    for field, value in (("n_views", 0), ("width", 1), ("height", 0), ("fx", 0.0), ("view", None)):
        v = L.LnbViews.from_buffer_copy(b.views)
        setattr(v, field, value)
        a = L.LnbStepArgs()
        a.R, a.S, a.n_rows, a.target_w, a.ws, a.bs, a.target, a.pe_bands = R, S, R * S, 3, w_.data_ptr(), b_.data_ptr(), b.target.data_ptr(), E
        assert ctx.lib.lnb_nerf_step_views(ctx.h, ctypes.byref(mlp), ctypes.byref(a), ctypes.byref(v), None) == L.LNB_ERR_ARG, field
    v = L.LnbViews.from_buffer_copy(b.views)
    v.width, v.height = 65536, 32768
    assert ctx.lib.lnb_nerf_step_views(ctx.h, ctypes.byref(mlp), ctypes.byref(a), ctypes.byref(v), None) == L.LNB_ERR_ARG
    a.S = 4097
    assert ctx.lib.lnb_nerf_step_views(ctx.h, ctypes.byref(mlp), ctypes.byref(a), ctypes.byref(b.views), None) == L.LNB_ERR_ARG


def test_scene_from_blender(env, tmp_path):
    torch, api, ctx = env
    from PIL import Image
    from loma_nerf_b200 import render
    from loma_nerf_b200.dataset import BlenderScene
    rng = np.random.default_rng(71)
    frames = []
    for i in range(3):
        rgba = rng.integers(0, 256, (8, 8, 4), dtype=np.uint8)
        Image.fromarray(rgba, "RGBA").save(tmp_path / ("r_%d.png" % i))
        frames.append({"file_path": "./r_%d" % i, "transform_matrix": render.pose_spherical(40.0 * i, -30.0, 4.0).tolist()})
    with open(tmp_path / "transforms_train.json", "w") as fh:
        json.dump({"camera_angle_x": 0.6911, "frames": frames}, fh)
    for white in (False, True):
        bl = BlenderScene(str(tmp_path), img_size=8, white_background=white)
        sc = api.Scene.from_blender(ctx, bl)
        assert (sc.n_views, sc.width, sc.height) == (3, 8, 8)
        want = np.stack([bl[i]["image"] for i in range(3)]).reshape(3, 64, 3)
        assert np.array_equal(_np(sc.images), want)
        assert np.array_equal(_np(sc.poses), np.stack([bl[i]["pose"][:3, :4].reshape(12) for i in range(3)]))
        b = sc.batch(50, seed=3)
        b.draw()
        ctx.synchronize()
        assert np.array_equal(_np(b.target), want[_np(b.view), _np(b.pixels)])
