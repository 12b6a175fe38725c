"""Hierarchical sampling on the device: lnb_sample_pdf bit for bit against its float64 statement (oracle/hierarchical.py),
the coarse weights out of a trainer step on every route, the CoarseFine train step and the coarse-to-fine frame render."""
import numpy as np
import pytest

from conftest import rel_err
from oracle import hierarchical as Hs
from oracle import oracle as O
from oracle import tc_model as M
from oracle import viewdirs as V
from test_gpu_tc_model import adam_emulate, assert_update, live_masks

pytestmark = pytest.mark.gpu

TC_TOL, WIDE_TOL, EXACT_TOL = 3e-2, 6e-2, 1e-5   # each path against the float64 restatement
FUSED_MODEL_TOL = 4e-4                          # the fused kernels against the bf16 model (test_gpu_tc_model's "out")


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
    return x.detach().cpu().numpy()


def _inputs(rng, R, S, wkind, tkind):
    if tkind == "linspace":
        t = np.broadcast_to(np.linspace(2.0, 6.0, S), (R, S)).copy()
    elif tkind == "stratified":
        t = 2.0 + (np.arange(S)[None, :] + rng.uniform(0, 1, (R, S))) * 4.0 / S
    else:   # repeated depths
        t = np.sort(np.repeat(rng.uniform(2.0, 6.0, (R, (S + 1) // 2)), 2, axis=1)[:, :S], axis=1)
    if wkind == "random":
        w = rng.uniform(0, 1, (R, S)).astype(np.float32) ** 2
    elif wkind == "zero":
        w = np.zeros((R, S), np.float32)
    elif wkind == "onehot":
        w = np.zeros((R, S), np.float32)
        w[np.arange(R), rng.integers(0, S, R)] = 1.0
    else:   # subnormal float32 weights
        w = (rng.uniform(0, 1, (R, S)) * 1e-40).astype(np.float32)
    return np.ascontiguousarray(t), w


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [3, 4, 33, 64, 128, 192])
@pytest.mark.parametrize("n_fine", [1, 2, 31, 64, 128])
def test_sampler_bit_equal_to_the_rule(env, S, n_fine):
    torch, api, ctx = env
    rng = np.random.default_rng(1000 * S + n_fine)
    for k, wkind in enumerate(("random", "zero", "onehot", "subnormal")):
        tkind = ("linspace", "stratified", "repeated")[(k + S + n_fine) % 3]
        for stratified in (False, True):
            R = 1 if k == 3 else 37
            t, w = _inputs(rng, R, S, wkind, tkind)
            got = _np(ctx.sample_pdf(_cv(torch, t, torch.float64), _cv(torch, w), n_fine, stratified=stratified, seed=77,
                                     ray0=5000))
            want = Hs.sample_pdf_f64(t, w, n_fine, stratified=stratified, seed=77, ray0=5000)
            assert got.shape == (R, S + n_fine)
            assert np.array_equal(got, want), (wkind, tkind, stratified, np.abs(got - want).max())


def test_sampler_chunks_reproduce_the_whole_call(env):
    torch, api, ctx = env
    R, S, n = 301, 64, 128
    t, w = _inputs(np.random.default_rng(5), R, S, "random", "stratified")
    td, wd = _cv(torch, t, torch.float64), _cv(torch, w)
    whole = _np(ctx.sample_pdf(td, wd, n, stratified=True, seed=3, ray0=900))
    parts = [_np(ctx.sample_pdf(td[a:b].contiguous(), wd[a:b].contiguous(), n, stratified=True, seed=3, ray0=900 + a))
             for a, b in ((0, 100), (100, 255), (255, 301))]
    assert np.array_equal(np.concatenate(parts), whole)
    assert np.array_equal(whole, Hs.sample_pdf_f64(t, w, n, stratified=True, seed=3, ray0=900))


def test_sampler_refusals_and_empty_batch(env):
    torch, api, ctx = env
    t = _cv(torch, np.linspace(2, 6, 8)[None, :].repeat(4, 0), torch.float64)
    w = _cv(torch, np.ones((4, 8), np.float32))
    for bad in (lambda: ctx.sample_pdf(t.float(), w, 4), lambda: ctx.sample_pdf(t, w.double(), 4),
                lambda: ctx.sample_pdf(t, w[:3].contiguous(), 4),
                lambda: ctx.sample_pdf(t, w, 4, out=torch.empty((4, 11), dtype=torch.float64, device=t.device))):
        with pytest.raises(ValueError):
            bad()
    with pytest.raises(api.LnbError):
        ctx._check(ctx.lib.lnb_sample_pdf(ctx.h, None, w.data_ptr(), 4, 8, 4, 0, 0, 0, t.data_ptr()))
    for S, n in ((2, 4), (8, 0), (8, 4089)):
        ts = _cv(torch, np.linspace(2, 6, S)[None, :].repeat(4, 0), torch.float64)
        ws = _cv(torch, np.ones((4, S), np.float32))
        with pytest.raises(api.LnbError):
            ctx.sample_pdf(ts, ws, n)
    t8 = np.ones((4, 8)) * np.arange(8.0)
    ok = ctx.sample_pdf(_cv(torch, t8, torch.float64), w, 4088, stratified=True)   # S + n_fine = 4096
    assert np.array_equal(_np(ok), Hs.sample_pdf_f64(t8, np.ones((4, 8), np.float32), 4088, stratified=True))
    n0 = ctx.launches
    e = ctx.sample_pdf(torch.empty((0, 8), dtype=torch.float64, device=t.device),
                       torch.empty((0, 8), dtype=torch.float32, device=t.device), 4)
    assert tuple(e.shape) == (0, 12) and ctx.launches == n0


# ---------------------------------------------------------------------------------------------------------------------
ROUTES = [  # route, input width, hidden width, layers, R, S, path, kernel the profiler names (None: no dominant kernel)
    ("fused", 33, 30, 3, 256, 64, "tc", "fused_mg_kernel"),
    ("wide", 90, 256, 9, 24, 64, "tc", "chain_tc_kernel"),
    ("exact", 33, 30, 3, 64, 64, "f32", None),
]


@pytest.mark.parametrize("route,c_in,H,L,R,S,path,kernel", ROUTES)
def test_trainer_step_weights(env, monkeypatch, route, c_in, H, L, R, S, path, kernel):
    torch, api, ctx = env
    if c_in == 33:
        case = O.make_nerf_case(300 + R, R, S, E=5, width=H, n_layers=L)
    else:
        case = V.make_nerf_case(300 + R, R, S, E=10, E_dir=4, width=H, n_layers=L)
    dims = [int(v) for v in case["dims"]]
    batch = dict(X=_cv(torch, case["X"]), dists=_cv(torch, case["dists"]), target=_cv(torch, case["target"]), path=path)
    tr_w, tr_p = api.Trainer(ctx, dims, case["ws"], case["bs"]), api.Trainer(ctx, dims, case["ws"], case["bs"])
    try:
        w = torch.full((R, S), float("nan"), dtype=torch.float32, device="cuda")
        prof = ctx.profile_dominant(lambda: tr_w.step_weights(w, **batch))
        if kernel is None:
            assert prof is None or not prof["kernel"].startswith("fused_"), prof
        else:
            assert prof is not None and prof["kernel"].startswith(kernel), prof
        g = _np(tr_w.grad_buffer()).copy()
        if route == "exact":   # the step with weights runs on the layerwise kernels: the plain step the same way
            monkeypatch.setenv("LNB_F32_NO_FUSED", "1")
        tr_p.step(**batch)
        monkeypatch.delenv("LNB_F32_NO_FUSED", raising=False)
        (ww, bw, lw), (wp, bp, lp) = tr_w.read(), tr_p.read()
        got_w = _np(w)
        f = O.nerf_f64(case["X"], case["ws"], case["bs"], dims, case["target"], case["dists"], R, S, g=1.0)
        tol = dict(fused=TC_TOL, wide=WIDE_TOL, exact=EXACT_TOL)[route]
        e64 = rel_err(got_w, f["weights"])
        msg = "step_weights %s: weights vs f64 %.3g" % (route, e64)
        assert np.isfinite(got_w).all() and e64 <= tol, msg
        if route == "fused":
            m = M.nerf_tc_model(case["X"], case["ws"], case["bs"], dims, case["target"], case["dists"], R, S, 1.0, "fused")
            em = rel_err(got_w, m["weights"])
            msg += ", vs the bf16 model %.3g" % em
            assert em <= FUSED_MODEL_TOL, msg
        print(msg)
        assert lw == lp, (lw, lp)                       # the loss bit for bit
        p0 = np.concatenate([case["ws"].ravel(), case["bs"].ravel()]).astype(np.float32)
        got = np.concatenate([ww.ravel(), bw.ravel()])
        live = live_masks(dims, case["ws"].shape, case["bs"].shape)
        if route == "fused":
            m0, v0 = np.zeros_like(p0), np.zeros_like(p0)
            assert_update(got, p0, adam_emulate(p0, g[:-1], m0, v0, 1, 5e-4, 0.9, 0.999, 1e-8), live)
        else:
            assert_update(got, p0, np.concatenate([wp.ravel(), bp.ravel()]), live)
    finally:
        tr_w.close()
        tr_p.close()


def test_step_weights_refuses_a_wrong_buffer(env):
    torch, api, ctx = env
    case = O.make_nerf_case(330, 8, 16)
    tr = api.Trainer(ctx, [int(v) for v in case["dims"]], case["ws"], case["bs"])
    with pytest.raises(ValueError):
        tr.step_weights(torch.empty((8, 15), dtype=torch.float32, device="cuda"), X=_cv(torch, case["X"]),
                        dists=_cv(torch, case["dists"]), target=_cv(torch, case["target"]))
    tr.close()


# ---------------------------------------------------------------------------------------------------------------------
def _scene(theta=35.0):
    from loma_nerf_b200 import render
    focal = 0.5 / np.tan(0.5 * 0.6911)
    K = np.array([[focal, 0, 0.5], [0, focal, 0.5], [0, 0, 1]], np.float64)
    return K, render.pose_spherical(theta, -30.0, 4.0)


CF = [  # input width (E, E_d), hidden width, layers, S, n_fine, R, batch form, tolerance
    (5, None, 30, 3, 64, 64, 128, "cam", TC_TOL),
    (5, None, 30, 3, 64, 64, 128, "rays", TC_TOL),
    (5, 4, 30, 3, 64, 64, 128, "cam", TC_TOL),
    (5, 4, 30, 3, 64, 64, 128, "rays", TC_TOL),
    (10, 4, 256, 9, 64, 128, 24, "cam", WIDE_TOL),
]


@pytest.mark.parametrize("E,E_d,H,L,S,n_fine,R,form,tol", CF)
def test_coarse_fine_step(env, E, E_d, H, L, S, n_fine, R, form, tol):
    torch, api, ctx = env
    rng = np.random.default_rng(400 + E + H + R)
    dims = O.mlp_dims(api.rays_input_width(E, E_d), H, L, 4)
    (wc, bc), (wf, bf) = O.init_mlp(rng, dims, 1.0), O.init_mlp(rng, dims, 1.0)
    target = rng.uniform(0, 1, (R, 3)).astype(np.float32)
    coarse, fine = api.Trainer(ctx, dims, wc, bc), api.Trainer(ctx, dims, wf, bf)
    cf = api.CoarseFine(coarse, fine, n_fine)
    K, pose = _scene()
    W = 64
    pix = rng.choice(W * W, R, replace=False).astype(np.int32)
    cam = api.make_camera(pose, K, W, pixels=torch.as_tensor(pix).cuda(), stratified=True, seed=410)
    try:
        if form == "cam":
            out = cf.step(camera=cam, S=S, pe_bands=E, dir_bands=E_d, target=_cv(torch, target), path="tc")
            seed = 410
        else:
            o, d, t = ctx.camera_rays(cam, R, S)
            out = cf.step(rays=(o, d, t), pe_bands=E, dir_bands=E_d, target=_cv(torch, target), path="tc", seed=411)
            seed = 411
        o, d, t, w, tf = (_np(out[k]) for k in ("o", "d", "t", "w", "t_fine"))
        assert np.array_equal(tf, Hs.sample_pdf_f64(t, w, n_fine, stratified=True, seed=seed, ray0=0))
        _, _, loss_f = fine.read()
        _, _, loss_c = coarse.read()
        X, dists = V.features(o, d, t, E, E_d)
        fc = O.nerf_f64(X, wc, bc, dims, target, dists, R, S, g=1.0)
        Xf, dists_f = V.features(o, d, tf, E, E_d)
        ff = O.nerf_f64(Xf, wf, bf, dims, target, dists_f, R, S + n_fine, g=1.0)
        errs = dict(weights=rel_err(w, fc["weights"]), coarse_loss=rel_err(loss_c, fc["loss"]), fine_loss=rel_err(loss_f, ff["loss"]))
        print("coarse-fine %s E_d=%s H=%d L=%d %d+%d: %s" % (form, E_d, H, L, S, n_fine, errs))
        assert max(errs.values()) <= tol, errs
    finally:
        coarse.close()
        fine.close()


def test_coarse_fine_exact_path_end_to_end(env):
    torch, api, ctx = env
    E, S, n_fine, R = 5, 64, 64, 48
    rng = np.random.default_rng(450)
    dims = O.mlp_dims(33, 30, 3, 4)
    (wc, bc), (wf, bf) = O.init_mlp(rng, dims, 1.0), O.init_mlp(rng, dims, 1.0)
    case = O.make_nerf_case(451, R, S, E=E)
    target = case["target"]
    coarse, fine = api.Trainer(ctx, dims, wc, bc), api.Trainer(ctx, dims, wf, bf)
    cf = api.CoarseFine(coarse, fine, n_fine)
    try:
        rays = tuple(_cv(torch, case[k], torch.float64) for k in ("rays_o", "rays_d", "t"))
        out = cf.step(rays=rays, pe_bands=E, target=_cv(torch, target), path="f32", seed=452)
        rc, tf_ref, rf = Hs.coarse_fine_f64(case["rays_o"], case["rays_d"], case["t"], (dims, wc, bc), (dims, wf, bf), target,
                                           E, n_fine, stratified=True, seed=452, g=1.0)
        tf = _np(out["t_fine"])
        errs = dict(weights=rel_err(_np(out["w"]), rc["weights"]), t_fine=float(np.abs(tf - tf_ref).max()),
                    coarse_loss=rel_err(coarse.read()[2], rc["loss"]), fine_loss=rel_err(fine.read()[2], rf["loss"]))
        print("coarse-fine exact path vs coarse_fine_f64: %s" % errs)
        # weights within the exact path's 1e-5; a depth moves by the cdf's error times the bin width over the bin's mass
        assert errs["weights"] <= EXACT_TOL and errs["coarse_loss"] <= EXACT_TOL, errs
        assert errs["t_fine"] <= 1e-3 and errs["fine_loss"] <= 1e-3, errs
    finally:
        coarse.close()
        fine.close()


def test_coarse_fine_graph_equals_eager(env):
    torch, api, ctx = env
    E, S, n_fine, R, W = 5, 32, 32, 64, 48
    rng = np.random.default_rng(460)
    dims = O.mlp_dims(33, 30, 3, 4)
    (wc, bc), (wf, bf) = O.init_mlp(rng, dims, 1.0), O.init_mlp(rng, dims, 1.0)
    target = _cv(torch, rng.uniform(0, 1, (R, 3)).astype(np.float32))
    K, pose = _scene(50.0)
    pix = torch.as_tensor(rng.choice(W * W, R, replace=False).astype(np.int32)).cuda()
    cams = [api.make_camera(pose, K, W, pixels=pix, stratified=True, seed=461 + i) for i in range(4)]
    pairs = [(api.Trainer(ctx, dims, wc, bc), api.Trainer(ctx, dims, wf, bf)) for _ in range(2)]
    eager, graphed = (api.CoarseFine(c, f, n_fine) for c, f in pairs)
    kw = dict(S=S, pe_bands=E, target=target, path="f32")
    try:
        for cf in (eager, graphed):            # the first step allocates the buffers
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
        assert np.array_equal(_np(eager._buf["t_fine"]), _np(graphed._buf["t_fine"]))
    finally:
        for c, f in pairs:
            c.close()
            f.close()


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["tc", "f32"])
def test_render_frame_with_fine_pass(env, path):
    torch, api, ctx = env
    from loma_nerf_b200 import render
    E, S, n_fine, W, chunk = 5, 32, 32, 40, 611
    rng = np.random.default_rng(470)
    dims = O.mlp_dims(33, 30, 3, 4)
    (wc, bc), (wf, bf) = O.init_mlp(rng, dims, 1.0), O.init_mlp(rng, dims, 1.0)
    wc_d, bc_d, wf_d, bf_d = (_cv(torch, a) for a in (wc, bc, wf, bf))
    K, pose = _scene(75.0)
    img = render.render_frame_device(ctx, dims, wc_d, bc_d, W, W, K, pose, S, E, path=path, rays_per_call=chunk,
                                     fine=(dims, wf_d, bf_d, n_fine))
    # the same pipeline from the individual calls
    n = W * W
    color = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    for r0 in range(0, n, chunk):
        k = min(n, r0 + chunk) - r0
        cam = api.make_camera(pose, K, W, W, first_pixel=r0)
        o, d, t = ctx.camera_rays(cam, k, S)
        w = ctx.nerf_step_camera(dims, cam, k, S, E, wc_d, bc_d, outputs=("weights",), path=path)["weights"]
        tf = ctx.sample_pdf(t, w, n_fine, ray0=r0)
        color[r0:r0 + k] = ctx.nerf_step_rays(dims, o, d, tf, E, wf_d, bf_d, outputs=("color",), path=path)["color"]
    want = ctx.color_to_u8(color).reshape(W, W, 3)
    ctx.synchronize()
    assert np.array_equal(_np(img), _np(want))
    # the host-buffer form renders the frame in one call: the same rays, chunked differently
    host = render.render_frame(ctx, dims, wc, bc, W, W, K, pose, S, E, path=path, fine=(dims, wf, bf, n_fine))
    diff = np.abs(np.rint(255 * host.clip(0, 1)).astype(np.int32) - _np(img).astype(np.int32)).max()
    print("render %s: one call vs chunks of %d rays, max difference %d levels" % (path, chunk, diff))
    assert diff <= 1
