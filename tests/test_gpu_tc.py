"""Tensor-core path (LNB_PATH_TC, fused_tc.cu): bf16 operands, fp32 accumulation in TMEM.
Compared with the reference golden vectors and the float64 restatement under the bf16 bound stated
in DESIGN.md 2.2: norm-wise relative error <= TC_TOL on loss, colour and weight gradients (measured
7e-5 .. 2e-3 on loss, 1e-3 .. 2e-2 on gradients).  These bounds check the semantics and absorb the
whole bf16 error; the kernels' own arithmetic is held 100x tighter in test_gpu_tc_model.py, against
the bf16-faithful model oracle/tc_model.py (4e-4 on colour, 6e-5 on gradients for the fused kernels,
measured on one B200 at 1000 W: DESIGN.md 2.2)."""
import os

import numpy as np
import pytest

from conftest import golden_files, grad_errs, load_golden, rel_err
from oracle import oracle as O

pytestmark = pytest.mark.gpu
TC_TOL = 3e-2     # bf16 operands: 2^-9 relative per element; measured errors are logged below
# The gradient bounds are stated three ways (DESIGN.md 2.2 "Numerics"): norm-wise over the whole padded array
# (TC_TOL), PER LAYER (max|a_l-b_l| / max|b_l|: a small layer cannot hide behind a large one) and in L2.
TC_LAYER_TOL = 4e-2
TC_L2_TOL = 2e-2


def check_grads(errs):
    assert max(errs["d_ws"], errs["d_bs"]) <= TC_TOL, errs
    assert max(errs["d_ws_layer"], errs["d_bs_layer"]) <= TC_LAYER_TOL, errs
    assert max(errs["d_ws_l2"], errs["d_bs_l2"]) <= TC_L2_TOL, errs


NERF_GOLDEN = [p for p in golden_files("nerf_") if "c5" not in p and "s192" not in p]
FIT_GOLDEN = golden_files("fit_")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module")
def ctx(torch_cuda):
    from loma_nerf_b200 import api
    c = api.Context(0)
    yield c
    c.close()


def dev(torch, a):
    return torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda().contiguous()


def host(t):
    return t.detach().cpu().numpy()


def log(msg):
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/tc_errors.log", "a") as fh:
        fh.write(msg + "\n")


def run_tc(ctx, torch, case, seed, grad=True, outputs=("color", "loss")):
    R, S = int(case["R"]), int(case["S"])
    out = ctx.nerf_step([int(v) for v in case["dims"]], dev(torch, case["X"]), dev(torch, case["ws"]),
                        dev(torch, case["bs"]), dev(torch, case["dists"]), dev(torch, case["target"]),
                        R=R, S=S, grad=grad, seed=seed, outputs=outputs, path="tc")
    ctx.synchronize()
    return {k: host(v) for k, v in out.items()}


@pytest.mark.parametrize("gpath", NERF_GOLDEN, ids=os.path.basename)
def test_tc_nerf_against_reference_golden(ctx, torch_cuda, gpath):
    gd = load_golden(gpath)
    o = run_tc(ctx, torch_cuda, gd, "loss")
    errs = dict(loss=rel_err(o["loss"][0], gd["loss"]), color=rel_err(o["color"], gd["color"]), **grad_errs(o, gd))
    log("%s %s" % (os.path.basename(gpath), errs))
    assert max(errs["loss"], errs["color"]) <= TC_TOL, errs
    check_grads(errs)


@pytest.mark.parametrize("gpath", FIT_GOLDEN, ids=os.path.basename)
def test_tc_fit_against_reference_golden(ctx, torch_cuda, gpath):
    torch = torch_cuda
    gd = load_golden(gpath)
    out = ctx.fit_step([int(v) for v in gd["dims"]], dev(torch, gd["X"]), dev(torch, gd["ws"]), dev(torch, gd["bs"]),
                       dev(torch, gd["target"]), grad=True, seed="loss", outputs=("loss",), path="tc")
    ctx.synchronize()
    o = {k: host(v) for k, v in out.items()}
    errs = dict(loss=rel_err(o["loss"][0], gd["loss"]), **grad_errs(o, gd))
    log("%s %s" % (os.path.basename(gpath), errs))
    assert errs["loss"] <= TC_TOL, errs
    check_grads(errs)


@pytest.mark.parametrize("R,S", [(4096, 64), (1000, 30), (257, 128), (64, 32), (700, 7)])
def test_tc_full_batches_against_f64_restatement(ctx, torch_cuda, R, S):
    case = O.make_nerf_case(500 + S, R, S)
    o = run_tc(ctx, torch_cuda, case, 1.0)
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=1.0)
    errs = dict(loss=rel_err(o["loss"][0], f["loss"]), color=rel_err(o["color"], f["color"]), **grad_errs(o, f))
    log("R=%d S=%d %s" % (R, S, errs))
    assert max(errs["loss"], errs["color"]) <= TC_TOL, errs
    check_grads(errs)


def test_tc_render_only_and_unsupported_requests(ctx, torch_cuda):
    torch = torch_cuda
    from loma_nerf_b200 import api
    case = O.make_nerf_case(610, 300, 64)
    dims = [int(v) for v in case["dims"]]
    out = ctx.nerf_step(dims, dev(torch, case["X"]), dev(torch, case["ws"]), dev(torch, case["bs"]),
                        dev(torch, case["dists"]), None, grad=False, outputs=("color",), path="tc")
    ctx.synchronize()
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], 300, 64)
    assert rel_err(host(out["color"]), f["color"]) <= TC_TOL
    # per-sample by-products are not produced by the fused kernel: refused, never silently rerouted
    with pytest.raises(api.LnbError):
        ctx.nerf_step(dims, dev(torch, case["X"]), dev(torch, case["ws"]), dev(torch, case["bs"]),
                      dev(torch, case["dists"]), dev(torch, case["target"]), grad=True, outputs=("d_X",), path="tc")


@pytest.mark.parametrize("dtype", ["float64", "float32"])
@pytest.mark.parametrize("R,S,E", [(4096, 64, 5), (333, 30, 5), (200, 128, 5), (64, 64, 10), (100, 7, 2)])
def test_tc_rays_mode_fused_positional_encoding(ctx, torch_cuda, R, S, E, dtype):
    """Rays mode: sample positions, positional encoding and dists computed inside the fused kernel
    (train_nerf.py:289-311 + pos_encoding.py:38-70), checked against the float64 restatement fed
    with the host-built features."""
    torch = torch_cuda
    width = 30
    case = O.make_nerf_case(700 + S + E, R, S, E=E, width=width)
    tdt = getattr(torch, dtype)
    cvr = lambda a: torch.as_tensor(np.ascontiguousarray(a)).to(tdt).cuda().contiguous()  # noqa: E731
    out = ctx.nerf_step_rays([int(v) for v in case["dims"]], cvr(case["rays_o"]), cvr(case["rays_d"]), cvr(case["t"]), E,
                             dev(torch, case["ws"]), dev(torch, case["bs"]), dev(torch, case["target"]), grad=True,
                             seed=1.0, outputs=("color", "loss"), path="tc")
    ctx.synchronize()
    o = {k: host(v) for k, v in out.items()}
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=1.0)
    errs = dict(loss=rel_err(o["loss"][0], f["loss"]), color=rel_err(o["color"], f["color"]), **grad_errs(o, f))
    log("rays %s R=%d S=%d E=%d %s" % (dtype, R, S, E, errs))
    assert max(errs["loss"], errs["color"]) <= TC_TOL, errs
    check_grads(errs)


@pytest.mark.parametrize("path,tol", [("f32", 2e-5), ("tc", 5e-2)])
def test_trainer_follows_the_reference_host_loop(ctx, torch_cuda, path, tol):
    """lnb_trainer (weights, Adam state and gradients resident on the device) against the reference
    host loop restated with the float64 oracle gradients and numpy Adam (train_nerf.py:133-161,
    :395-499): 5 steps on different ray batches, features in and rays in."""
    torch = torch_cuda
    from loma_nerf_b200 import api
    R, S, E = 256, 64, 5
    cases = [O.make_nerf_case(900 + i, R, S) for i in range(5)]
    ws0, bs0 = cases[0]["ws"].copy(), cases[0]["bs"].copy()
    dims = [int(v) for v in cases[0]["dims"]]
    lr, b1, b2, eps = 5e-4, 0.9, 0.999, 1e-8
    ws, bs = ws0.astype(np.float64), bs0.astype(np.float64)
    m = [np.zeros_like(ws), np.zeros_like(bs)]; v = [np.zeros_like(ws), np.zeros_like(bs)]
    losses = []
    for t, c in enumerate(cases, start=1):
        f = O.nerf_f64(c["X"], ws.astype(np.float32), bs.astype(np.float32), c["dims"], c["target"], c["dists"], R, S, g=1.0)
        losses.append(f["loss"])
        lr_t = lr * (np.sqrt(1 - b2 ** t) / (1 - b1 ** t))
        for i, (p_, g_) in enumerate(((ws, f["d_ws"]), (bs, f["d_bs"]))):
            m[i] = b1 * m[i] + (1 - b1) * g_
            v[i] = b2 * v[i] + (1 - b2) * g_ ** 2
            p_ -= lr_t * (m[i] / (1 - b1 ** t)) / (np.sqrt(v[i] / (1 - b2 ** t)) + eps)
    for mode in ("features", "rays"):
        tr = api.Trainer(ctx, dims, ws0, bs0, optimizer="adam", lr=lr, beta1=b1, beta2=b2, eps=eps)
        got_losses = []
        for i, c in enumerate(cases):
            tg = dev(torch, c["target"])
            if mode == "features":
                batch = dict(X=dev(torch, c["X"]), dists=dev(torch, c["dists"]), target=tg, path=path)
            else:
                rays = tuple(torch.as_tensor(np.ascontiguousarray(c[k])).cuda() for k in ("rays_o", "rays_d", "t"))
                batch = dict(rays=rays, pe_bands=E, target=tg, path=path)
            if i % 2 == 0:
                tr.step(**batch)
            else:                      # the split form used for data-parallel training
                tr.grad(**batch)
                g = tr.grad_buffer()
                assert g.numel() == ws0.size + bs0.size + 1
                tr.apply()
            got_losses.append(tr.read()[2])
        w, b, _ = tr.read()
        tr.close()
        errs = dict(ws=rel_err(w, ws), bs=rel_err(b, bs), loss=rel_err(got_losses, losses))
        log("trainer %s %s %s" % (path, mode, errs))
        # Adam normalises every step to ~lr * sign(g): where a gradient entry is below the bf16 noise
        # its sign (hence the whole update of that entry) is arbitrary, so the tensor-core path is
        # held to an L2 bound on the update vector; the exact path to a max-norm one
        du, dr = (w - ws0).ravel().astype(np.float64), (ws - ws0).ravel()
        upd_l2 = float(np.linalg.norm(du - dr) / np.linalg.norm(dr))
        upd_max = rel_err(du, dr)
        log("trainer %s %s update error: l2 %.3g max %.3g" % (path, mode, upd_l2, upd_max))
        assert errs["loss"] <= tol, errs
        assert (upd_l2 <= 0.15) if path == "tc" else (upd_max <= 1e-3), (upd_l2, upd_max)


def test_training_on_a_synthetic_scene_improves_psnr(ctx, torch_cuda):
    """End-to-end quality check of the trainer in rays mode (the reference logs PSNR 12.3 -> 14.8 dB
    over its first 25 iterations, logs_3d/25.png): fit a fixed set of rays whose target colours come
    from a different random MLP, and require the training loss to fall and PSNR to rise."""
    torch = torch_cuda
    from loma_nerf_b200 import api, render
    rng = np.random.default_rng(5)
    E, S, R = 5, 64, 4096
    dims = O.mlp_dims(3 + 6 * E, 30, 3, 4)
    ws_t, bs_t = O.init_mlp(np.random.default_rng(50), dims, 1.0)       # "ground-truth" field
    ws0, bs0 = O.init_mlp(np.random.default_rng(51), dims, 1.0)
    o, d = O.synthetic_rays(rng, R, n_views=4)
    t = O.stratified_t(rng, R, S)
    target = render.render_rays(ctx, dims, ws_t, bs_t, o, d, t, E, path="f32")
    rays = tuple(torch.as_tensor(v).cuda() for v in (o, d, t))
    tg = torch.as_tensor(target).cuda()
    for path, n_it in (("tc", 300), ("f32", 60)):
        tr = api.Trainer(ctx, dims, ws0, bs0, optimizer="adam", lr=5e-3)
        losses = []
        for it in range(n_it):
            tr.step(rays=rays, pe_bands=E, target=tg, path=path)
            if it % 20 == 0 or it == n_it - 1:
                losses.append(tr.read()[2])
        w, b, _ = tr.read()
        tr.close()
        before = render.compute_psnr(render.render_rays(ctx, dims, ws0, bs0, o, d, t, E, path="f32"), target)
        after = render.compute_psnr(render.render_rays(ctx, dims, w, b, o, d, t, E, path="f32"), target)
        log("train-demo %s: loss %.2f -> %.2f, PSNR %.2f -> %.2f dB" % (path, losses[0], losses[-1], before, after))
        assert losses[-1] < 0.7 * losses[0] and after > before + 1.0, (path, losses, before, after)


def test_context_runs_on_torchs_current_stream_by_default(torch_cuda):
    """The library's kernels and torch's own work on the same tensors (zero fills, collectives, allocator
    reuse) must be ordered without the caller doing anything: a new Context adopts torch's current stream."""
    torch = torch_cuda
    from loma_nerf_b200 import api
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        c = api.Context(0)
        assert c._stream_raw == side.cuda_stream and c._on_torch_current()
    assert not c._on_torch_current()          # torch moved back to its default stream, the context did not
    # a step issued now is ordered behind torch's current stream (order_after_torch) and its inputs are
    # recorded on the context's stream; results must not depend on the race either way
    case = O.make_nerf_case(333, 64, 64)
    o = run_tc(c, torch, case, 1.0)
    c2 = api.Context(0)
    assert c2._on_torch_current()
    o2 = run_tc(c2, torch, case, 1.0)
    # colours are a per-ray computation (bit-identical); the weight gradients of one launch are accumulated in TMEM by several
    # issuing threads / groups in completion order, so their last bits may differ between launches (fp32 addition order)
    assert np.array_equal(o["color"], o2["color"])
    assert rel_err(o["d_ws"], o2["d_ws"]) <= 1e-5 and rel_err(o["d_bs"], o2["d_bs"]) <= 1e-5
    c.close(); c2.close()


def test_trainer_takes_an_empty_batch_and_a_batch_the_fused_kernel_cannot(ctx, torch_cuda):
    """(1) R = 0 (a rank whose shard is empty when R < world): the step counter still advances and nothing
    becomes NaN.  (2) S = 192 on the 30-wide net: the MLP fits the fused kernel, the batch does not --
    lnb_trainer_step falls through to the layerwise tensor-core kernels exactly as lnb_nerf_step does."""
    torch = torch_cuda
    from loma_nerf_b200 import api
    case = O.make_nerf_case(77, 16, 192)
    dims = [int(v) for v in case["dims"]]
    tr = api.Trainer(ctx, dims, case["ws"], case["bs"])
    z = lambda *shape: torch.zeros(shape, device="cuda")  # noqa: E731
    tr.step(X=z(0, dims[0]), dists=z(0, 64), target=z(0, 3), R=0, S=64, path="tc")
    w, b, loss = tr.read()
    assert np.isfinite(w).all() and np.isfinite(b).all() and loss == 0.0
    assert np.array_equal(w, case["ws"]) and np.allclose(b, case["bs"], atol=1e-6)   # zero gradient: Adam moves nothing
    tr.step(X=dev(torch, case["X"]), dists=dev(torch, case["dists"]), target=dev(torch, case["target"]), path="tc")
    w, b, loss = tr.read()
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], 16, 192, g=1.0)
    assert rel_err(loss, f["loss"]) <= TC_TOL
    assert np.isfinite(w).all() and np.abs(w - case["ws"]).max() > 0            # the update happened (t = 2)
    tr.close()


@pytest.mark.parametrize("pinned", [True, False])
def test_pipelined_host_steps_equal_the_synchronous_ones(ctx, torch_cuda, pinned):
    """lnb_trainer_submit_host / lnb_trainer_wait (H2D of batch i+1 under step i, two staging slots) must walk the trajectory
    of lnb_trainer_step_host: same losses and weights (to fp32 rounding: the gradient sum order inside a launch is not fixed),
    features and rays batches interleaved."""
    torch = torch_cuda
    from loma_nerf_b200 import api
    R, S, E = 128, 64, 5
    cases = [O.make_nerf_case(1200 + i, R, S) for i in range(7)]
    dims = [int(v) for v in cases[0]["dims"]]
    ws0, bs0 = cases[0]["ws"].copy(), cases[0]["bs"].copy()

    def hostbuf(a, dt=np.float32):
        a = np.ascontiguousarray(a, dt)
        return torch.as_tensor(a).pin_memory() if pinned else a

    batches = []
    for i, c in enumerate(cases):
        if i % 3 == 2:
            batches.append(dict(rays=tuple(hostbuf(c[k], np.float64) for k in ("rays_o", "rays_d", "t")), pe_bands=E,
                                target=hostbuf(c["target"]), path="tc"))
        else:
            batches.append(dict(X=hostbuf(c["X"]), dists=hostbuf(c["dists"]), target=hostbuf(c["target"]), path="tc"))
    ta = api.Trainer(ctx, dims, ws0, bs0)
    want = [ta.step_host(**b) for b in batches]
    wa, ba, _ = ta.read()
    ta.close()
    tb = api.Trainer(ctx, dims, ws0, bs0)
    for b in batches[:3]:
        tb.submit_host(**b)
    got = tb.wait()
    for b in batches[3:]:
        tb.submit_host(tb.prepare(**b))          # a batch marshalled once and handed over as such
    got += tb.wait()
    assert tb.wait() == []
    wb, bb, _ = tb.read()
    tb.close()
    assert len(got) == len(want) and rel_err(got, want) <= 1e-5, (got, want)
    assert rel_err(wb, wa) <= 2e-5 and rel_err(bb, ba) <= 2e-5


@pytest.mark.parametrize("R,S,E", [(500, 64, 2), (257, 40, 8), (64, 64, 10), (300, 16, 0)])
def test_forward_only_kernel_rays_mode_band_counts(ctx, torch_cuda, R, S, E):
    """The forward-only kernel skips the positional-encoding bands that are switched off by warp-uniform branches: every band
    count from none to the maximum must fill exactly the slabs the first-layer MMA reads."""
    torch = torch_cuda
    case = O.make_nerf_case(900 + S + E, R, S, E=E, width=30)
    d64 = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float64)).cuda().contiguous()  # noqa: E731
    out = ctx.nerf_step_rays([int(v) for v in case["dims"]], d64(case["rays_o"]), d64(case["rays_d"]), d64(case["t"]), E,
                             dev(torch, case["ws"]), dev(torch, case["bs"]), None, grad=False, outputs=("color",), path="tc")
    ctx.synchronize()
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=None)
    assert rel_err(host(out["color"]), f["color"]) <= TC_TOL
