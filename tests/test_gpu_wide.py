"""Wide-MLP tensor-core path (wide_tc.cu): the TMA-fed tcgen05 chain kernel run as a one-layer GEMM, and the
weight-gradient kernel with the step's reduction, against fp32 matrix products of the same bf16-rounded operands
(torch is only the checker here), then the whole layerwise step against the reference golden vectors of the 8x256
net."""
import ctypes

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module")
def ctx(torch_cuda):
    from loma_nerf_b200 import api
    c = api.Context(0)
    c.set_stream(torch_cuda.cuda.current_stream())
    yield c
    c.close()


@pytest.mark.parametrize("M,N,K", [(128, 16, 64), (1000, 64, 64), (4096 + 77, 256, 256), (300, 32, 128), (20000, 256, 64)])
def test_wide_gemm_matches_fp32_product_of_bf16_operands(ctx, torch_cuda, M, N, K):
    torch = torch_cuda
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16).contiguous()
    B = torch.randn(N, K, device="cuda", generator=g).to(torch.bfloat16).contiguous()
    bias = torch.randn(N, device="cuda", generator=g)
    C = torch.full((M, N), float("nan"), device="cuda")
    lib = ctx.lib
    lib.lnb_test_wide_gemm.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_longlong, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    ctx._check(lib.lnb_test_wide_gemm(ctx.h, A.data_ptr(), B.data_ptr(), M, N, K, bias.data_ptr(), C.data_ptr()))
    ctx.synchronize()
    ref = A.float() @ B.float().t() + bias
    assert rel_err(C.cpu().numpy(), ref.cpu().numpy()) <= 2e-5


def _pack_bits(torch, positive):
    """[M][N] bool -> [M][N/32] int32 in the kernel's ReLU-pattern layout (wide_tc.cu ChainLayer): word w
    covers columns 32w..32w+31, column 32w + 8g + 2j + p at bit 16p + 4g + j."""
    pos = positive.cpu().numpy().astype(np.uint64)
    M, N = pos.shape
    c = np.arange(32)
    shift = (16 * (c % 2) + 4 * (c // 8) + (c % 8) // 2).astype(np.uint64)
    words = (pos.reshape(M, N // 32, 32) << shift).sum(axis=2).astype(np.uint32)
    return torch.as_tensor(np.ascontiguousarray(words).view(np.int32)).cuda()


@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (1000, 256, 256), (4096 + 77, 128, 64), (50000, 256, 256), (777, 192, 128)])
@pytest.mark.parametrize("masked", [False, True])
def test_wide_gemm_bf16_epilogues(ctx, torch_cuda, M, N, K, masked):
    torch = torch_cuda
    g = torch.Generator(device="cuda").manual_seed(M + N + K + int(masked))
    A = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16).contiguous()
    B = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).to(torch.bfloat16).contiguous()
    bias = torch.randn(N, device="cuda", generator=g)
    positive = torch.randn(M, N, device="cuda", generator=g) > 0
    bits_in = _pack_bits(torch, positive)
    bits_out = torch.full((M, N // 32), -1, dtype=torch.int32, device="cuda")
    C = torch.full((M, N), float("nan"), device="cuda").to(torch.bfloat16)
    lib = ctx.lib
    lib.lnb_test_wide_gemm_bf16.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_longlong, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 4
    ctx._check(lib.lnb_test_wide_gemm_bf16(ctx.h, A.data_ptr(), B.data_ptr(), M, N, K, None if masked else bias.data_ptr(),
                                           bits_in.data_ptr() if masked else None, None if masked else bits_out.data_ptr(), C.data_ptr()))
    ctx.synchronize()
    acc = A.float() @ B.float().t()
    ref = torch.where(positive, acc, torch.zeros_like(acc)) if masked else torch.relu(acc + bias)
    got = C.float().cpu().numpy()
    assert np.isfinite(got).all()
    assert rel_err(got, ref.to(torch.bfloat16).float().cpu().numpy()) <= 1e-2    # one bf16 rounding of the output
    if masked:
        assert (got[~positive.cpu().numpy()] == 0).all()
    else:   # the recorded pattern is exactly the sign pattern of what was stored
        assert (bits_out.cpu().numpy() == _pack_bits(torch, C.float() > 0).cpu().numpy()).all()


@pytest.mark.parametrize("rows,in_pad,out_pad", [(64, 64, 64), (1000, 256, 256), (100000, 64, 256), (33333, 256, 64), (5000, 128, 192)])
def test_wide_dw_matches_fp32_product(ctx, torch_cuda, rows, in_pad, out_pad):
    torch = torch_cuda
    g = torch.Generator(device="cuda").manual_seed(rows + in_pad)
    H = torch.relu(torch.randn(rows, in_pad, device="cuda", generator=g)).to(torch.bfloat16).contiguous()
    Z = (torch.randn(rows, out_pad, device="cuda", generator=g) * 0.1).to(torch.bfloat16).contiguous()
    dW = torch.full((in_pad, out_pad), float("nan"), device="cuda")
    db = torch.full((out_pad,), float("nan"), device="cuda")
    lib = ctx.lib
    lib.lnb_test_wide_dw.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong,
                                     ctypes.c_void_p, ctypes.c_void_p]
    ctx._check(lib.lnb_test_wide_dw(ctx.h, H.data_ptr(), in_pad, Z.data_ptr(), out_pad, rows, dW.data_ptr(), db.data_ptr()))
    ctx.synchronize()
    ref = (H.double().t() @ Z.double()).float()
    assert rel_err(dW.cpu().numpy(), ref.cpu().numpy()) <= 2e-5
    assert rel_err(db.cpu().numpy(), Z.double().sum(0).float().cpu().numpy()) <= 2e-5


from conftest import golden_files, load_golden  # noqa: E402
from oracle import oracle as O  # noqa: E402

WIDE_TOL = 6e-2   # bf16 operands through up to 9 layers of 256; measured errors are logged
WIDE_LAYER_TOL = 1e-1   # per layer: max|a_l - b_l| / max|b_l|
WIDE_L2_TOL = 5e-2      # ||a - b||_2 / ||b||_2


def _log(msg):
    import os
    os.makedirs("gpurun_out", exist_ok=True)
    with open("gpurun_out/tc_errors.log", "a") as fh:
        fh.write(msg + "\n")


def _run_wide(ctx, torch, case, seed, rays=False):
    cv = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    dims = [int(v) for v in case["dims"]]
    R, S = int(case["R"]), int(case["S"])
    if rays:
        r = [torch.as_tensor(np.ascontiguousarray(case[k], np.float64)).cuda() for k in ("rays_o", "rays_d", "t")]
        out = ctx.nerf_step_rays(dims, r[0], r[1], r[2], int(case["E"]), cv(case["ws"]), cv(case["bs"]), cv(case["target"]),
                                 grad=True, seed=seed, outputs=("color", "loss"), path="tc")
    else:
        out = ctx.nerf_step(dims, cv(case["X"]), cv(case["ws"]), cv(case["bs"]), cv(case["dists"]), cv(case["target"]), R=R, S=S,
                            grad=True, seed=seed, outputs=("color", "loss"), path="tc")
    ctx.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}


def test_wide_path_paper_size_mlp_against_reference_golden(ctx, torch_cuda):
    """BASELINE config 5 shape: 63 -> 8 x 256 -> 4, 192 samples per ray, golden vector recorded from the
    real reference (max_iter-only edit of scripts/nerf.py)."""
    gd = load_golden([p for p in golden_files("nerf_") if "c5" in p][0])
    o = _run_wide(ctx, torch_cuda, gd, "loss")
    errs = dict(loss=rel_err(o["loss"][0], gd["loss"]), color=rel_err(o["color"], gd["color"]),
                d_ws=rel_err(o["d_ws"], gd["d_ws"]), d_bs=rel_err(o["d_bs"], gd["d_bs"]))
    _log("wide c5 golden %s" % errs)
    # a single ray: the gradient is proportional to the residual colour - target (0.05-0.1 here), so
    # the 1 % bf16 error of the colour itself shows up ten times larger in d_ws / d_bs; batches of
    # rays average it out (next test, same network: 2e-3)
    assert errs["loss"] <= 1e-2 and errs["color"] <= 3e-2 and max(errs["d_ws"], errs["d_bs"]) <= 0.2, errs


def test_wide_path_paper_size_mlp_against_eight_ray_reference_golden(ctx, torch_cuda):
    """The same network on EIGHT rays of the real reference (unit seed; tests/golden/make_golden_c5_r8.py): with
    more than one ray the residuals no longer cancel to a tenth of the colour, and the bounds are the batch ones --
    norm-wise, per layer and in L2."""
    import os
    from conftest import GOLDEN_DIR, grad_errs
    gd = load_golden(os.path.join(GOLDEN_DIR, "wide_c5_r8_s192.npz"))
    o = _run_wide(ctx, torch_cuda, gd, 1.0)
    errs = dict(loss=rel_err(o["loss"][0], gd["loss"]), color=rel_err(o["color"], gd["color"]), **grad_errs(o, gd, "_g1"))
    _log("wide c5 8-ray golden %s" % errs)
    assert errs["loss"] <= 1e-2 and errs["color"] <= 2e-2, errs
    assert max(errs["d_ws"], errs["d_bs"]) <= WIDE_TOL, errs
    assert max(errs["d_ws_layer"], errs["d_bs_layer"]) <= WIDE_LAYER_TOL, errs
    assert max(errs["d_ws_l2"], errs["d_bs_l2"]) <= WIDE_L2_TOL, errs
    # and the exact path on the same vectors
    cv = lambda a: torch_cuda.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    out = ctx.nerf_step([int(v) for v in gd["dims"]], cv(gd["X"]), cv(gd["ws"]), cv(gd["bs"]), cv(gd["dists"]), cv(gd["target"]),
                        R=8, S=192, grad=True, seed=1.0, outputs=("color", "loss"), path="f32")
    ctx.synchronize()
    ex = {k: v.cpu().numpy() for k, v in out.items()}
    assert rel_err(ex["loss"][0], gd["loss"]) <= 1e-5 and rel_err(ex["color"], gd["color"]) <= 1e-5
    assert rel_err(ex["d_ws"], gd["d_ws_g1"]) <= 1e-5 and rel_err(ex["d_bs"], gd["d_bs_g1"]) <= 1e-5


@pytest.mark.parametrize("R,S,E,width,layers,rays", [(64, 192, 10, 256, 9, False), (300, 64, 10, 256, 5, True), (1000, 33, 5, 128, 4, False),
                                                      (50, 128, 4, 200, 3, True), (2048, 64, 10, 64, 6, False)])
def test_wide_path_against_f64_restatement(ctx, torch_cuda, R, S, E, width, layers, rays):
    case = O.make_nerf_case(1300 + width + layers, R, S, E=E, width=width, n_layers=layers)
    o = _run_wide(ctx, torch_cuda, case, 1.0, rays=rays)
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=1.0)
    from conftest import grad_errs
    errs = dict(loss=rel_err(o["loss"][0], f["loss"]), color=rel_err(o["color"], f["color"]), **grad_errs(o, f))
    _log("wide R=%d S=%d E=%d w=%d L=%d rays=%s %s" % (R, S, E, width, layers, rays, errs))
    assert max(errs["loss"], errs["color"], errs["d_ws"], errs["d_bs"]) <= WIDE_TOL, errs
    assert max(errs["d_ws_layer"], errs["d_bs_layer"]) <= WIDE_LAYER_TOL, errs
    assert max(errs["d_ws_l2"], errs["d_bs_l2"]) <= WIDE_L2_TOL, errs


def test_trainer_on_a_wide_mlp_follows_numpy_adam(ctx, torch_cuda):
    """lnb_trainer with a network the fused kernel cannot take (5 layers of 128): the generic step runs
    the layerwise tensor-core kernels, then Adam (train_nerf.py:133-161); compared with the float64
    gradients + numpy Adam over 3 steps, features in and rays in."""
    torch = torch_cuda
    from loma_nerf_b200 import api
    R, S, E = 96, 40, 6
    cases = [O.make_nerf_case(2100 + i, R, S, E=E, width=128, n_layers=5) for i in range(3)]
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
    cv = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    for mode in ("features", "rays"):
        tr = api.Trainer(ctx, dims, ws0, bs0, optimizer="adam", lr=lr, beta1=b1, beta2=b2, eps=eps)
        got = []
        for i, c in enumerate(cases):
            if mode == "features":
                batch = dict(X=cv(c["X"]), dists=cv(c["dists"]), target=cv(c["target"]), path="tc")
            else:
                rays = tuple(torch.as_tensor(np.ascontiguousarray(c[k])).cuda() for k in ("rays_o", "rays_d", "t"))
                batch = dict(rays=rays, pe_bands=E, target=cv(c["target"]), path="tc")
            if i == 1:
                tr.grad(**batch); tr.apply()
            else:
                tr.step(**batch)
            got.append(tr.read()[2])
        w, b, _ = tr.read()
        tr.close()
        du, dr = (w - ws0).ravel().astype(np.float64), (ws - ws0).ravel()
        upd_l2 = float(np.linalg.norm(du - dr) / np.linalg.norm(dr))
        _log("wide trainer %s: loss err %.3g, update l2 err %.3g" % (mode, rel_err(got, losses), upd_l2))
        assert rel_err(got, losses) <= WIDE_TOL
        assert upd_l2 <= 0.2   # Adam turns every entry into ~lr*sign(g): entries below the bf16 noise flip freely


def test_chain_kernel_equals_one_launch_per_layer():
    """chain_tc_kernel with all layers of a pass in one launch (activations handed over through L2) runs the very
    same MMAs and epilogues as one one-layer launch per layer (LNB_WIDE_NO_CHAIN=1, no hand-over inside the
    kernel), and as blocks of 3 or of single tiles (LNB_WIDE_CHAIN_G): loss and colour of a 345 600-sample step
    must agree to the last printed digit, run after run (a lost hand-over would show up here); the gradient
    checksums are compared to 1e-5.  The switches are environment variables read once per process, hence the
    subprocesses."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def run(env_extra):
        env = dict(os.environ, **env_extra)
        out = subprocess.run([sys.executable, os.path.join(root, "tools", "t_chain.py"), "1800"], cwd=root, env=env, capture_output=True,
                             text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-2000:]
        lines = [ln for ln in out.stdout.splitlines() if ln.startswith("loss ")]
        assert len(lines) == 3 and len(set(lines)) == 1, lines      # three repetitions, identical
        tok = lines[0].split()
        return tok[1], tok[3], np.array([float(tok[5]), float(tok[7]), float(tok[9])])

    a, b, c = run({}), run({"LNB_WIDE_NO_CHAIN": "1"}), run({"LNB_WIDE_CHAIN_G": "3"})
    d = run({"LNB_WIDE_CHAIN_G": "1"})                                # single-tile blocks
    assert a[0] == b[0] == c[0] == d[0] and a[1] == b[1] == c[1] == d[1], (a, b, c, d)
    assert np.allclose(a[2], b[2], rtol=1e-5) and np.allclose(a[2], c[2], rtol=1e-5) and np.allclose(a[2], d[2], rtol=1e-5), (a, b, c, d)


@pytest.mark.parametrize("N,width,layers", [(5000, 128, 5), (20000, 256, 9), (300, 70, 3)])
def test_wide_path_mlp_fit_against_f64_restatement(ctx, torch_cuda, N, width, layers):
    """mlp_fit (scripts/mlp_fit.py:39-147: sigmoid head, SSE over the 3 colour channels) with a network too wide for
    the fused kernel: the layerwise tensor-core kernels with the fit head, against the float64 restatement."""
    torch = torch_cuda
    case = O.make_fit_case(3100 + width, N, E=5, width=width, n_layers=layers)
    cv = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    dims = [int(v) for v in case["dims"]]
    out = ctx.fit_step(dims, cv(case["X"]), cv(case["ws"]), cv(case["bs"]), cv(case["target"]), grad=True, seed=1.0, outputs=("loss",), path="tc")
    ctx.synchronize()
    f = O.mlp_fit_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], g=1.0)
    errs = dict(loss=rel_err(out["loss"].cpu().numpy()[0], f["loss"]), d_ws=rel_err(out["d_ws"].cpu().numpy(), f["d_ws"]),
                d_bs=rel_err(out["d_bs"].cpu().numpy(), f["d_bs"]))
    _log("wide fit N=%d w=%d L=%d %s" % (N, width, layers, errs))
    assert max(errs.values()) <= WIDE_TOL, errs


@pytest.mark.parametrize("R,S,width,layers", [(96, 64, 256, 5), (77, 33, 200, 4), (50, 20, 130, 3), (3, 100, 128, 6)])
def test_exact_path_on_wide_layers_against_f64_restatement(ctx, torch_cuda, R, S, width, layers):
    """The fp32 CUDA-core path on wide layers takes the register-blocked 128 x 128 kernels (sgemm128_kernel,
    dw128_kernel in kernels_f32.cu) where shapes allow and the generic ones elsewhere; both within 1e-5."""
    torch = torch_cuda
    case = O.make_nerf_case(4100 + width, R, S, E=10, width=width, n_layers=layers)
    cv = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    dims = [int(v) for v in case["dims"]]
    out = ctx.nerf_step(dims, cv(case["X"]), cv(case["ws"]), cv(case["bs"]), cv(case["dists"]), cv(case["target"]), R=R, S=S, grad=True, seed="loss",
                        outputs=("color", "loss", "d_X", "d_dists"), path="f32")
    ctx.synchronize()
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g="loss")
    errs = {k: rel_err(out[k].cpu().numpy().reshape(np.asarray(f[k]).shape), f[k]) for k in ("color", "d_ws", "d_bs", "d_X", "d_dists")}
    errs["loss"] = rel_err(out["loss"].cpu().numpy()[0], f["loss"])
    _log("exact wide R=%d S=%d w=%d L=%d %s" % (R, S, width, layers, errs))
    assert max(errs.values()) <= 1e-5, errs


def test_wide_path_random_shapes(ctx, torch_cuda):
    """Sixteen random (bands, width, depth, rays, samples, input mode, forward-only or train) draws, fixed seed: odd
    widths (padding to 64), ragged last tiles, a single sample per ray, up to 11 layers -- each within the wide bound."""
    torch = torch_cuda
    rng = np.random.default_rng(20261018)
    cv = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    worst = 0.0
    for it in range(16):
        E = int(rng.integers(1, 11)); width = int(rng.integers(63, 257)); layers = int(rng.integers(2, 12))
        R = int(rng.integers(1, 400)); S = int(rng.integers(1, 200)); rays = bool(rng.integers(0, 2)); grad = bool(rng.integers(0, 4))
        case = O.make_nerf_case(6000 + it, R, S, E=E, width=width, n_layers=layers)
        dims = [int(v) for v in case["dims"]]
        if rays:
            r = [torch.as_tensor(np.ascontiguousarray(case[k], np.float64)).cuda() for k in ("rays_o", "rays_d", "t")]
            out = ctx.nerf_step_rays(dims, r[0], r[1], r[2], E, cv(case["ws"]), cv(case["bs"]), cv(case["target"]), grad=grad, seed=1.0,
                                     outputs=("color", "loss"), path="tc")
        else:
            out = ctx.nerf_step(dims, cv(case["X"]), cv(case["ws"]), cv(case["bs"]), cv(case["dists"]), cv(case["target"]), R=R, S=S, grad=grad,
                                seed=1.0, outputs=("color", "loss"), path="tc")
        ctx.synchronize()
        f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=1.0)
        errs = dict(loss=rel_err(out["loss"].cpu().numpy()[0], f["loss"]), color=rel_err(out["color"].cpu().numpy(), f["color"]))
        if grad:
            errs.update(d_ws=rel_err(out["d_ws"].cpu().numpy(), f["d_ws"]), d_bs=rel_err(out["d_bs"].cpu().numpy(), f["d_bs"]))
        shape = dict(E=E, width=width, layers=layers, R=R, S=S, rays=rays, grad=grad)
        _log("wide random %s %s" % (shape, errs))
        # a draw with one or two rays carries the single-ray amplification of the golden-vector test above
        bound = WIDE_TOL if R >= 8 else 0.2
        assert all(np.isfinite(v) for v in errs.values()) and max(errs.values()) <= bound, (shape, errs)
        worst = max(worst, max(errs.values()))
    _log("wide random worst %.3g" % worst)


@pytest.mark.parametrize("R,S,width,layers", [(96, 64, 128, 4), (40, 192, 256, 9)])
def test_wide_path_compositing_by_products_and_ray_adjoints(ctx, torch_cuda, R, S, width, layers):
    """rgba / alpha / cumprod / weights and d_dists / d_accumulated_color / d_target on the layerwise tensor-core path (they
    come from the fp32 compositing kernels fed with the tensor-core head), seed = loss, += into the caller's buffers."""
    torch = torch_cuda
    case = O.make_nerf_case(3300 + width, R, S, E=10, width=width, n_layers=layers)
    cv = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    outs = ("color", "loss", "rgba", "alpha", "cumprod", "weights", "d_dists", "d_color", "d_target")
    pre = {k: torch.full(shape, 0.5, device="cuda") for k, shape in (("d_dists", (R, S)), ("d_color", (R, 3)), ("d_target", (R, 3)))}
    out = ctx.nerf_step([int(v) for v in case["dims"]], cv(case["X"]), cv(case["ws"]), cv(case["bs"]), cv(case["dists"]), cv(case["target"]),
                        R=R, S=S, grad=True, seed="loss", outputs=outs, out=dict(pre), path="tc")
    ctx.synchronize()
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g="loss")
    o = {k: v.cpu().numpy() for k, v in out.items()}
    for k in ("rgba", "alpha", "cumprod", "weights", "color"):
        assert rel_err(o[k].reshape(np.asarray(f[k]).shape), f[k]) <= WIDE_TOL, k
    for k, fk in (("d_dists", "d_dists"), ("d_color", "d_acc"), ("d_target", "d_target")):
        got = o[k] - 0.5                                            # accumulated onto the 0.5 already there
        assert rel_err(got.reshape(np.asarray(f[fk]).shape), f[fk]) <= 2 * WIDE_TOL, k
    assert rel_err(o["d_ws"], f["d_ws"]) <= 2 * WIDE_TOL            # seed = loss carries the loss's own error too
