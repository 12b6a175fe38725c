"""The two fused train-step kernels on shapes the goldens do not cover (B200).

* fused_f32_kernel (LNB_PATH_F32 asked for loss / colour / d_ws / d_bs only): the reference goldens again -- this time through the
  fused kernel, proven by the profiler hook naming it -- then 2- and 3-layer networks of every supported width, tail tiles,
  tiles whose start is not 16-byte aligned (S = 7: 126 rows x 33 floats), the mlp_fit head, forward-only calls.  <= 1e-5.
* fused_mg_kernel (LNB_PATH_TC train steps): hidden widths that pick the 16 / 32 / 64-column forms, 2 / 3 / 4 layers, 1 .. 7
  groups per CTA (LNB_TC_GROUPS), features and rays input, against the float64 restatement within the stated bf16 bounds, and
  against the one-tile-per-CTA kernel (LNB_TC_V1=1), which computes the same products in a different schedule.
"""
import os

import numpy as np
import pytest

from conftest import golden_files, grad_errs, load_golden, rel_err
from oracle import oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-5
TC_TOL, TC_LAYER_TOL, TC_L2_TOL = 3e-2, 6e-2, 3e-2
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


def dev(torch, a, dtype=np.float32):
    return torch.as_tensor(np.ascontiguousarray(a, dtype)).cuda().contiguous()


def host(t):
    return t.detach().cpu().numpy()


def nerf_step(ctx, torch, case, path, seed=1.0, grad=True, outputs=("color", "loss"), expect_kernel=None):
    R, S = int(case["R"]), int(case["S"])
    box = {}

    def call():
        box["out"] = ctx.nerf_step([int(v) for v in case["dims"]], dev(torch, case["X"]), dev(torch, case["ws"]), dev(torch, case["bs"]),
                                   dev(torch, case["dists"]), dev(torch, case["target"]) if grad or "loss" in outputs else None,
                                   R=R, S=S, grad=grad, seed=seed, outputs=outputs, path=path)
    prof = ctx.profile_dominant(call)
    if expect_kernel:
        assert prof is not None and prof["kernel"].startswith(expect_kernel), prof
    return {k: host(v) for k, v in box["out"].items()}


def rays_step(ctx, torch, case, grad=True):
    out = ctx.nerf_step_rays([int(v) for v in case["dims"]], dev(torch, case["rays_o"], np.float64), dev(torch, case["rays_d"], np.float64),
                             dev(torch, case["t"], np.float64), int(case["E"]), dev(torch, case["ws"]), dev(torch, case["bs"]),
                             dev(torch, case["target"]) if grad else None, grad=grad, seed=1.0,
                             outputs=("color", "loss") if grad else ("color",), path="tc")
    ctx.synchronize()
    return {k: host(v) for k, v in out.items()}


# ------------------------------------------------------------------------------------------------
# fused exact kernel
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", ["loss", 1.0])
@pytest.mark.parametrize("gpath", NERF_GOLDEN, ids=os.path.basename)
def test_fused_f32_nerf_against_reference_golden(ctx, torch_cuda, gpath, seed):
    gd = load_golden(gpath)
    sfx = "" if seed == "loss" else "_g1"
    o = nerf_step(ctx, torch_cuda, gd, "f32", seed=seed, expect_kernel="fused_f32_kernel")
    assert rel_err(o["loss"][0], gd["loss"]) <= TOL and rel_err(o["color"], gd["color"]) <= TOL
    for k in ("d_ws", "d_bs"):
        assert rel_err(o[k], gd[k + sfx]) <= TOL, k


@pytest.mark.parametrize("gpath", FIT_GOLDEN, ids=os.path.basename)
def test_fused_f32_fit_against_reference_golden(ctx, torch_cuda, gpath):
    torch = torch_cuda
    gd = load_golden(gpath)
    box = {}

    def call():
        box["o"] = ctx.fit_step([int(v) for v in gd["dims"]], dev(torch, gd["X"]), dev(torch, gd["ws"]), dev(torch, gd["bs"]), dev(torch, gd["target"]),
                                grad=True, seed="loss", outputs=("loss",), path="f32")
    prof = ctx.profile_dominant(call)
    assert prof and prof["kernel"] == "fused_f32_kernel", prof
    o = {k: host(v) for k, v in box["o"].items()}
    assert rel_err(o["loss"][0], gd["loss"]) <= TOL
    assert rel_err(o["d_ws"], gd["d_ws"]) <= TOL and rel_err(o["d_bs"], gd["d_bs"]) <= TOL


@pytest.mark.parametrize("R,S,E,width,layers", [
    (4096, 64, 5, 30, 3),      # BASELINE config 2
    (1000, 30, 5, 30, 3),      # 120-row tiles, a tail tile
    (700, 7, 5, 30, 3),        # 126-row tiles: tile starts are not 16-byte aligned (scalar feature loads)
    (257, 128, 4, 31, 3),      # one ray per tile, the widest hidden layer
    (333, 2, 5, 9, 3),         # 64 rays per tile, narrow layers
    (500, 64, 5, 30, 2),       # two layers
    (90, 100, 3, 16, 2),
    (64, 33, 0, 5, 3),         # no encoding bands: 3 input features
])
def test_fused_f32_shapes_against_f64_restatement(ctx, torch_cuda, R, S, E, width, layers):
    case = O.make_nerf_case(4000 + R + S, R, S, E=E, width=width, n_layers=layers)
    o = nerf_step(ctx, torch_cuda, case, "f32", expect_kernel="fused_f32_kernel")
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=1.0)
    assert rel_err(o["loss"][0], f["loss"]) <= TOL and rel_err(o["color"], f["color"]) <= TOL
    assert rel_err(o["d_ws"], f["d_ws"]) <= TOL and rel_err(o["d_bs"], f["d_bs"]) <= TOL
    # bit-reproducible: static tile assignment, fixed-order sums
    o2 = nerf_step(ctx, torch_cuda, case, "f32")
    assert all(np.array_equal(o[k], o2[k]) for k in o)
    # and the layerwise kernels agree with it far inside the tolerance
    ol = nerf_step(ctx, torch_cuda, case, "f32_layerwise")
    assert rel_err(o["d_ws"], ol["d_ws"]) <= 2e-6 and rel_err(o["color"], ol["color"]) <= 2e-6


def test_fused_f32_forward_only_fit_shapes_and_fallback(ctx, torch_cuda):
    torch = torch_cuda
    case = O.make_nerf_case(4100, 300, 64)
    o = nerf_step(ctx, torch, case, "f32", grad=False, outputs=("color",), expect_kernel="fused_f32_kernel")
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], 300, 64)
    assert rel_err(o["color"], f["color"]) <= TOL
    for N, E, width, layers in [(65536, 5, 16, 3), (1000, 8, 31, 2), (129, 1, 4, 3)]:
        fc = O.make_fit_case(4200 + N, N, E=E, width=width, n_layers=layers)
        out = ctx.fit_step([int(v) for v in fc["dims"]], dev(torch, fc["X"]), dev(torch, fc["ws"]), dev(torch, fc["bs"]), dev(torch, fc["target"]),
                           grad=True, seed=1.0, outputs=("loss",), path="f32")
        ctx.synchronize()
        ff = O.mlp_fit_f64(fc["X"], fc["ws"], fc["bs"], fc["dims"], fc["target"], g=1.0)
        assert rel_err(host(out["loss"])[0], ff["loss"]) <= TOL
        assert rel_err(host(out["d_ws"]), ff["d_ws"]) <= TOL and rel_err(host(out["d_bs"]), ff["d_bs"]) <= TOL
    # what the fused kernel does not produce (per-sample by-products, wide or deep networks) runs on the layerwise kernels:
    # same path, same tolerance, never an error
    wide = O.make_nerf_case(4300, 40, 64, width=64, n_layers=4)
    ow = nerf_step(ctx, torch, wide, "f32")
    fw = O.nerf_f64(wide["X"], wide["ws"], wide["bs"], wide["dims"], wide["target"], wide["dists"], 40, 64, g=1.0)
    assert rel_err(ow["d_ws"], fw["d_ws"]) <= TOL
    od = nerf_step(ctx, torch, case, "f32", outputs=("color", "loss", "d_dists"))
    fd = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], 300, 64, g=1.0)
    assert rel_err(od["d_dists"], fd["d_dists"]) <= TOL and rel_err(od["d_ws"], fd["d_ws"]) <= TOL


# ------------------------------------------------------------------------------------------------
# multi-group tensor-core kernel
# ------------------------------------------------------------------------------------------------
def tc_check(o, f):
    errs = dict(loss=rel_err(o["loss"][0], f["loss"]), color=rel_err(o["color"], f["color"]), **grad_errs(o, f))
    assert max(errs["loss"], errs["color"]) <= TC_TOL, errs
    assert max(errs["d_ws"], errs["d_bs"]) <= TC_TOL, errs
    assert max(errs["d_ws_layer"], errs["d_bs_layer"]) <= TC_LAYER_TOL, errs
    assert max(errs["d_ws_l2"], errs["d_bs_l2"]) <= TC_L2_TOL, errs


@pytest.mark.parametrize("R,S,E,width,layers", [
    (2048, 64, 5, 30, 3),      # 7 groups per CTA
    (2000, 30, 5, 15, 3),      # 16-column form
    (1500, 64, 5, 8, 2),       # two layers
    (900, 64, 5, 48, 3),       # 64-column form (four groups)
    (600, 100, 3, 62, 2),
    (1200, 40, 2, 20, 4),      # four layers
    (300, 128, 8, 31, 3),      # 51 input features + ones column: K padded to 64
])
def test_multi_group_kernel_shapes_against_f64_restatement(ctx, torch_cuda, R, S, E, width, layers):
    torch = torch_cuda
    case = O.make_nerf_case(5000 + R + width, R, S, E=E, width=width, n_layers=layers)
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=1.0)
    o = nerf_step(ctx, torch, case, "tc", expect_kernel="fused_mg_kernel")
    tc_check(o, f)
    # rays input: features generated in the kernel
    out = ctx.nerf_step_rays([int(v) for v in case["dims"]], dev(torch, case["rays_o"], np.float64), dev(torch, case["rays_d"], np.float64),
                             dev(torch, case["t"], np.float64), E, dev(torch, case["ws"]), dev(torch, case["bs"]), dev(torch, case["target"]),
                             grad=True, seed=1.0, outputs=("color", "loss"), path="tc")
    ctx.synchronize()
    tc_check({k: host(v) for k, v in out.items()}, f)


def test_multi_group_kernel_agrees_with_the_one_tile_per_cta_kernel(ctx, torch_cuda):
    """Same bf16 products, different schedule (groups per CTA, in-place adjoints, per-layer M = 64 gradient MMAs): the two
    kernels must agree to fp32 summation order, for every group count."""
    torch = torch_cuda
    case = O.make_nerf_case(5100, 3000, 64)
    os.environ["LNB_TC_V1"] = "1"
    try:
        ref = nerf_step(ctx, torch, case, "tc")
    finally:
        del os.environ["LNB_TC_V1"]
    for ng in (1, 2, 3, 5, 7):
        os.environ["LNB_TC_GROUPS"] = str(ng)
        try:
            o = nerf_step(ctx, torch, case, "tc")
        finally:
            del os.environ["LNB_TC_GROUPS"]
        assert np.array_equal(o["color"], ref["color"]), ng
        assert rel_err(o["loss"][0], ref["loss"][0]) <= 1e-6
        assert rel_err(o["d_ws"], ref["d_ws"]) <= 1e-5 and rel_err(o["d_bs"], ref["d_bs"]) <= 1e-5, ng
    # the forward-only (render) kernel computes the train step's colours to the bit, from features and from rays
    fwd = nerf_step(ctx, torch, case, "tc", grad=False, outputs=("color",), expect_kernel="fused_v1_kernel")
    assert np.array_equal(fwd["color"], ref["color"])
    assert np.array_equal(rays_step(ctx, torch, case, grad=False)["color"], rays_step(ctx, torch, case)["color"])
