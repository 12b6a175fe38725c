"""Operands of the multi-group train kernel (fused_mg_kernel) at the edges of its tensor-memory budget (B200).

Every forward MMA takes its A operand from tensor memory, the layer-0 one included (K0P / 2 columns per group, K padding
written as zeros).  These shapes reach what the shapes of test_gpu_fused.py do not: the widest first layer (63 input
features + ones column, K0P = 64: all 32 A columns of a group live; seven groups and 496 of 512 tensor-memory columns from
rays) and four layers at the 32-column width.  Each runs from features and from rays, against the float64 restatement
within the bf16 bounds of test_gpu_fused.py, and its colours must be bit-equal to the forward-only (render) kernel and to the
one-tile-per-CTA train kernel (LNB_TC_V1=1, A_0 from shared memory) wherever that kernel takes the shape.
"""
import os

import numpy as np
import pytest

from oracle import oracle as O
from test_gpu_fused import nerf_step, rays_step, tc_check

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
    yield c
    c.close()


def one_tile_per_cta(fn):
    os.environ["LNB_TC_V1"] = "1"
    try:
        return fn()
    finally:
        del os.environ["LNB_TC_V1"]


@pytest.mark.parametrize("E,width,layers,v1", [
    (10, 30, 2, True),         # c_in 63, K0P = 64: A_0 fills all 32 operand columns of a group
    (5, 30, 4, False),         # four layers (the one-tile-per-CTA kernel needs <= 128 features in total)
    (4, 30, 4, True),          # four layers, 27 input features: small enough for the one-tile-per-CTA kernel
])
def test_multi_group_operands_against_f64_and_the_one_tile_per_cta_kernel(ctx, torch_cuda, E, width, layers, v1):
    torch = torch_cuda
    R, S = 2100, 64
    case = O.make_nerf_case(6000 + 10 * E + layers, R, S, E=E, width=width, n_layers=layers)
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=1.0)
    o = nerf_step(ctx, torch, case, "tc", expect_kernel="fused_mg_kernel")
    tc_check(o, f)
    orays = rays_step(ctx, torch, case)
    tc_check(orays, f)
    # the forward-only (render) kernel computes the train step's colours to the bit
    assert np.array_equal(nerf_step(ctx, torch, case, "tc", grad=False, outputs=("color",))["color"], o["color"])
    assert np.array_equal(rays_step(ctx, torch, case, grad=False)["color"], orays["color"])
    if v1:
        ref = one_tile_per_cta(lambda: nerf_step(ctx, torch, case, "tc"))
        ref_rays = one_tile_per_cta(lambda: rays_step(ctx, torch, case))
        assert np.array_equal(o["color"], ref["color"])
        assert np.array_equal(orays["color"], ref_rays["color"])
