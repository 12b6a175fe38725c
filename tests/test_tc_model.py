"""The bf16 model of the tensor-core path (oracle/tc_model.py), on the CPU: its bf16 rounding bit for bit against torch's,
its agreement with the float64 restatement when rounding is off, and the power of the GPU bounds of
tests/test_gpu_tc_model.py: for every case there, each of these kernel faults, computed in the model, must move what the
test compares by at least 10x that case's bound --
  (a) one kernel tile's rows left out of dW / db (floor(128 / S) S rows in the fused kernels, 128 in the wide path),
  (b) the last ray of a tail tile left out of dW / db,
  (c) the hidden biases in the other path's precision (bf16 inside the MMA / fp32 in the epilogue),
  (d) the head bias rounded to bf16.
A mutation that changes nothing for a case (no tail tile; biases that are bf16 numbers already) is not applicable there.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as O
from oracle import tc_model as M
from test_gpu_tc_model import ALL_CASES, EXACT_CASES, F64_BOUNDS, UNRESOLVED, assert_exact_forward, bounds_of, errors, make_case, \
    model, over, variant_of


def torch_bf16(x32):
    return torch.from_numpy(np.ascontiguousarray(x32, np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


def test_bf16_rounding_matches_torch_bit_for_bit():
    rng = np.random.default_rng(1)
    vals = [rng.normal(0, 1, 20000), rng.normal(0, 1e30, 2000), rng.uniform(-1e-38, 1e-38, 2000)]     # normals, subnormals
    bits = rng.integers(0, 2 ** 32, 20000, dtype=np.uint64).astype(np.uint32)                         # every bit pattern
    vals.append(bits.view(np.float32))
    # exact ties (lower 16 bits 0x8000) with even and odd bf16 mantissas, one above and below them, the largest finite
    # values, the smallest subnormals, +-0, +-inf, NaN
    base = rng.integers(0, 2 ** 16, 4000, dtype=np.uint64).astype(np.uint32) << 16
    ties = np.concatenate([base | 0x8000, base | 0x7FFF, base | 0x8001]).astype(np.uint32)
    vals.append(ties.view(np.float32))
    special = np.array([0x7F7FFFFF, 0xFF7FFFFF, 0x7F7F8000, 0x00000001, 0x80000001, 0x00008000, 0x00018000, 0x007FFFFF,
                        0x00000000, 0x80000000, 0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00001, 0x7F800001], np.uint32)
    vals.append(special.view(np.float32))
    x = np.concatenate([np.asarray(v, np.float64).astype(np.float32) if v.dtype != np.float32 else v for v in vals])
    got = M.bf16(x).astype(np.float32)
    want = torch_bf16(x)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))
    # float64 input is rounded to float32 first, as the kernels round an fp32 accumulator
    y = rng.normal(0, 1, 1000)
    assert np.array_equal(M.bf16(y), M.bf16(y.astype(np.float32)))


@pytest.mark.parametrize("seed", ["loss", 0.7])
def test_model_without_rounding_is_the_f64_restatement(seed):
    for case in (O.make_nerf_case(11, 40, 33, width=30, n_layers=3), O.make_nerf_case(12, 9, 64, E=10, width=62, n_layers=4)):
        a = (case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], case["R"], case["S"])
        f = O.nerf_f64(*a, g=seed)
        for variant in ("fused", "wide"):
            m = M.nerf_tc_model(*a, g=seed, variant=variant, _exact=True)
            for k in ("loss", "color", "d_ws", "d_bs"):
                assert np.abs(np.asarray(m[k]) - f[k]).max() <= 1e-12 * max(np.abs(f[k]).max(), 1.0), (variant, k)
    fc = O.make_fit_case(13, 300, width=16)
    a = (fc["X"], fc["ws"], fc["bs"], fc["dims"], fc["target"])
    f = O.mlp_fit_f64(*a, g=seed)
    m = M.fit_tc_model(*a, g=seed, _exact=True)
    for k in ("loss", "d_ws", "d_bs"):
        assert np.abs(np.asarray(m[k]) - f[k]).max() <= 1e-12 * max(np.abs(f[k]).max(), 1.0), k


def test_model_rounds_where_the_kernels_do():
    """With rounding on, the model's operands are bf16 numbers and its forward-only values fp32 ones, and the two bias
    variants differ exactly when a hidden bias is not a bf16 number."""
    case = O.make_nerf_case(14, 30, 16, width=20)
    a = (case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], case["R"], case["S"])
    m = M.nerf_tc_model(*a, g=1.0)
    for A in m["A_l"] + m["dz"]:
        assert np.array_equal(M.bf16(A), A)
    assert np.array_equal(M.f32(m["hz"]), m["hz"])
    assert rel_err_max(m["color"], M.nerf_tc_model(*a, g=1.0, variant="wide")["color"]) > 0
    bs = case["bs"].copy()
    bs[:-1] = M.bf16(bs[:-1])
    a2 = a[:2] + (bs,) + a[3:]
    assert np.array_equal(M.nerf_tc_model(*a2, g=1.0)["d_ws"], M.nerf_tc_model(*a2, g=1.0, variant="wide")["d_ws"])


def rel_err_max(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(b).max())


@pytest.mark.parametrize("c", EXACT_CASES, ids=lambda c: c["id"])
def test_exact_cases_meet_their_precondition(c):
    case = make_case(c)
    assert_exact_forward(c, case, model(c, case))


def tile_rows(c):
    if c["path"] == "wide" or c["kind"] == "fit":
        return 128
    return (128 // c["S"]) * c["S"]


def mutations(c, case, m):
    """{name: the model's result under that kernel fault} for the faults that change something in case c."""
    out = {}
    grad = c.get("grad", True)
    N, S, T = case["R"] * case["S"], case["S"], tile_rows(c)
    if grad:
        mid = (N // T // 2) * T                                 # the middle tile
        out["(a) tile left out"] = M.without_rows(m, np.arange(mid, min(mid + T, N)))
        if N % T:
            out["(b) tail tile's last ray left out"] = M.without_rows(m, np.arange(N - S, N))
    L = len(case["dims"]) - 1
    hidden = case["bs"][:L - 1]
    if not np.array_equal(M.bf16(hidden), hidden):
        out["(c) hidden biases in the other precision"] = model(c, case, variant="fused" if variant_of(c) == "wide" else "wide")
    bs = case["bs"].copy()
    bs[L - 1] = M.bf16(bs[L - 1])
    if not np.array_equal(bs, case["bs"]):
        out["(d) head bias in bf16"] = model(c, case, bs=bs)
    return out


@pytest.mark.parametrize("c", ALL_CASES, ids=lambda c: c["id"])
def test_every_kernel_fault_lands_10x_above_the_gpu_bound(c):
    case = make_case(c)
    m = model(c, case)
    muts = mutations(c, case, m)
    assert muts, c["id"]
    f64 = F64_BOUNDS["wide" if variant_of(c) == "wide" else "fused"]
    for name, mm in muts.items():
        errs = errors(mm, m, c.get("grad", True))
        key, r = next(iter(over(errs, bounds_of(c)).items()))
        r64 = over(errs, f64)[key]
        print("%-24s %-42s %-10s %.3g = %6.1f x the bf16-model bound, %.3g x the f64 bound" % (c["id"], name, key, errs[key], r, r64))
        if (c["id"], name[:3]) not in UNRESOLVED:
            assert r >= 10.0, (c["id"], name, errs)
