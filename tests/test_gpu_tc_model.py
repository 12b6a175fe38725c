"""The tensor-core path against its own stated arithmetic (oracle/tc_model.py: float64, rounded to bf16 where the kernels
round), on a B200.

The f64 tests (test_gpu_tc.py, test_gpu_fused.py, test_gpu_mg_operands.py, test_gpu_wide.py) check the semantics: they
must leave room for the whole bf16 error, 3e-2 .. 1e-1.  A lost or doubled tile, a bias in the wrong precision or a stale
weight-image entry moves the result by 1e-3 .. 1e-2, well inside that room.  Against the bf16 model the kernels differ
only by their fp32 summation order and fast transcendentals, so the bounds here are 100x tighter, and
tests/test_tc_model.py proves on the CPU that every one of those mutations lands at least 10x above them.

* Exact-arithmetic cases: dyadic operands (X on a 2^-4 grid, weights k/16 or k/32, biases on coarse grids) for which
  every fp32 sum of the forward pass is exact in any order (asserted per layer): the hidden activations and the head's
  pre-activations are then bit-identical to the model, and only the head, compositing and the backward's roundings
  differ.  They cover the train kernel's widths, input widths, depths, tile shapes, group counts, the one-tile-per-CTA
  and forward-only kernels, the sigmoid head and the wide path, and pin each path's bias precision.
* Realistic cases: the shapes of the f64 tests, from features and (E <= 2) from rays.
* The trainer: Adam through step() (fused reduce + Adam) and grad() + apply(), SGD with the sigmoid head, a batch the
  fused kernel cannot take; every update against an fp32 emulation of adam_one fed with the kernel's own gradients, and
  the refreshed bf16 weight image against one built afresh.
"""
import os

import numpy as np
import pytest

from conftest import grad_errs, rel_err
from test_gpu_tc import log   # the measured-error log the f64 tests write too
from oracle import oracle as O
from oracle import tc_model as M

pytestmark = pytest.mark.gpu

# Bounds against the bf16 model, by family: "out" = loss and colour (norm-wise), "grad" = d_ws / d_bs norm-wise and per
# layer, "l2" = d_ws / d_bs in L2.  Set at about 3x the largest error of the family measured on one B200 (1000 W), written
# to the error log by every run.
BOUNDS = {
    "exact": dict(out=1e-6, grad=3e-4, l2=3e-5),
    "fused": dict(out=4e-4, grad=6e-5, l2=5e-5),
    "wide": dict(out=1.5e-3, grad=7e-5, l2=2e-5),
    # 5 - 9 layers of 256: a flipped bf16 rounding of one activation travels through every later layer
    "wide-deep": dict(out=4e-4, grad=2.5e-3, l2=7e-4),
}
# The f64 bounds the same cases are held to in the f64 tests (logged next to the mutation signals).
F64_BOUNDS = {"fused": dict(out=3e-2, grad=6e-2, l2=3e-2), "wide": dict(out=6e-2, grad=1e-1, l2=5e-2)}
# Faults the bounds cannot resolve at that depth, by (case, mutation): tests/test_tc_model.py logs them and does not hold
# them to the 10x margin.
UNRESOLVED = {
    ("wide-9x256", "(d)"): "the head bias in bf16 moves d_ws by 3.0e-4 in L2, 0.4x the bound",
    ("wide-5x256", "(d)"): "the head bias in bf16 moves d_bs by 8.5e-4 in L2, 2.1x the bound",
    ("wide-fit-9x256", "(d)"): "the head bias in bf16 moves d_ws by 1.3e-3 in L2, 1.9x the bound",
    ("wide-fit-9x256", "(a)"): "a lost tile moves d_ws by 6.1e-3 in L2, 8.8x the bound",
    ("wide-fit-9x256", "(c)"): "the other bias precision moves d_bs by 6.5e-3 in L2, 9.3x the bound",
    ("wide-5x256", "(c)"): "the other bias precision moves d_ws by 3.7e-3 in L2, 9.2x the bound",
    ("wide-9x256", "(c)"): "the other bias precision moves d_bs by 6.8e-3 in L2, 9.7x the bound",
}


# ------------------------------------------------------------------------------------------------
# cases
# ------------------------------------------------------------------------------------------------
def _c(id, kind, path, R, S, c_in, width, layers, family, **kw):
    return dict(id=id, kind=kind, path=path, R=R, S=S, c_in=c_in, width=width, layers=layers, family=family, **kw)


EXACT_CASES = [
    _c("mg-hp16-L2", "nerf", "mg", 500, 64, 12, 15, 2, "exact"),
    _c("mg-hp32-L4-S33-tail", "nerf", "mg", 100, 33, 27, 30, 4, "exact", seed="loss"),
    _c("mg-hp64-L3-k0p64-S100", "nerf", "mg", 300, 100, 63, 62, 3, "exact"),
    _c("mg-hp32-L3-S7", "nerf", "mg", 700, 7, 33, 30, 3, "exact"),
    _c("mg-hp32-L3-S128", "nerf", "mg", 150, 128, 33, 30, 3, "exact"),
    _c("mg-few-tiles", "nerf", "mg", 5, 64, 33, 30, 3, "exact"),
    _c("mg-groups1", "nerf", "mg", 2100, 64, 33, 30, 3, "exact", env={"LNB_TC_GROUPS": "1"}),
    _c("mg-groups7", "nerf", "mg", 2100, 64, 33, 30, 3, "exact", env={"LNB_TC_GROUPS": "7"}),
    _c("v1-S1", "nerf", "v1", 1000, 1, 33, 30, 3, "exact"),
    _c("v1-env", "nerf", "v1", 1000, 64, 33, 30, 3, "exact", env={"LNB_TC_V1": "1"}),
    _c("fwd-only", "nerf", "fwd", 1000, 64, 33, 30, 3, "exact", grad=False),
    _c("fit-sigmoid", "fit", "mg", 1000, 1, 22, 16, 3, "exact"),
    _c("wide-64-L2", "nerf", "wide", 300, 64, 33, 64, 2, "exact"),
    _c("wide-256-L3", "nerf", "wide", 64, 96, 63, 256, 3, "exact"),
    _c("wide-fit-128-L3", "fit", "wide", 3000, 1, 22, 128, 3, "exact"),
    _c("bias-fused", "nerf", "mg", 400, 64, 33, 30, 3, "exact", offgrid_bias=True),
    _c("bias-wide", "nerf", "wide", 200, 64, 33, 128, 3, "exact", offgrid_bias=True),
]

REAL_CASES = [
    _c("c2", "nerf", "mg", 4096, 64, 5, 30, 3, "fused", seed="loss"),
    _c("w15", "nerf", "mg", 2000, 30, 5, 15, 3, "fused"),
    _c("L2-w8", "nerf", "mg", 1500, 64, 5, 8, 2, "fused", bounds=dict(out=1e-4, grad=6e-6, l2=5e-6)),
    _c("w48", "nerf", "mg", 900, 64, 5, 48, 3, "fused"),
    _c("w62-S100", "nerf", "mg", 600, 100, 3, 62, 2, "fused"),
    _c("L4-w20-rays", "nerf", "mg", 1200, 40, 2, 20, 4, "fused", rays=True),
    _c("k0p64-S128", "nerf", "mg", 300, 128, 8, 31, 3, "fused"),
    _c("E10-L2", "nerf", "mg", 2100, 64, 10, 30, 2, "fused"),
    _c("E5-L4", "nerf", "mg", 2100, 64, 5, 30, 4, "fused"),
    _c("E2-rays", "nerf", "mg", 500, 64, 2, 30, 3, "fused", rays=True),
    _c("c1-fit", "fit", "mg", 65536, 1, 5, 16, 3, "fused", bounds=dict(out=1e-7, grad=3e-6, l2=2e-6)),
    _c("fit-E8-L2", "fit", "mg", 1000, 1, 8, 31, 2, "fused"),
    _c("fit-129", "fit", "mg", 129, 1, 1, 4, 3, "fused"),
    _c("wide-9x256", "nerf", "wide", 64, 192, 10, 256, 9, "wide-deep"),
    _c("wide-5x256", "nerf", "wide", 300, 64, 10, 256, 5, "wide-deep", bounds=dict(out=4e-4, grad=1.2e-3, l2=4e-4)),
    _c("wide-4x128", "nerf", "wide", 1000, 33, 5, 128, 4, "wide"),
    _c("wide-3x200", "nerf", "wide", 50, 128, 4, 200, 3, "wide"),
    _c("wide-6x64", "nerf", "wide", 2048, 64, 10, 64, 4, "wide"),
    _c("wide-rays-E2", "nerf", "wide", 200, 64, 2, 128, 3, "wide", rays=True),
    _c("wide-fit-5x128", "fit", "wide", 5000, 1, 5, 128, 5, "wide"),
    _c("wide-fit-9x256", "fit", "wide", 20480, 1, 5, 256, 9, "wide-deep", bounds=dict(out=4e-4, grad=1.2e-3, l2=7e-4)),
    _c("wide-fit-3x70", "fit", "wide", 300, 1, 5, 70, 3, "wide"),
]
ALL_CASES = EXACT_CASES + REAL_CASES
# (a case's own `bounds`: 3x its own measured errors where they sit far below its family's)


def exact_case(c):
    """Dyadic operands: X = k/16 (|k| <= 16), weights k/16 (fan-in <= 64) or k/32 with |k| <= 3, hidden biases k/16 (or,
    with offgrid_bias, +-(1 + k/16) +- 2^-10: not bf16 numbers, but their bf16 rounding is on the k/16 grid), head biases
    k/16 + 2^-9 + 2^-14 (fp32 numbers, mostly not bf16 ones)."""
    rng = np.random.default_rng(sum(map(ord, c["id"])))
    nerf = c["kind"] == "nerf"
    R, S = c["R"], c["S"]
    N = R * S
    dims = O.mlp_dims(c["c_in"], c["width"], c["layers"], 4 if nerf else 3)
    L = len(dims) - 1
    ws = np.zeros((L, max(dims[:-1]), max(dims[1:])), np.float32)
    bs = np.zeros((L, max(dims[1:])), np.float32)
    for l in range(L):
        i, o = dims[l], dims[l + 1]
        ws[l, :i, :o] = rng.integers(-3, 4, (i, o)) / (16.0 if i <= 64 else 32.0)
        if l < L - 1 and c.get("offgrid_bias"):
            sign = rng.choice([-1.0, 1.0], o)
            bs[l, :o] = sign * (1.0 + rng.integers(0, 16, o) / 16.0) + rng.choice([-1.0, 1.0], o) * 2.0 ** -10
        else:
            bs[l, :o] = rng.integers(-8, 9, o) / 16.0
    bs[L - 1, :dims[L]] += 2.0 ** -9 + 2.0 ** -14
    if nerf:
        bs[L - 1, 3] += 1.0
    case = dict(X=(rng.integers(-16, 17, (N, dims[0])) / 16.0).astype(np.float32), ws=ws, bs=bs,
                dims=np.array(dims, np.int32), R=R, S=S)
    if nerf:
        case["target"] = rng.uniform(0, 1, (R, 3)).astype(np.float32)
        t = O.stratified_t(rng, R, S)
        case["dists"] = np.concatenate([t[:, 1:] - t[:, :-1], np.full((R, 1), 1e8)], 1).astype(np.float32)
    else:
        case["target"] = rng.uniform(0, 1, (R, 3)).astype(np.float32)
    return case


def make_case(c):
    if c["family"] == "exact":
        return exact_case(c)
    if c["kind"] == "fit":
        case = O.make_fit_case(3100 + c["width"] + c["layers"] + c["R"], c["R"], E=c["c_in"], width=c["width"], n_layers=c["layers"])
        case.update(R=c["R"], S=1)
        return case
    return O.make_nerf_case(5000 + c["R"] + c["width"], c["R"], c["S"], E=c["c_in"], width=c["width"], n_layers=c["layers"])


def bounds_of(c):
    return c.get("bounds") or BOUNDS[c["family"]]


def variant_of(c):
    return "wide" if c["path"] == "wide" else "fused"


def seed_of(c):
    return None if c.get("grad", True) is False else c.get("seed", 1.0)


def model(c, case, variant=None, bs=None):
    """The bf16 model of case c (variant: the path's own unless given; bs: replaces the biases)."""
    variant = variant or variant_of(c)
    bs = case["bs"] if bs is None else bs
    if c["kind"] == "fit":
        return M.fit_tc_model(case["X"], case["ws"], bs, case["dims"], case["target"], seed_of(c), variant)
    rays = (case["rays_o"], case["rays_d"], case["t"], case["E"]) if c.get("rays") else None
    return M.nerf_tc_model(case["X"], case["ws"], bs, case["dims"], case["target"], case["dists"], case["R"], case["S"],
                           seed_of(c), variant, rays=rays)


def errors(o, m, grad=True):
    """Every metric a bound is stated in: loss, colour, and the gradient metrics of conftest.grad_errs."""
    e = dict(loss=rel_err(np.ravel(o["loss"])[0], m["loss"]))
    if "color" in o and "color" in m:
        e["color"] = rel_err(o["color"], m["color"])
    if grad:
        e.update(grad_errs(o, m))
    return e


def over(errs, bounds):
    """errs / their bounds, largest first: a value above 1 is a failure."""
    r = {}
    for k, v in errs.items():
        b = bounds["out"] if k in ("loss", "color") else bounds["l2"] if k.endswith("_l2") else bounds["grad"]
        r[k] = v / b
    return dict(sorted(r.items(), key=lambda kv: -kv[1]))


def grid_exp(a):
    """The smallest e >= 0 with every value of a a multiple of 2^-e."""
    a = np.asarray(a, np.float64)
    for e in range(64):
        if np.all(np.mod(a * 2.0 ** e, 1.0) == 0):
            return e
    raise AssertionError("not dyadic")


def assert_exact_forward(c, case, m):
    """The exact-arithmetic precondition: for every layer, every term of every pre-activation sum (and the bias) lies on
    the grid 2^-g of the layer and the sum of their magnitudes is below 2^24 2^-g, so every fp32 partial sum is exact
    whatever the order (and whatever the tensor core's alignment of its addends)."""
    dims = [int(v) for v in case["dims"]]
    L = len(dims) - 1
    for l in range(L):
        A = m["A_l"][l]
        W = M.bf16(case["ws"][l, :dims[l], :dims[l + 1]])
        b = np.asarray(case["bs"][l, :dims[l + 1]], np.float64)
        if l < L - 1 and variant_of(c) == "fused":
            b = M.bf16(b)
        elif l == L - 1:
            b = np.zeros_like(b)    # the head's bias is one fp32 addition after the sum: a single rounding either way
        g = max(grid_exp(A) + grid_exp(W), grid_exp(b))
        total = np.abs(A) @ np.abs(W) + np.abs(b)
        assert total.max() < 2.0 ** (24 - g), (c["id"], l, g, total.max())


# ------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


@pytest.fixture(scope="module")
def ctx(torch_cuda):
    from loma_nerf_b200 import api
    cx = api.Context(0)
    yield cx
    cx.close()


def dev(torch, a, dtype=np.float32):
    return torch.as_tensor(np.ascontiguousarray(a, dtype)).cuda().contiguous()


EXPECT_KERNEL = {"mg": "fused_mg_kernel", "v1": "fused_v1_kernel", "fwd": "fused_v1_kernel", "wide": "chain_tc_kernel"}


def run(ctx, torch, c, case):
    """One step of case c on the tensor-core path; asserts which kernel ran."""
    dims = [int(v) for v in case["dims"]]
    grad = c.get("grad", True)
    seed = seed_of(c) or 1.0
    box = {}

    def call():
        if c["kind"] == "fit":
            box["o"] = ctx.fit_step(dims, dev(torch, case["X"]), dev(torch, case["ws"]), dev(torch, case["bs"]), dev(torch, case["target"]),
                                    grad=grad, seed=seed, outputs=("loss",), path="tc")
        elif c.get("rays"):
            r = [dev(torch, case[k], np.float64) for k in ("rays_o", "rays_d", "t")]
            box["o"] = ctx.nerf_step_rays(dims, r[0], r[1], r[2], int(case["E"]), dev(torch, case["ws"]), dev(torch, case["bs"]),
                                          dev(torch, case["target"]), grad=grad, seed=seed, outputs=("color", "loss"), path="tc")
        else:
            box["o"] = ctx.nerf_step(dims, dev(torch, case["X"]), dev(torch, case["ws"]), dev(torch, case["bs"]), dev(torch, case["dists"]),
                                     dev(torch, case["target"]), R=case["R"], S=case["S"], grad=grad, seed=seed,
                                     outputs=("color", "loss"), path="tc")
    saved = {k: os.environ.get(k) for k in c.get("env", {})}
    os.environ.update(c.get("env", {}))
    try:
        prof = ctx.profile_dominant(call)
        ctx.synchronize()
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    assert prof is not None and prof["kernel"].startswith(EXPECT_KERNEL[c["path"]]), (c["id"], prof)
    return {k: v.cpu().numpy() for k, v in box["o"].items()}


@pytest.mark.parametrize("c", EXACT_CASES, ids=lambda c: c["id"])
def test_exact_arithmetic_cases_against_the_bf16_model(ctx, torch_cuda, c):
    case = make_case(c)
    m = model(c, case)
    assert_exact_forward(c, case, m)
    o = run(ctx, torch_cuda, c, case)
    grad = c.get("grad", True)
    errs = errors(o, m, grad)
    log("tc-model exact %s %s" % (c["id"], {k: "%.3g" % v for k, v in errs.items()}))
    r = over(errs, BOUNDS["exact"])
    assert max(r.values()) <= 1.0, (c["id"], errs)
    if c.get("offgrid_bias"):
        # each path's bias precision: its own variant within the bound, the other one at least 100x farther (colour: the
        # forward is exact, so the distance to the own variant there is the compositing's fp32 rounding only)
        other = model(c, case, variant="fused" if variant_of(c) == "wide" else "wide")
        e_other = rel_err(o["color"], other["color"])
        log("tc-model exact %s colour vs the other bias variant %.3g" % (c["id"], e_other))
        assert e_other >= 100 * max(errs["color"], 1e-9), (c["id"], errs["color"], e_other)


@pytest.mark.parametrize("c", REAL_CASES, ids=lambda c: c["id"])
def test_realistic_cases_against_the_bf16_model(ctx, torch_cuda, c):
    case = make_case(c)
    m = model(c, case)
    o = run(ctx, torch_cuda, c, case)
    errs = errors(o, m)
    log("tc-model real %s %s" % (c["id"], {k: "%.3g" % v for k, v in errs.items()}))
    r = over(errs, bounds_of(c))
    assert max(r.values()) <= 1.0, (c["id"], errs)


# ------------------------------------------------------------------------------------------------
# trainer
# ------------------------------------------------------------------------------------------------
def pow_int(b, t):
    """beta^t by squaring in float64, as pow_int in fused_tc.cu."""
    r = 1.0
    while t > 0:
        if t & 1:
            r *= b
        b *= b
        t >>= 1
    return r


def adam_emulate(p0, g, m, v, t, lr, b1, b2, eps):
    """adam_one (fused_tc.cu) in float32 numpy: returns the new parameters, updates m and v in place."""
    f = np.float32
    c1, c2 = 1.0 - pow_int(b1, t), 1.0 - pow_int(b2, t)
    lr_t, c1f, c2f = f(lr * (np.sqrt(c2) / c1)), f(c1), f(c2)
    m[...] = f(b1) * m + f(1.0 - b1) * g
    v[...] = f(b2) * v + f(1.0 - b2) * (g * g)
    return (p0 - lr_t * (m / c1f) / (np.sqrt(v / c2f) + f(eps))).astype(np.float32)


def assert_update(got, p0, want, live):
    """Every live parameter within 2 ulp of the emulation (nvcc may contract to FMA; an ulp of the update is allowed for
    each rounding it goes through); padded ones bit-identical to what they were."""
    upd = np.abs(want.astype(np.float64) - p0)
    tol = 2 * np.spacing(np.abs(want)).astype(np.float64) + 4 * np.spacing(upd.astype(np.float32)).astype(np.float64)
    diff = np.abs(got.astype(np.float64) - want)
    bad = live & (diff > tol)
    assert not bad.any(), (int(bad.sum()), float((diff / np.maximum(tol, 1e-45))[live].max()))
    assert np.array_equal(got[~live], p0[~live])


def live_masks(dims, ws_shape, bs_shape):
    lw, lb = np.zeros(ws_shape, bool), np.zeros(bs_shape, bool)
    for l in range(len(dims) - 1):
        lw[l, :dims[l], :dims[l + 1]] = True
        lb[l, :dims[l + 1]] = True
    return np.concatenate([lw.ravel(), lb.ravel()])


def fresh_step(ctx, torch, dims, p, ws_shape, batch, fit):
    """The same batch through ctx.nerf_step / fit_step: a weight image built afresh by tc_prep_kernel from p."""
    nw = int(np.prod(ws_shape))
    ws, bs = p[:nw].reshape(ws_shape), p[nw:].reshape(ws_shape[0], ws_shape[2])
    if fit:
        out = ctx.fit_step(dims, batch["X"], dev(torch, ws), dev(torch, bs), batch["target"], grad=True, seed=1.0, outputs=("loss",), path="tc")
    else:
        out = ctx.nerf_step(dims, batch["X"], dev(torch, ws), dev(torch, bs), batch["dists"], batch["target"], grad=True, seed=1.0,
                            outputs=("loss",), path="tc")
    ctx.synchronize()
    return np.concatenate([out["d_ws"].cpu().numpy().ravel(), out["d_bs"].cpu().numpy().ravel()]), float(out["loss"].cpu().numpy()[0])


def trainer_walk(ctx, torch, dims, ws0, bs0, batches, forms, fit=False, optimizer="adam", lr=5e-4, b1=0.9, b2=0.999, eps=1e-8,
                 label=""):
    """Update after update, check the trainer against the emulation of its optimiser fed with its own gradients, and the
    gradients / loss it computed on its (refreshed) weight image against a freshly built image of the same parameters.
    forms[i]: "step" (fused reduce + update), "grad+apply" (tc_adam_img_kernel)."""
    from loma_nerf_b200 import api
    head = api.L.HEAD_SIGMOID if fit else api.L.HEAD_NERF
    tr = api.Trainer(ctx, dims, ws0, bs0, head=head, optimizer=optimizer, lr=lr, beta1=b1, beta2=b2, eps=eps)
    live = live_masks(dims, ws0.shape, bs0.shape)
    nw = ws0.size
    m = np.zeros(ws0.size + bs0.size, np.float32)
    v = np.zeros_like(m)
    worst = 0.0
    try:
        for t, (batch, form) in enumerate(zip(batches, forms), start=1):
            w, b, _ = tr.read()
            p0 = np.concatenate([w.ravel(), b.ravel()])
            tb = dict(batch, path="tc")
            if form == "step":
                tr.step(**tb)
            else:
                tr.grad(**tb)
            ctx.synchronize()
            gbuf = tr.grad_buffer().cpu().numpy().copy()
            g, loss = gbuf[:-1], float(gbuf[-1])
            if form != "step":
                tr.apply()
            w, b, loss_read = tr.read()
            got = np.concatenate([w.ravel(), b.ravel()])
            # the image the step ran on (refreshed in place by the previous update) = one built afresh
            g_fresh, loss_fresh = fresh_step(ctx, torch, dims, p0, ws0.shape, batch, fit)
            assert loss == loss_fresh, (label, t, loss, loss_fresh)
            e = max(rel_err(g[:nw], g_fresh[:nw]), rel_err(g[nw:], g_fresh[nw:]))
            worst = max(worst, e)
            assert e <= 1e-5, (label, t, e)
            if optimizer == "sgd":
                want = (p0 - np.float32(lr) * g).astype(np.float32)
            else:
                want = adam_emulate(p0, g, m, v, t, lr, b1, b2, eps)
            assert_update(got, p0, want, live)
    finally:
        tr.close()
    log("tc-model trainer %s: %d updates exact to 2 ulp, refreshed vs fresh image: loss bit-equal, gradients %.3g" % (label, len(batches), worst))


def test_trainer_adam_fused_update_and_image_refresh(ctx, torch_cuda):
    torch = torch_cuda
    cases = [O.make_nerf_case(7100 + i, 256, 64) for i in range(5)]
    dims = [int(v) for v in cases[0]["dims"]]
    batches = [dict(X=dev(torch, c["X"]), dists=dev(torch, c["dists"]), target=dev(torch, c["target"])) for c in cases]
    trainer_walk(ctx, torch, dims, cases[0]["ws"], cases[0]["bs"], batches, ["step", "grad+apply", "step", "step", "grad+apply"],
                 label="adam C2-net")


def test_trainer_sgd_sigmoid_head_c1_shape(ctx, torch_cuda):
    """What bench.py --workload c1 trains: the sigmoid head with SGD (lr 1e-4) on 65536-row batches."""
    torch = torch_cuda
    cases = [O.make_fit_case(7200 + i, 65536, E=5, width=16, n_layers=3) for i in range(4)]
    dims = [int(v) for v in cases[0]["dims"]]
    batches = [dict(X=dev(torch, c["X"]), target=dev(torch, c["target"])) for c in cases]
    trainer_walk(ctx, torch, dims, cases[0]["ws"], cases[0]["bs"], batches, ["step", "grad+apply", "step", "grad+apply"], fit=True,
                 optimizer="sgd", lr=1e-4, label="sgd C1")


def test_trainer_batch_the_fused_kernel_cannot_take(ctx, torch_cuda):
    """S = 192 > 128: the step falls back to the layerwise tensor-core kernels and the update to tc_adam_img_kernel, whose
    image refresh the next (fused) batch then runs on."""
    torch = torch_cuda
    big = O.make_nerf_case(7300, 16, 192)
    small = [O.make_nerf_case(7301 + i, 128, 64) for i in range(2)]
    dims = [int(v) for v in big["dims"]]
    bt = lambda c: dict(X=dev(torch, c["X"]), dists=dev(torch, c["dists"]), target=dev(torch, c["target"]))  # noqa: E731
    trainer_walk(ctx, torch, dims, big["ws"], big["bs"], [bt(big), bt(small[0]), bt(big), bt(small[1])],
                 ["step", "step", "grad+apply", "grad+apply"], label="adam S=192 fallback")
