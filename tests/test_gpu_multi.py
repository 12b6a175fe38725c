"""Data-parallel training on 2, 3, 4 and 8 GPUs (the worlds the box has) against the whole-batch step.

Two routes combine the ranks' gradients: the peer exchange fused into the tensor-core step's reduction kernel
(Trainer.enable_peer_allreduce, then step / step_host / submit_host) and sharding.data_parallel_step (grad, an NCCL
all-reduce of the grad buffer, apply), which the wide and the exact path always take.  One mp.spawn per world runs every
case on every rank; each rank saves, per step, its parameters before and after the step and its reduced grad buffer
[d_ws | d_bs | loss].  The parent process then holds every step to:
  * rank agreement: grad buffers and parameters bit-identical on every rank;
  * the whole batch: the reduced gradient and loss against the whole batch's reference at the pre-step parameters --
    the bf16 model (oracle/tc_model.py, tests/composite_model.py with a background) at the bounds of
    test_gpu_tc_model.py for the tensor-core routes (sharding changes only the fp32 order in which partial sums are
    added, not where bf16 rounding happens), the float64 restatement at test_gpu_parity.py's tolerance for the exact one;
  * the update: the fp32 emulation of the kernels' Adam fed with the rank's own reduced gradient, to 2 ulp, padding
    untouched;
  * the losses wait() and step_host() return: the reduced buffer's, in submission order.
Every case runs with seed 1.0 and seed "loss" (the whole batch's loss times its unit-seed gradient).  Per case the parent
also shows, on the CPU, that the bound would catch the two faults a data-parallel step can make: adding up the shards'
loss-seeded gradients (sum_r L_r g_r) and losing one rank's shard.
"""
import os
import socket
import sys
import traceback
from datetime import timedelta

import numpy as np
import pytest

import composite_model as CM
from conftest import ROOT, rel_err
from oracle import oracle as O
from oracle import tc_model as M
from oracle import viewdirs as V
from test_gpu_parity import TOL as F64_TOL
from test_gpu_tc import log
from test_gpu_tc_model import BOUNDS, adam_emulate, assert_update, errors, live_masks, over

pytestmark = pytest.mark.gpu

WORLDS = (2, 3, 4, 8)
SEEDS = (1.0, "loss")
STEPS = 2                     # steps per case (the walk takes more)
LR, B1, B2, EPS = 5e-4, 0.9, 0.999, 1e-8   # the Trainer's Adam defaults


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _c(id, route, path, R, S, E=5, width=30, layers=3, **kw):
    return dict(id=id, route=route, path=path, R=R, S=S, E=E, width=width, layers=layers, seed=sum(map(ord, id)) * 10, **kw)


# Cases that BOUNDS["fused"] does not fit, for reasons that have nothing to do with the sharding: the errors below are the
# same on both routes and at every world (2, 3, 4, 8), so they come from the input.  Bounds at about 3x of them, the
# worst over all steps, worlds, routes and seeds, measured on a B200 (1000 W) and written to the error log by every run.
# Rays mode: the kernels encode with fast sin / cos (and their own fp32 unit direction), so a bf16 rounding of A_0 can flip
# against the model's float64 encoding (oracle/tc_model.py).  Which roundings flip depends on the data: test_gpu_tc_model's
# "E2-rays" batch stays within BOUNDS["fused"], this one measures d_ws 8.3e-5 per layer and 3.9e-5 in L2.  With
# directions a flipped feature is shared by a ray's 64 samples: d_ws 4.1e-4 per layer, 2.6e-4 in L2.
RAYS_BOUNDS = dict(out=4e-4, grad=2.5e-4, l2=1.2e-4)
DIRS_BOUNDS = dict(out=4e-4, grad=1.25e-3, l2=8e-4)
# A batch of 1 - 5 rays is 64 - 320 sample rows: one flipped bf16 rounding of an adjoint weighs 1/64 .. 1/320 of a weight
# gradient there, where the fused family's batches sum over thousands: d_ws 6.2e-5 per layer and 2.6e-5 in L2 at R = 2.
FEW_RAYS_BOUNDS = dict(out=4e-4, grad=2e-4, l2=8e-5)


def cases(world):
    """Every (route, shape) of the matrix at this world size.  R = 480 divides every world; 4097 and 241 do not (and leave
    tail tiles); a C2 batch of fewer rays than ranks leaves some shards empty."""
    few = {2: 1, 3: 2, 4: 3, 8: 5}[world]
    fused = [_c("c2", None, "tc", 480, 64), _c("c2-4097", None, "tc", 4097, 64), _c("c2-empty", None, "tc", few, 64, bounds=FEW_RAYS_BOUNDS),
             _c("rays-E2", None, "tc", 480, 64, E=2, rays=True, bounds=RAYS_BOUNDS),
             _c("rays-E2-dirs", None, "tc", 480, 64, E=2, rays=True, dir_bands=2, bounds=DIRS_BOUNDS),
             _c("bg", None, "tc", 480, 64, bg=(1.0, 1.0, 1.0))]
    out = [dict(c, id=route + "-" + c["id"], route=route) for route in ("peer", "nccl") for c in fused]
    out += [_c("nccl-wide", "nccl", "tc", 240, 64, E=10, width=128, layers=4),
            _c("nccl-wide-uneven", "nccl", "tc", 241, 64, E=10, width=128, layers=4),
            _c("nccl-exact", "nccl", "f32", 240, 32),
            _c("nccl-exact-uneven", "nccl", "f32", 241, 32)]
    return out


# The peer walk: one trainer through every entry point, the step tag and slot parity advancing through all of them (each
# parity buffer is reused several times), two steps it must refuse in the middle, and one grad + NCCL all-reduce + apply.
WALK_CASE = _c("walk", "peer", "tc", 480, 64)
WALK = ["step", "step_host", "submit", "submit+wait", "refuse-S192", "nccl", "refuse-f32", "step", "submit+wait", "step_host",
        "step"]


def family(c):
    return "exact" if c["path"] == "f32" else "wide" if c["width"] > 63 else "fused"


def make_batch(c, step):
    """Step `step`'s whole batch of case c (numpy; step 0 also carries the initial parameters) and Xm, the bf16 model's
    input rows (in rays mode: the features of the fp32 sample positions, as the kernels form them)."""
    b = V.make_nerf_case(c["seed"] + step, c["R"], c["S"], E=c["E"], E_dir=c.get("dir_bands"), width=c["width"],
                         n_layers=c["layers"])
    b["Xm"] = b["X"]
    if c.get("rays"):
        b["Xm"] = M.rays_features(b["rays_o"], b["rays_d"], b["t"], c["E"])
        if c.get("dir_bands") is not None:
            b["Xm"] = np.concatenate([b["Xm"], V.view_encoding(b["rays_d"], c["dir_bands"], c["S"])], 1)
    return b


def reference(c, b, ws, bs, seed, lo=0, hi=None):
    """Case c's reference on rays [lo, hi) of batch b at the parameters (ws, bs)."""
    S = c["S"]
    hi = c["R"] if hi is None else hi
    X, dists, target = b["Xm"][lo * S:hi * S], b["dists"][lo:hi], b["target"][lo:hi]
    if c["path"] == "f32":
        return O.nerf_f64(X, ws, bs, b["dims"], target, dists, hi - lo, S, g=seed)
    return CM.nerf_tc_model(X, ws, bs, b["dims"], target, dists, hi - lo, S, g=seed,
                            variant="wide" if family(c) == "wide" else "fused", bg=c.get("bg"))


# ------------------------------------------------------------------------------------------------
# worker (one process per rank)
# ------------------------------------------------------------------------------------------------
def _kernel_batch(torch, c, b, world, rank, host=False):
    from loma_nerf_b200 import sharding
    keys = ("rays_o", "rays_d", "t", "target") if c.get("rays") else ("X", "dists", "target")
    sh = sharding.shard_rays({k: b[k] for k in keys}, world, rank, c["S"])
    if host:
        sh = {k: np.ascontiguousarray(v, np.float32) for k, v in sh.items()}
    else:
        sh = {k: torch.as_tensor(np.ascontiguousarray(v, np.float64 if k in ("rays_o", "rays_d", "t") else np.float32)).cuda()
              for k, v in sh.items()}
    if c.get("rays"):
        return dict(rays=(sh["rays_o"], sh["rays_d"], sh["t"]), pe_bands=c["E"], dir_bands=c.get("dir_bands"),
                    target=sh["target"], path=c["path"])
    return dict(sh, path=c["path"])


def _params(tr):
    w, b, _ = tr.read()
    return np.concatenate([w.ravel(), b.ravel()])


def _run_steps(ctx, torch, c, seed, forms, world, rank, rec):
    from loma_nerf_b200 import api, sharding
    b0 = make_batch(c, 0)
    tr = api.Trainer(ctx, [int(v) for v in b0["dims"]], b0["ws"], b0["bs"], background=c.get("bg"))
    try:
        if c["route"] == "peer":
            tr.enable_peer_allreduce()
        for i, form in enumerate(forms):
            if form.startswith("refuse"):
                bad = dict(c, S=192, R=2 * world) if form == "refuse-S192" else dict(c, path="f32")
                kb = _kernel_batch(torch, bad, make_batch(bad, i), world, rank)
            else:
                b = make_batch(c, i)
                kb = _kernel_batch(torch, c, b, world, rank, host=form.startswith(("step_host", "submit")))
            rec["p0_%d" % i] = _params(tr)
            try:
                if form.startswith("refuse") or form == "step":
                    tr.step(**kb, seed=seed)
                elif form == "step_host":
                    rec["loss_%d" % i] = np.float32(tr.step_host(**kb, seed=seed))
                elif form.startswith("submit"):
                    tr.submit_host(**kb, seed=seed)
                else:
                    sharding.data_parallel_step(tr, dict(kb, seed=seed))
                rec["refused_%d" % i] = np.array("")
            except api.LnbError as e:
                if not form.startswith("refuse"):
                    raise
                rec["refused_%d" % i] = np.array(str(e))
            ctx.synchronize()
            rec["g_%d" % i] = tr.grad_buffer().cpu().numpy().copy()
            if form.endswith("+wait"):
                rec["wait_%d" % i] = np.array(tr.wait(), np.float32)
            rec["p1_%d" % i] = _params(tr)
        rec["status"] = np.int32(tr.comm_status() if c["route"] == "peer" else 0)
    finally:
        torch.cuda.synchronize()
        tr.close()


def _refuse_wide(ctx, torch, world, rank, rec):
    """A wide MLP cannot join the peer exchange: attaching it is refused on every rank, before any collective."""
    from loma_nerf_b200 import api
    b = make_batch(_c("refuse-wide", "peer", "tc", 2 * world, 64, width=128), 0)
    tr = api.Trainer(ctx, [int(v) for v in b["dims"]], b["ws"], b["bs"])
    try:
        rec["p0_0"] = _params(tr)
        try:
            tr.enable_peer_allreduce()
            rec["refused_0"] = np.array("")
        except api.LnbError as e:
            rec["refused_0"] = np.array(str(e))
        rec["p1_0"] = _params(tr)
    finally:
        tr.close()


def _path(out_dir, name, seed, rank):
    return os.path.join(out_dir, "%s_%s_r%d.npz" % (name, seed, rank))


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from loma_nerf_b200 import api
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank),
                            timeout=timedelta(seconds=120))
    ctx = api.Context(rank)
    ctx.set_stream(torch.cuda.current_stream())
    jobs = [(c["id"], s, lambda rec, c=c, s=s: _run_steps(ctx, torch, c, s, ["step" if c["route"] == "peer" else "nccl"] * STEPS,
                                                          world, rank, rec)) for c in cases(world) for s in SEEDS]
    jobs += [("walk", s, lambda rec, s=s: _run_steps(ctx, torch, WALK_CASE, s, WALK, world, rank, rec)) for s in SEEDS]
    jobs += [("refuse-wide", 1.0, lambda rec: _refuse_wide(ctx, torch, world, rank, rec))]
    for name, seed, job in jobs:
        rec = {}
        try:
            job(rec)
        except Exception:
            # A rank that fails mid-case may leave its peers inside a collective it will never join.  It records the error
            # and ends with it: mp.spawn then stops every rank at once, instead of the peers waiting out the NCCL timeout.
            np.savez(_path(out_dir, name, seed, rank), error=np.array(traceback.format_exc()))
            raise
        np.savez(_path(out_dir, name, seed, rank), **rec)
        dist.barrier()
    ctx.close()
    dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# parent
# ------------------------------------------------------------------------------------------------
_RUNS = {}


def _run_world(world, tmp_path_factory):
    """Spawn the world's ranks once.  The outcome -- success, or the error that ended the run -- is kept for every later
    test of that world: those read the records written before the run ended and never spawn the world again."""
    if world not in _RUNS:
        import torch.multiprocessing as mp
        out = str(tmp_path_factory.mktemp("world%d" % world))
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        try:
            mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
            _RUNS[world] = (out, None)
        except Exception as e:
            _RUNS[world] = (out, "%s: %s" % (type(e).__name__, e))
    return _RUNS[world]


def _load(run, name, seed, world):
    out, failure = run
    paths = [_path(out, name, seed, r) for r in range(world)]
    recs = [dict(np.load(p)) for p in paths if os.path.exists(p)]
    errs = [str(r["error"]) for r in recs if "error" in r]
    assert not errs, errs[0]
    if len(recs) < world:
        pytest.fail("the world %d run ended before %s (seed %s): %s" % (world, name, seed, failure))
    return recs


def _split(c, b, flat):
    nw = b["ws"].size
    return flat[:nw].reshape(b["ws"].shape), flat[nw:nw + b["bs"].size].reshape(b["bs"].shape)


def _errs(c, o, ref):
    """The metrics case c is bounded in, and the bound as a function of them (a value above 1 fails)."""
    if family(c) == "exact":
        e = dict(loss=rel_err(o["loss"], ref["loss"]), d_ws=rel_err(o["d_ws"], ref["d_ws"]), d_bs=rel_err(o["d_bs"], ref["d_bs"]))
        return e, max(e.values()) / F64_TOL
    e = errors(o, ref)
    return e, max(over(e, c.get("bounds") or BOUNDS[family(c)]).values())


def _as_output(c, b, g):
    d_ws, d_bs = _split(c, b, g[:-1])
    return dict(loss=np.float64(g[-1]), d_ws=d_ws, d_bs=d_bs)


def _discrimination(c, b, ws, bs, seed, world, ref, label):
    """The faults the bounds must catch, from the reference's own pieces: each rank's unit-seed gradient and loss."""
    from loma_nerf_b200 import sharding
    spans = [sharding.shard_bounds(c["R"], world, r) for r in range(world)]
    parts = [reference(c, b, ws, bs, 1.0, lo, hi) for lo, hi in spans if hi > lo]
    scale = float(ref["loss"]) if seed == "loss" else 1.0
    zero = {k: np.zeros_like(ref[k]) for k in ("d_ws", "d_bs")}
    faults = {"rank 0's shard dropped": dict(ref, **{k: scale * sum((p[k] for p in parts[1:]), zero[k]) for k in zero})}
    if seed == "loss" and len(parts) > 1:     # (with one non-empty shard the two combinations agree)
        faults["sum_r L_r g_r"] = dict(ref, **{k: sum(p["loss"] * p[k] for p in parts) for k in zero})
    for name, f in faults.items():
        e, r = _errs(c, f, ref)
        log("multi-gpu %s fault %-22s %.3g x the bound %s" % (label, name, r, {k: "%.3g" % v for k, v in e.items()}))
        assert r >= 10.0, (label, name, e)


def check_steps(c, seed, world, recs, forms, label):
    b0 = make_batch(c, 0)
    dims = [int(v) for v in b0["dims"]]
    live = live_masks(dims, b0["ws"].shape, b0["bs"].shape)
    m = np.zeros(b0["ws"].size + b0["bs"].size, np.float32)
    v = np.zeros_like(m)
    t, pending, worst = 0, [], {}
    assert all(int(r.get("status", 0)) == 0 for r in recs), label
    for i, form in enumerate(forms):
        for k in ("p0_%d" % i, "g_%d" % i, "p1_%d" % i):
            for r, rec in enumerate(recs[1:], 1):
                assert np.array_equal(rec[k], recs[0][k]), (label, i, form, k, r)      # the replicas never diverge
        p0, g, p1 = (recs[0][k % i] for k in ("p0_%d", "g_%d", "p1_%d"))
        if form.startswith("refuse"):
            msgs = [str(rec["refused_%d" % i]) for rec in recs]
            assert all(msgs), (label, i, form, msgs)                   # every rank refused ...
            assert np.array_equal(p1, p0), (label, i, form)            # ... and its parameters did not move
            continue
        assert not str(recs[0]["refused_%d" % i]), (label, i, form)
        t += 1
        b = make_batch(c, i)
        ws, bs = _split(c, b, p0)
        ref = reference(c, b, ws, bs, seed)
        e, r = _errs(c, _as_output(c, b, g), ref)
        worst = {k: max(worst.get(k, 0.0), x) for k, x in e.items()}
        assert r <= 1.0, (label, i, form, e)
        if i == 0:
            _discrimination(c, b, ws, bs, seed, world, ref, label)
        want = adam_emulate(p0, g[:-1], m, v, t, LR, B1, B2, EPS)
        assert_update(p1, p0, want, live)
        if form == "step_host":
            assert recs[0]["loss_%d" % i] == g[-1], (label, i)
        if form.startswith("submit"):
            pending.append(g[-1])
        if form.endswith("+wait"):
            assert np.array_equal(recs[0]["wait_%d" % i], np.array(pending, np.float32)), (label, i)
            pending = []
    log("multi-gpu %s: %d steps, worst %s" % (label, t, {k: "%.3g" % x for k, x in worst.items()}))


def _params_of(world):
    return [pytest.param(world, c, s, id="%d-%s-%s" % (world, c["id"], s),
                         marks=pytest.mark.skipif(_n_gpus() < world, reason="needs %d GPUs" % world))
            for c in cases(world) for s in SEEDS]


@pytest.mark.parametrize("world,c,seed", [p for w in WORLDS for p in _params_of(w)])
def test_data_parallel_step_is_the_whole_batch_step(tmp_path_factory, world, c, seed):
    recs = _load(_run_world(world, tmp_path_factory), c["id"], seed, world)
    forms = ["step" if c["route"] == "peer" else "nccl"] * STEPS
    check_steps(c, seed, world, recs, forms, "world %d %s seed %s" % (world, c["id"], seed))


@pytest.mark.parametrize("world,seed", [pytest.param(w, s, id="%d-%s" % (w, s), marks=pytest.mark.skipif(_n_gpus() < w, reason="needs %d GPUs" % w))
                                        for w in WORLDS for s in SEEDS])
def test_peer_allreduce_matches_nccl_path_and_ranks_agree(tmp_path_factory, world, seed):
    """The two routes on the same shards from the same parameters: the same reduced gradient up to the order of the
    ranks' sum (which two ranks cannot change: the parameters then agree too)."""
    run = _run_world(world, tmp_path_factory)
    p, n = (_load(run, route + "-c2", seed, world)[0] for route in ("peer", "nccl"))
    assert np.array_equal(p["p0_0"], n["p0_0"])
    assert rel_err(p["g_0"][:-1], n["g_0"][:-1]) <= 1e-6 and abs(float(p["g_0"][-1]) - float(n["g_0"][-1])) <= 1e-6 * abs(float(n["g_0"][-1]))
    if world == 2:
        for i in range(STEPS):
            assert rel_err(p["p1_%d" % i], n["p1_%d" % i]) <= 1e-6, i


@pytest.mark.parametrize("world,seed", [pytest.param(w, s, id="%d-%s" % (w, s), marks=pytest.mark.skipif(_n_gpus() < w, reason="needs %d GPUs" % w))
                                        for w in WORLDS for s in SEEDS])
def test_peer_walk_through_every_entry_point(tmp_path_factory, world, seed):
    check_steps(WALK_CASE, seed, world, _load(_run_world(world, tmp_path_factory), "walk", seed, world), WALK, "world %d walk seed %s" % (world, seed))


@pytest.mark.parametrize("world", [pytest.param(w, marks=pytest.mark.skipif(_n_gpus() < w, reason="needs %d GPUs" % w)) for w in WORLDS])
def test_wide_mlp_cannot_join_the_peer_exchange(tmp_path_factory, world):
    recs = _load(_run_world(world, tmp_path_factory), "refuse-wide", 1.0, world)
    assert all(str(r["refused_0"]) for r in recs)
    for r in recs:
        assert np.array_equal(r["p1_0"], r["p0_0"]) and np.array_equal(r["p0_0"], recs[0]["p0_0"])
