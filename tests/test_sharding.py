"""Host-side logic of the multi-GPU path, on CPU with the gloo backend: shard boundaries never split
a ray, the all-reduced sum of per-shard gradients equals the whole-batch gradient (the property
data-parallel training rests on, SURVEY.md 8e), data_parallel_step applies the whole batch's
gradient under either seed rule, frames are disjoint."""
import os
import socket
import sys

import numpy as np
import pytest

from conftest import ROOT, rel_err


def test_shard_bounds_cover_everything_once():
    from loma_nerf_b200 import sharding
    for n in (0, 1, 7, 4096, 4097):
        for w in (1, 2, 3, 8):
            spans = [sharding.shard_bounds(n, w, r) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            assert max(b - a for a, b in spans) - min(b - a for a, b in spans) <= 1
    with pytest.raises(ValueError):
        sharding.shard_bounds(4, 2, 2)


def test_shard_rays_keeps_rays_whole():
    from loma_nerf_b200 import sharding
    R, S = 10, 7
    batch = dict(X=np.arange(R * S * 3).reshape(R * S, 3), dists=np.arange(R * S).reshape(R, S),
                 target=np.arange(R * 3).reshape(R, 3), path="f32", pe_bands=5)
    got = [sharding.shard_rays(batch, 3, r, S) for r in range(3)]
    assert sum(g["target"].shape[0] for g in got) == R
    for g in got:
        assert g["X"].shape[0] == g["target"].shape[0] * S and g["path"] == "f32" and g["pe_bands"] == 5
    assert np.array_equal(np.concatenate([g["X"] for g in got]), batch["X"])
    assert sorted(sum((sharding.frames_for_rank(120, 8, r) for r in range(8)), [])) == list(range(120))


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from loma_nerf_b200 import sharding
    from oracle import oracle as O
    dist.init_process_group("gloo", rank=rank, world_size=world)
    R, S = 12, 16
    case = O.make_nerf_case(4242, R, S)
    batch = dict(X=case["X"], dists=case["dists"], target=case["target"])
    mine = sharding.shard_rays(batch, world, rank, S)
    r_loc = mine["target"].shape[0]
    # per-shard gradient from the oracle (the CUDA path is checked against it on the GPU box)
    f = O.nerf_f64(mine["X"], case["ws"], case["bs"], case["dims"], mine["target"], mine["dists"], r_loc, S, g=1.0)
    flat = np.concatenate([f["d_ws"].ravel(), f["d_bs"].ravel(), [f["loss"]]]).astype(np.float32)
    sharding.allreduce_gradients(flat)
    np.save(os.path.join(out_dir, "flat_%d.npy" % rank), flat)
    dist.destroy_process_group()


def test_allreduced_shard_gradients_equal_whole_batch_gradient(tmp_path):
    import torch.multiprocessing as mp
    from oracle import oracle as O
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    R, S = 12, 16
    case = O.make_nerf_case(4242, R, S)
    f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, S, g=1.0)
    whole = np.concatenate([f["d_ws"].ravel(), f["d_bs"].ravel(), [f["loss"]]])
    a, b = (np.load(os.path.join(tmp_path, "flat_%d.npy" % r)) for r in range(2))
    assert np.array_equal(a, b)                         # every rank ends with the same buffer
    assert rel_err(a, whole) <= 1e-5                    # reduction order changes rounding only


# data_parallel_step with a stand-in trainer: the float64 oracle gradient of the shard under the kernels' seed rule (seed
# "loss": the shard's own loss), the float32 buffer the library hands to the all-reduce, and an apply() that records it
DP_S = 16
DP_R = (12, 13, 1)            # rays per batch: divisible by 2, uneven at 3, and fewer rays than ranks (an empty shard)
DP_SEEDS = (1.0, "loss")


class _Ctx:
    def order_torch_after(self):
        pass

    def order_after_torch(self):
        pass


class _OracleTrainer:
    def __init__(self, case):
        self.case, self.ctx, self.applied = case, _Ctx(), []

    def grad(self, X, dists, target, seed=1.0, path="tc"):
        import torch
        from oracle import oracle as O
        c = self.case
        f = O.nerf_f64(X, c["ws"], c["bs"], c["dims"], target, dists, target.shape[0], DP_S, g=seed)
        self.buf = torch.from_numpy(np.concatenate([f["d_ws"].ravel(), f["d_bs"].ravel(), [f["loss"]]]).astype(np.float32))

    def grad_buffer(self):
        return self.buf

    def apply(self):
        self.applied.append(self.buf.numpy().copy())


def _dp_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from loma_nerf_b200 import sharding
    from oracle import oracle as O
    dist.init_process_group("gloo", rank=rank, world_size=world)
    for R in DP_R:
        case = O.make_nerf_case(4242 + R, R, DP_S)
        for seed in DP_SEEDS:
            tr = _OracleTrainer(case)
            batch = dict(X=case["X"], dists=case["dists"], target=case["target"])
            sharding.data_parallel_step(tr, dict(sharding.shard_rays(batch, world, rank, DP_S), seed=seed, path="tc"))
            assert len(tr.applied) == 1
            np.save(os.path.join(out_dir, "dp_%d_%s_%d.npy" % (R, seed, rank)), tr.applied[0])
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_data_parallel_step_applies_the_whole_batch_gradient(tmp_path, world):
    """Every rank applies the whole batch's gradient and loss, for a unit seed and for the loss seed (the whole batch's
    loss times its unit-seed gradient, not the sum of the shards' loss-seeded gradients), on even and uneven shards and
    with a rank whose shard is empty."""
    import torch.multiprocessing as mp
    from oracle import oracle as O
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_dp_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    for R in DP_R:
        case = O.make_nerf_case(4242 + R, R, DP_S)
        for seed in DP_SEEDS:
            f = O.nerf_f64(case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], R, DP_S, g=seed)
            whole = np.concatenate([f["d_ws"].ravel(), f["d_bs"].ravel()])
            got = [np.load(os.path.join(tmp_path, "dp_%d_%s_%d.npy" % (R, seed, r))) for r in range(world)]
            for g in got[1:]:
                assert np.array_equal(g, got[0]), (R, seed)      # every rank applies the same buffer
            assert rel_err(got[0][:-1], whole) <= 1e-5, (R, seed, rel_err(got[0][:-1], whole))
            assert rel_err(got[0][-1], f["loss"]) <= 1e-5, (R, seed)
