"""Cost of the view-direction input in camera mode: positions only vs positions + a 4-band direction, on the workloads
the direction form changes.  python tools/t_viewdirs.py [--min-ms 50]

  C2-shaped train step   4096 rays x 64 samples, 33->30->30->4  vs  60->30->30->4   (fused_mg_kernel)
  render frame           800 x 800 x 64, the same two nets, forward only           (fused_v1_kernel)
  C5 train step          4096 rays x 192 samples, 63->256x8->4  vs  90->256x8->4    (wide path: layer 0 padded 64 -> 128)

Each line: the card's name and power limit, then per net the time per step (CUDA events over >= --min-ms after warm-up),
samples/s, rays/s and the algorithmic FLOP rate (2 / 6 FLOP per MAC forward / train: 482 816 MAC per sample for the 90-input
C5 net).  Camera mode reads only a pixel list and the targets per batch; the script still cycles 8 batches (different
pixels and stratified seeds) and 12 poses so that no timed step repeats its predecessor's inputs.  The groups per CTA
the launcher picked for fused_mg_kernel are read off its block size in a separate torch.profiler run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover
        q = "unknown (%s)" % e
    return name, q


def timed(fn, min_ms):
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 4
    while True:
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= min_ms:
            return ms / n, n, ms
        n = max(n * 2, int(n * 1.2 * min_ms / max(ms, 1e-3)))


def mac_per_sample(dims):
    return sum(int(a) * int(b) for a, b in zip(dims[:-1], dims[1:]))


def mg_groups(fn):
    """Threads per block of the fused_mg_kernel launch of fn() / 128, from a torch.profiler trace."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "trace.json")
        prof.export_chrome_trace(p)
        ev = json.load(open(p))
    for e in ev.get("traceEvents", []):
        if "fused_mg_kernel" in str(e.get("name", "")) and "block" in e.get("args", {}):
            return e["args"]["block"][0] // 128
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-ms", type=float, default=50.0)
    args = ap.parse_args()
    import torch
    from loma_nerf_b200 import api, render, synthetic
    name, plimit = card()
    print("card: %s, power limit %s" % (name, plimit), flush=True)
    ctx = api.Context(0)
    dev = torch.device("cuda", 0)
    K = np.array([[synthetic.FOCAL, 0, 0.5], [0, synthetic.FOCAL, 0.5], [0, 0, 1.0]])
    poses = [render.pose_spherical(30.0 * i, -30.0, 4.0) for i in range(12)]
    rng = np.random.default_rng(5)
    results = []

    def report(label, dims, ms, n, tot, R, S, train, extra=""):
        smp = R * S / (ms * 1e-3)
        fl = (6 if train else 2) * mac_per_sample(dims) * smp
        line = ("%-22s in=%-3d %8.3f ms/step (%d steps, %.0f ms)  %7.3f G samples/s  %8.2f M rays/s  %7.1f TFLOP/s%s"
                % (label, dims[0], ms, n, tot, smp * 1e-9, R / (ms * 1e-3) * 1e-6, fl * 1e-12, extra))
        print(line, flush=True)
        results.append(dict(label=label, c_in=dims[0], ms=ms, steps=n, samples_per_s=smp, rays_per_s=R / (ms * 1e-3),
                            tflops=fl * 1e-12, extra=extra))

    def train_case(label, E, width, layers, R, S, E_d):
        c_in = 3 + 6 * E + (0 if E_d is None else 3 + 6 * E_d)
        dims = synthetic.mlp_dims(c_in, width, layers, 4)
        ws, bs = synthetic.init_mlp(np.random.default_rng(216), dims)
        tr = api.Trainer(ctx, dims, ws, bs)
        batches = []
        for k in range(8):
            pix = torch.as_tensor(rng.integers(0, 800 * 800, R).astype(np.int32)).cuda()
            cam = api.make_camera(poses[k], K, 800, 800, near=synthetic.NEAR, far=synthetic.FAR, pixels=pix,
                                  stratified=True, seed=k)
            tgt = torch.rand((R, 3), device=dev)
            batches.append(tr.prepare(camera=cam, S=S, pe_bands=E, dir_bands=E_d, target=tgt, path="tc"))
        it = [0]

        def step():
            tr.step(batches[it[0] % 8])
            it[0] += 1
        groups = mg_groups(step)
        ms, n, tot = timed(step, args.min_ms)
        report(label, dims, ms, n, tot, R, S, True, "" if groups is None else "  fused_mg_kernel groups/CTA %d" % groups)
        tr.close()

    def render_case(E, E_d):
        c_in = 3 + 6 * E + (0 if E_d is None else 3 + 6 * E_d)
        dims = synthetic.mlp_dims(c_in, 30, 3, 4)
        ws_np, bs_np = synthetic.init_mlp(np.random.default_rng(216), dims)
        ws, bs = torch.as_tensor(ws_np).cuda(), torch.as_tensor(bs_np).cuda()
        color = torch.empty((640000, 3), dtype=torch.float32, device=dev)
        u8 = torch.empty((640000, 3), dtype=torch.uint8, device=dev)
        it = [0]

        def frame():
            render.render_frame_device(ctx, dims, ws, bs, 800, 800, K, poses[it[0] % 12], 64, E, near=synthetic.NEAR,
                                       far=synthetic.FAR, out_u8=u8, color=color, dir_bands=E_d)
            it[0] += 1
        ms, n, tot = timed(frame, args.min_ms)
        report("render 800x800x64", dims, ms, n, tot, 640000, 64, False)

    train_case("C2 camera train", 5, 30, 3, 4096, 64, None)
    train_case("C2 camera train", 5, 30, 3, 4096, 64, 4)
    render_case(5, None)
    render_case(5, 4)
    train_case("C5 camera train", 10, 256, 9, 4096, 192, None)
    train_case("C5 camera train", 10, 256, 9, 4096, 192, 4)
    print(json.dumps(dict(card=name, power_limit=plimit, results=results)))
    ctx.close()


if __name__ == "__main__":
    main()
