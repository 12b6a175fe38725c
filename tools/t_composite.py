"""Cost of the compositing extras (lnb_composite: acc / depth maps, background colour) on the workloads they touch.
python tools/t_composite.py [--min-ms 50] [--rounds 3]

  render frame        800 x 800 x 64 camera mode, 33->30->30->4 (C4's render net), plain vs acc + depth + white
                      background, and the same with a 4-band view direction (60->30->30->4)   (fused_v1_kernel)
  C2 camera train     4096 rays x 64 samples through the Trainer, a CUDA graph of 8 steps, without vs with a white
                      background (fused_mg_kernel: plain vs the extras instantiation)
  C5 camera train     4096 rays x 192 samples, 63->256x8->4 (wide path), without vs with a background

The card's name and power limit are printed first.  Each workload's two variants are timed alternately, --rounds times
(CUDA events over >= --min-ms after warm-up each); every line gives the per-round times and the median ratio.
"""
import argparse
import json
import os
import subprocess
import sys

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
            return ms / n
        n = max(n * 2, int(n * 1.2 * min_ms / max(ms, 1e-3)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-ms", type=float, default=50.0)
    ap.add_argument("--rounds", type=int, default=3)
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
    white = (1.0, 1.0, 1.0)

    def compare(label, a, b, unit_rays):
        ta, tb = [], []
        for _ in range(args.rounds):
            ta.append(timed(a, args.min_ms))
            tb.append(timed(b, args.min_ms))
        ma, mb = float(np.median(ta)), float(np.median(tb))
        line = ("%-34s plain %s ms  extras %s ms  median %.4f -> %.4f ms (x%.3f)  %.1f -> %.1f M rays/s"
                % (label, " ".join("%.4f" % v for v in ta), " ".join("%.4f" % v for v in tb), ma, mb, mb / ma,
                   unit_rays / (ma * 1e-3) * 1e-6, unit_rays / (mb * 1e-3) * 1e-6))
        print(line, flush=True)
        results.append(dict(label=label, plain_ms=ta, extras_ms=tb, ratio=mb / ma))

    # ---- render 800 x 800 x 64
    for E_d in (None, 4):
        dims = synthetic.mlp_dims(33 + (0 if E_d is None else 3 + 6 * E_d), 30, 3, 4)
        ws_np, bs_np = synthetic.init_mlp(np.random.default_rng(216), dims)
        ws, bs = torch.as_tensor(ws_np).cuda(), torch.as_tensor(bs_np).cuda()
        color = torch.empty((640000, 3), dtype=torch.float32, device=dev)
        u8 = torch.empty((640000, 3), dtype=torch.uint8, device=dev)
        acc, depth = torch.empty(640000, device=dev), torch.empty(640000, device=dev)
        it = [0]

        def frame(extras):
            kw = dict(background=white, acc=acc, depth=depth) if extras else {}
            render.render_frame_device(ctx, dims, ws, bs, 800, 800, K, poses[it[0] % 12], 64, 5, near=synthetic.NEAR,
                                       far=synthetic.FAR, out_u8=u8, color=color, dir_bands=E_d, **kw)
            it[0] += 1
        compare("render 800x800x64 in=%d" % dims[0], lambda: frame(False), lambda: frame(True), 640000)

    # ---- train steps through the Trainer
    def train(label, E, width, layers, R, S, graph):
        dims = synthetic.mlp_dims(3 + 6 * E, width, layers, 4)
        ws, bs = synthetic.init_mlp(np.random.default_rng(216), dims)
        trs = {False: api.Trainer(ctx, dims, ws, bs), True: api.Trainer(ctx, dims, ws, bs, background=white)}
        batches = {}
        for bg, tr in trs.items():
            batches[bg] = []
            for k in range(8):
                pix = torch.as_tensor(rng.integers(0, 800 * 800, R).astype(np.int32)).cuda()
                cam = api.make_camera(poses[k], K, 800, 800, near=synthetic.NEAR, far=synthetic.FAR, pixels=pix,
                                      stratified=True, seed=k)
                tgt = torch.rand((R, 3), device=dev)
                batches[bg].append(tr.prepare(camera=cam, S=S, pe_bands=E, target=tgt, path="tc"))
        fns = {}
        for bg, tr in trs.items():
            if graph:
                for p in batches[bg]:
                    tr.step(p)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    ctx.set_stream(torch.cuda.current_stream())
                    for p in batches[bg]:
                        tr.step(p)
                ctx.set_stream(torch.cuda.current_stream())
                fns[bg] = g.replay
            else:
                it = [0]

                def step(tr=tr, bl=batches[bg], it=it):
                    tr.step(bl[it[0] % 8])
                    it[0] += 1
                fns[bg] = step
        n = 8 if graph else 1
        compare(label, fns[False], fns[True], n * R)
        for tr in trs.values():
            tr.close()

    train("C2 camera train (graph of 8 steps)", 5, 30, 3, 4096, 64, True)
    train("C5 camera train", 10, 256, 9, 4096, 192, False)
    print(json.dumps(dict(card=name, power_limit=plimit, results=results)))
    ctx.close()


if __name__ == "__main__":
    main()
