"""Cost of views mode (lnb_views) and of the on-device draw (lnb_views_draw) on the workloads they touch.
python tools/t_views.py [--min-ms 50] [--rounds 3]

  C2 step          4096 rays x 64 samples, 33->30->30->4, a CUDA graph of 8 trainer steps: camera mode, views mode on one
                   view and on 100 views with a fixed batch, and 8 x (draw + step) on 100 views (all views, and one view
                   per step)
  training loop    a synthetic 100-view 800 x 800 scene: a host-driven camera-mode loop (per step: pick a view, draw pixels,
                   gather the targets, make_camera, step) against replays of a graph of 8 x (draw + step); samples/s
  C5 step          4096 rays x 192 samples, 90->256x8->4 (wide path, 4-band view direction), camera vs views mode

The card's name and power limit are printed first.  Variants of a workload are timed alternately, --rounds times (CUDA
events over >= --min-ms after warm-up each); every line gives the per-round times and the median.
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
    NV, W = 100, 800
    poses = np.stack([render.pose_spherical(360.0 * i / NV, -30.0 + 20.0 * np.sin(i), 4.0) for i in range(NV)])
    images = torch.rand((NV, W, W, 3), device=dev)
    scene = api.Scene(ctx, poses, images, K, near=synthetic.NEAR, far=synthetic.FAR)
    one = api.Scene(ctx, poses[:1], images[:1], K, near=synthetic.NEAR, far=synthetic.FAR)
    rng = np.random.default_rng(5)
    results = []

    def compare(label, fns, unit_samples):
        ts = {k: [] for k in fns}
        for _ in range(args.rounds):
            for k, f in fns.items():
                ts[k].append(timed(f, args.min_ms))
        med = {k: float(np.median(v)) for k, v in ts.items()}
        base = next(iter(med.values()))
        for k in fns:
            print("%-28s %-30s %s ms  median %.4f ms (x%.3f)  %.2f G samples/s"
                  % (label, k, " ".join("%.4f" % v for v in ts[k]), med[k], med[k] / base, unit_samples / (med[k] * 1e-3) * 1e-9),
                  flush=True)
        results.append(dict(label=label, ms=ts, median_ms=med))

    def graph_of(steps):
        for s in steps:
            s()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            ctx.set_stream(torch.cuda.current_stream())
            for s in steps:
                s()
        ctx.set_stream(torch.cuda.current_stream())
        return g.replay

    def c_step(label, E, E_d, width, layers, R, S, graph):
        dims = synthetic.mlp_dims(api.rays_input_width(E, E_d), width, layers, 4)
        ws, bs = synthetic.init_mlp(np.random.default_rng(216), dims)
        trs = []
        kw = dict(S=S, pe_bands=E, dir_bands=E_d, path="tc")
        fns = {}
        # camera mode: 8 prepared batches of 8 poses
        tr = api.Trainer(ctx, dims, ws, bs)
        trs.append(tr)
        cams = []
        for k in range(8):
            pix = torch.as_tensor(rng.integers(0, W * W, R).astype(np.int32)).cuda()
            cam = api.make_camera(poses[k], K, W, W, near=synthetic.NEAR, far=synthetic.FAR, pixels=pix, stratified=True, seed=k)
            cams.append(tr.prepare(camera=cam, target=torch.rand((R, 3), device=dev), **kw))
        steps = [lambda p=p, tr=tr: tr.step(p) for p in cams]
        fns["camera"] = graph_of(steps) if graph else (lambda it=[0]: (steps[it[0] % 8](), it.__setitem__(0, it[0] + 1)))

        def views(sc, draw, one_view=False):
            tr = api.Trainer(ctx, dims, ws, bs)
            trs.append(tr)
            b = sc.batch(R, stratified=True, one_view=one_view, seed=3)
            b.draw()

            def st():
                if draw:
                    b.draw()
                tr.step(views=b, **kw)
            return graph_of([st] * 8) if graph else st
        fns["views, 1 view"] = views(one, False)
        fns["views, 100 views"] = views(scene, False)
        fns["draw + views, 100 views"] = views(scene, True)
        fns["draw + views, one view/step"] = views(scene, True, one_view=True)
        compare(label, fns, (8 if graph else 1) * R * S)
        for tr in trs:
            tr.close()

    c_step("C2 step (graph of 8)", 5, None, 30, 3, 4096, 64, True)

    # ---- a training loop over the 100-view scene
    E, R, S = 5, 4096, 64
    dims = synthetic.mlp_dims(3 + 6 * E, 30, 3, 4)
    ws, bs = synthetic.init_mlp(np.random.default_rng(216), dims)
    tr_h, tr_g = api.Trainer(ctx, dims, ws, bs), api.Trainer(ctx, dims, ws, bs)
    flat = scene.images

    def host_step():
        v = int(rng.integers(0, NV))
        pix = torch.as_tensor(rng.integers(0, W * W, R).astype(np.int32)).to(dev, non_blocking=True)
        tgt = flat[v].index_select(0, pix.long())
        cam = api.make_camera(poses[v], K, W, W, near=synthetic.NEAR, far=synthetic.FAR, pixels=pix, stratified=True,
                              seed=int(rng.integers(0, 2 ** 63)))
        tr_h.step(camera=cam, S=S, pe_bands=E, target=tgt, path="tc")

    b = scene.batch(R, stratified=True, one_view=True, seed=11)

    def dstep():
        b.draw()
        tr_g.step(views=b, S=S, pe_bands=E, path="tc")
    g8 = graph_of([dstep] * 8)
    compare("loop 100 x 800x800", {"host-driven camera (x8)": lambda: [host_step() for _ in range(8)], "graph 8 x (draw + step)": g8},
            8 * R * S)
    tr_h.close()
    tr_g.close()

    c_step("C5 step (E_d = 4)", 10, 4, 256, 9, 4096, 192, False)
    print(json.dumps(dict(card=name, power_limit=plimit, results=results)))
    ctx.close()


if __name__ == "__main__":
    main()
