"""Hierarchical sampling timings.  python tools/t_hierarchical.py [--min-ms 50] [--compare-tree DIR]

  sampler alone        lnb_sample_pdf at 4096 x (64 -> 128) and 640 000 x (64 -> 192): achieved GB/s against the bytes
                       the rule needs (12 S read + 8 (S + n_fine) written per ray) and the fraction of the copy bandwidth
                       measured in the same run (a 2 GiB device-to-device copy: read + write bytes over its time)
  CoarseFine step      33->30->30->4, 4096 rays, 64 + 64 samples (camera mode)  vs  one plain step at S = 128
  CoarseFine step      90->256x8->4, 4096 rays, 64 + 128 samples (both passes on the wide path)
  frame                800 x 800 coarse-to-fine render (render_frame_device(fine=...)), small nets 64 + 64 and paper
                       nets 64 + 128, against the plain frame at S = 64 + n_fine; the coarse pass with weights runs on the
                       wide path, and its cost is printed beside the fused forward pass of the same coarse net
  C2 trainer step      lnb_trainer_step at C2 (4096 x 64, 33->30->30->4, tensor cores) of this tree and, with
                       --compare-tree, of another built tree, in alternated child processes

CUDA events around >= --min-ms of work after warm-up; the card's name and power limit are printed first.  The 4096-ray
sampler case fits in L2 (9.4 MB); the 640 000-ray one (1.47 GB) does not.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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
    n = 2
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


def scene():
    from loma_nerf_b200 import render
    focal = 0.5 / np.tan(0.5 * 0.6911)
    K = np.array([[focal, 0, 0.5], [0, focal, 0.5], [0, 0, 1]], np.float64)
    return K, [render.pose_spherical(th, -30.0, 4.0) for th in np.linspace(0, 330, 12)]


def c2_child(min_ms):
    """One C2 lnb_trainer_step timing of the library this interpreter imports (printed as JSON)."""
    import torch
    from loma_nerf_b200 import api
    from oracle import oracle as O
    ctx = api.Context(0)
    case = O.make_nerf_case(1, 4096, 64, E=5)
    dims = [int(v) for v in case["dims"]]
    tr = api.Trainer(ctx, dims, case["ws"], case["bs"])
    cv = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()  # noqa: E731
    p = tr.prepare(X=cv(case["X"]), dists=cv(case["dists"]), target=cv(case["target"]), path="tc")
    ms = timed(lambda: tr.step(p), min_ms)
    print(json.dumps(dict(c2_step_ms=ms)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-ms", type=float, default=50.0)
    ap.add_argument("--compare-tree", default=None, help="a second built tree: C2 step timings alternate between the two")
    ap.add_argument("--c2-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.c2_child:   # the library comes from PYTHONPATH (the tree under test), the oracle from this tree
        sys.path.append(ROOT)
        return c2_child(args.min_ms)
    sys.path.insert(0, ROOT)
    import torch
    from loma_nerf_b200 import api, render
    from oracle import oracle as O
    name, power = card()
    print("card: %s, power limit %s" % (name, power))
    ctx = api.Context(0)
    dev = torch.device("cuda", 0)
    res = {}

    # copy bandwidth of this card in this run: the yardstick of the memory-bound sampler
    a = torch.empty(1 << 28, dtype=torch.float64, device=dev)
    b = torch.empty_like(a)
    ms = timed(lambda: b.copy_(a), args.min_ms)
    bw = 2 * a.numel() * 8 / (ms * 1e-3)
    del a, b
    print("device copy: %.2f TB/s (read + write of 2 GiB)" % (bw / 1e12))
    res["copy_tbps"] = bw / 1e12

    rng = np.random.default_rng(0)
    for R, S, n in ((4096, 64, 64), (640000, 64, 128)):
        t = torch.as_tensor(np.sort(rng.uniform(2, 6, (R, S)), axis=1)).to(dev)
        w = torch.as_tensor(rng.uniform(0, 1, (R, S)).astype(np.float32) ** 2).to(dev)
        out = torch.empty((R, S + n), dtype=torch.float64, device=dev)
        for strat in (False, True):
            ms = timed(lambda: ctx.sample_pdf(t, w, n, stratified=strat, out=out), args.min_ms)
            byt = R * (12 * S + 8 * (S + n))
            print("sample_pdf %d x (%d -> %d) %s: %.4f ms, %.0f GB/s, %.1f%% of the copy bandwidth (bound %.4f ms)"
                  % (R, S, S + n, "stratified" if strat else "deterministic", ms, byt / ms / 1e6, 100 * byt / bw / (ms * 1e-3),
                     byt / bw * 1e3))
            res["sample_pdf_%d_%s_ms" % (R, "strat" if strat else "det")] = ms
        del t, w, out

    K, poses = scene()
    W = 800
    R = 4096
    target = torch.as_tensor(rng.uniform(0, 1, (R, 3)).astype(np.float32)).to(dev)
    pix = [torch.as_tensor(rng.choice(W * W, R, replace=False).astype(np.int32)).to(dev) for _ in range(8)]
    cams = [api.make_camera(poses[i % 12], K, W, pixels=pix[i], stratified=True, seed=i) for i in range(8)]

    def run_cycle(fn):
        it = [0]

        def f():
            fn(cams[it[0] % 8])
            it[0] += 1
        return f

    for label, E, E_d, H, L, S, n_fine in (("small 33->30->30->4", 5, None, 30, 3, 64, 64),
                                           ("paper 90->256x8->4", 10, 4, 256, 9, 64, 128)):
        dims = O.mlp_dims(api.rays_input_width(E, E_d), H, L, 4)
        (wc, bc), (wf, bf) = O.init_mlp(rng, dims, 1.0), O.init_mlp(rng, dims, 1.0)
        coarse, fine, plain = api.Trainer(ctx, dims, wc, bc), api.Trainer(ctx, dims, wf, bf), api.Trainer(ctx, dims, wf, bf)
        cf = api.CoarseFine(coarse, fine, n_fine)
        ms_cf = timed(run_cycle(lambda c: cf.step(camera=c, S=S, pe_bands=E, dir_bands=E_d, target=target, path="tc")), args.min_ms)
        ms_pl = timed(run_cycle(lambda c: plain.step(camera=c, S=S + n_fine, pe_bands=E, dir_bands=E_d, target=target,
                                                     path="tc")), args.min_ms)
        print("CoarseFine %s, %d rays, %d + %d: %.3f ms per step; one plain step at S = %d: %.3f ms"
              % (label, R, S, n_fine, ms_cf, S + n_fine, ms_pl))
        res["coarse_fine_%s_ms" % label.split()[0]] = ms_cf
        res["plain_%s_ms" % label.split()[0]] = ms_pl
        for tr in (coarse, fine, plain):
            tr.close()
        # an 800 x 800 frame
        wc_d, bc_d, wf_d, bf_d = (torch.as_tensor(x).to(dev) for x in (wc, bc, wf, bf))
        u8 = torch.empty((W, W, 3), dtype=torch.uint8, device=dev)
        col = torch.empty((W * W, 3), dtype=torch.float32, device=dev)
        per = 1 << 17 if H > 64 else None
        ms_f = timed(lambda: render.render_frame_device(ctx, dims, wc_d, bc_d, W, W, K, poses[1], S, E, out_u8=u8, color=col,
                                                        rays_per_call=per, dir_bands=E_d, fine=(dims, wf_d, bf_d, n_fine)),
                     args.min_ms)
        ms_p = timed(lambda: render.render_frame_device(ctx, dims, wf_d, bf_d, W, W, K, poses[1], S + n_fine, E, out_u8=u8,
                                                        color=col, rays_per_call=per, dir_bands=E_d), args.min_ms)
        wbuf = torch.empty((W * W if per is None else per, S), dtype=torch.float32, device=dev)
        n_c = W * W if per is None else per
        cam0 = api.make_camera(poses[1], K, W, W)
        ms_cw = timed(lambda: ctx.nerf_step_camera(dims, cam0, n_c, S, E, wc_d, bc_d, outputs=("weights",),
                                                   out={"weights": wbuf}, path="tc", dir_bands=E_d), args.min_ms)
        ms_cc = timed(lambda: ctx.nerf_step_camera(dims, cam0, n_c, S, E, wc_d, bc_d, outputs=("color",),
                                                   out={"color": col[:n_c]}, path="tc", dir_bands=E_d), args.min_ms)
        print("frame %s 800x800, %d + %d: %.3f ms coarse-to-fine, %.3f ms plain at S = %d; coarse pass over %d rays: "
              "%.3f ms with weights, %.3f ms colour only" % (label, S, n_fine, ms_f, ms_p, S + n_fine, n_c, ms_cw, ms_cc))
        res["frame_%s_ms" % label.split()[0]] = ms_f
        res["frame_plain_%s_ms" % label.split()[0]] = ms_p
        res["coarse_weights_%s_ms" % label.split()[0]] = ms_cw
        res["coarse_color_%s_ms" % label.split()[0]] = ms_cc

    # lnb_trainer_step at C2: this tree and the other, alternated
    ctx.close()
    trees = [("this", ROOT)] + ([("compare", os.path.abspath(args.compare_tree))] if args.compare_tree else [])
    times = {k: [] for k, _ in trees}
    for _ in range(3):
        for k, tree in (trees if _ % 2 == 0 else trees[::-1]):
            env = dict(os.environ, PYTHONPATH=tree + os.pathsep + ROOT)
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--c2-child", "--min-ms", str(args.min_ms * 4)],
                                 capture_output=True, text=True, env=env, cwd=tree, check=True).stdout
            times[k].append(json.loads(out.strip().splitlines()[-1])["c2_step_ms"])
    for k, v in times.items():
        print("C2 lnb_trainer_step (%s tree): %s ms, median %.4f" % (k, ", ".join("%.4f" % x for x in v), float(np.median(v))))
        res["c2_step_%s_ms" % k] = float(np.median(v))
    print(json.dumps(dict(card=name, power_limit=power, **res)))


if __name__ == "__main__":
    main()
