"""Forward-only full-frame rendering and the hosts' small helpers around it.

The reference's render path is the eval block of train_nerf.py:558-700 (make_nerf_video.py only
stitches ground-truth PNGs, SURVEY.md 0): get_rays for one pose, 4-ray chunks through
nerf_evaluate_and_march, accumulated_color read back, PSNR against the ground truth.  Here a frame is
one call: all H*W rays go to the device in rays mode, colours come back.
"""
import numpy as np


def get_rays(height, width, normalized_K, c2w_pose):
    """Ray origins / directions of every pixel, exactly as train_nerf.py:23-62 builds them
    (normalised pixel grid linspace(0,1,width), directions NOT normalised, float64)."""
    rng = np.linspace(0, 1, width)
    i, j = np.meshgrid(rng, rng, indexing="xy")
    i, j = i.flatten(), j.flatten()
    dirs = np.stack([(i - normalized_K[0, 2]) / normalized_K[0, 0],
                     -(j - normalized_K[1, 2]) / normalized_K[1, 1], -np.ones_like(i)], axis=-1)
    R, T = c2w_pose[:3, :3], c2w_pose[:3, 3]
    return T[None, :].repeat(dirs.shape[0], 0), dirs @ R.T


def compute_psnr(img1, img2, max_val=1.0):
    """train_nerf.py:163-183."""
    mse = np.mean((np.asarray(img1, np.float64) - np.asarray(img2, np.float64)) ** 2)
    with np.errstate(divide="ignore"):      # identical images: +inf, as the reference's expression gives
        return 20 * np.log10(max_val / np.sqrt(mse))


def render_rays(ctx, dims, ws, bs, rays_o, rays_d, t, pe_bands, path="tc", rays_per_call=1 << 18, dir_bands=None,
                background=None):
    """Colours [R][3] (numpy float32) of R rays; rays_o/rays_d [R][3] and t [R][S] numpy (float64 as
    the reference makes them, or float32).  Host buffers in, host buffer out, chunked so the device
    staging stays bounded.  dir_bands: the net also takes the view direction (Context.nerf_step_rays).
    background=(r, g, b): composited onto that colour (e.g. (1, 1, 1) for a net trained on white)."""
    R = rays_o.shape[0]
    out = np.empty((R, 3), np.float32)
    ws = np.ascontiguousarray(ws, np.float32)
    bs = np.ascontiguousarray(bs, np.float32)
    for r0 in range(0, R, rays_per_call):
        r1 = min(R, r0 + rays_per_call)
        res = ctx.nerf_step_rays(dims, np.ascontiguousarray(rays_o[r0:r1]), np.ascontiguousarray(rays_d[r0:r1]),
                                 np.ascontiguousarray(t[r0:r1]), pe_bands, ws, bs, target=None, grad=False,
                                 outputs=("color",), path=path, dir_bands=dir_bands, background=background)
        out[r0:r1] = res["color"]
    return out


def render_frame(ctx, dims, ws, bs, height, width, normalized_K, c2w_pose, n_samples, pe_bands, near=2.0, far=6.0,
                 path="tc", dir_bands=None, fine=None, background=None):
    """One H x W frame: t = linspace(near, far, S) for every ray (train_nerf.py:589-605).  fine=(dims_f, ws_f, bs_f,
    n_fine): hierarchical sampling, the frame render_frame_device(fine=...) makes, as float colours.  background as in
    render_rays."""
    if fine is not None:
        import torch
        dev = torch.device("cuda", ctx.device)
        cv = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).to(dev)  # noqa: E731
        color = torch.empty((height * width, 3), dtype=torch.float32, device=dev)
        dims_f, ws_f, bs_f, n_fine = fine
        render_frame_device(ctx, dims, cv(ws), cv(bs), height, width, normalized_K, c2w_pose, n_samples, pe_bands, near=near,
                            far=far, path=path, color=color, dir_bands=dir_bands, fine=(dims_f, cv(ws_f), cv(bs_f), n_fine),
                            background=background)
        ctx.order_torch_after()
        return color.cpu().numpy().reshape(height, width, 3)
    o, d = get_rays(height, width, normalized_K, c2w_pose)
    t = np.broadcast_to(np.linspace(near, far, n_samples)[None, :], (o.shape[0], n_samples))
    return render_rays(ctx, dims, ws, bs, o, d, np.ascontiguousarray(t), pe_bands, path=path,
                       dir_bands=dir_bands, background=background).reshape(height, width, 3)


def render_frame_device(ctx, dims, ws_dev, bs_dev, height, width, normalized_K, c2w_pose, n_samples, pe_bands, near=2.0, far=6.0,
                        path="tc", out_u8=None, color=None, rays_per_call=None, dir_bands=None, fine=None, background=None,
                        acc=None, depth=None):
    """One frame with NOTHING per ray crossing the bus: the pose goes in (camera mode: rays and the linspace depths of
    train_nerf.py:589-605 are generated inside the kernels), a uint8 H x W x 3 frame (torch cuda tensor) comes out.
    ws_dev / bs_dev are cuda tensors in the padded layout.
    fine=(dims_f, ws_f, bs_f, n_fine) renders with hierarchical sampling: per chunk of rays, the camera's rays and S
    coarse depths (lnb_camera_rays), a forward-only coarse pass for the compositing weights, a deterministic sample_pdf
    of n_fine more depths, and the fine net's colour at all S + n_fine of them (rays mode).
    background=(r, g, b) composites the colour onto that background; acc= / depth= ([H*W] float32 CUDA tensors) receive
    the opacity and the expected-depth maps (sum of w_s, sum of w_s t_s), filled chunk by chunk in the same kernels as
    the colour (under fine=, from the fine pass)."""
    import torch
    from . import api
    n = height * width
    dev = ws_dev.device
    color = torch.empty((n, 3), dtype=torch.float32, device=dev) if color is None else color
    step = n if rays_per_call is None else int(rays_per_call)
    for name, m in (("acc", acc), ("depth", depth)):
        if m is not None and not (api._is_cuda(m) and m.dtype == torch.float32 and m.is_contiguous() and tuple(m.shape) == (n,)):
            raise ValueError("%s must be a contiguous [%d] float32 CUDA tensor" % (name, n))

    def maps(r0, r1):   # the colour and whichever maps were asked for, for rays r0 .. r1
        outs, bufs = ("color",), {"color": color[r0:r1]}
        for name, m in (("acc", acc), ("depth", depth)):
            if m is not None:
                outs, bufs[name] = outs + (name,), m[r0:r1]
        return outs, bufs
    if fine is not None:
        dims_f, ws_f, bs_f, n_fine = fine
        m = min(step, n)
        f64 = dict(dtype=torch.float64, device=dev)
        o, d, t = torch.empty((m, 3), **f64), torch.empty((m, 3), **f64), torch.empty((m, n_samples), **f64)
        w = torch.empty((m, n_samples), dtype=torch.float32, device=dev)
        t_fine = torch.empty((m, n_samples + int(n_fine)), **f64)
    for r0 in range(0, n, step):
        r1 = min(n, r0 + step)
        cam = api.make_camera(c2w_pose, normalized_K, width, height, near=near, far=far, first_pixel=r0)
        outs, bufs = maps(r0, r1)
        if fine is None:
            ctx.nerf_step_camera(dims, cam, r1 - r0, n_samples, pe_bands, ws_dev, bs_dev, target=None, grad=False,
                                 outputs=outs, out=bufs, path=path, dir_bands=dir_bands, background=background)
            continue
        k = r1 - r0
        ck, dk, tk, wk, tfk = o[:k], d[:k], t[:k], w[:k], t_fine[:k]
        ctx.camera_rays(cam, k, n_samples, out=(ck, dk, tk))
        ctx.nerf_step_camera(dims, cam, k, n_samples, pe_bands, ws_dev, bs_dev, target=None, grad=False,
                             outputs=("weights",), out={"weights": wk}, path=path, dir_bands=dir_bands)
        ctx.sample_pdf(tk, wk, n_fine, stratified=False, ray0=r0, out=tfk)
        ctx.nerf_step_rays(dims_f, ck, dk, tfk, pe_bands, ws_f, bs_f, target=None, grad=False, outputs=outs,
                           out=bufs, path=path, dir_bands=dir_bands, background=background)
    return ctx.color_to_u8(color, out_u8).reshape(height, width, 3)


def save_weights(prefix, ws_padded, bs_padded):
    """The padded (L,max_in,max_out) / (L,max_out) float32 arrays as models/weights.npy /
    models/biases.npy hold them (the save the reference has commented out, train_nerf.py:559-564)."""
    np.save(prefix + "weights.npy", np.ascontiguousarray(ws_padded, np.float32))
    np.save(prefix + "biases.npy", np.ascontiguousarray(bs_padded, np.float32))


def load_weights(prefix):
    ws, bs = np.load(prefix + "weights.npy"), np.load(prefix + "biases.npy")
    if ws.ndim != 3 or bs.ndim != 2 or ws.shape[0] != bs.shape[0] or ws.shape[2] != bs.shape[1]:
        raise ValueError("not a padded (L,max_in,max_out) / (L,max_out) weight pair")
    return ws.astype(np.float32), bs.astype(np.float32)


def pose_spherical(theta_deg, phi_deg, radius):
    """Camera-to-world matrix of a camera on a sphere around the origin looking at it (the orbit the Blender scenes'
    test poses follow, transforms_test.json; -z is the viewing direction as in get_rays above)."""
    th, ph = np.deg2rad(theta_deg), np.deg2rad(phi_deg)
    trans = np.eye(4); trans[2, 3] = radius
    rot_phi = np.array([[1, 0, 0, 0], [0, np.cos(ph), -np.sin(ph), 0], [0, np.sin(ph), np.cos(ph), 0], [0, 0, 0, 1.0]])
    rot_th = np.array([[np.cos(th), 0, -np.sin(th), 0], [0, 1, 0, 0], [np.sin(th), 0, np.cos(th), 0], [0, 0, 0, 1.0]])
    flip = np.array([[-1, 0, 0, 0], [0, 0, 1, 0], [0, 1, 0, 0], [0, 0, 0, 1.0]])
    return flip @ rot_th @ rot_phi @ trans


def write_mjpeg_avi(path, frames, fps=30, quality=90):
    """Motion-JPEG in an AVI container (RIFF: hdrl with avih / strh / strf, movi of '00dc' chunks, idx1), written with PIL
    alone: the video a stock Python can produce without ffmpeg / imageio (the hosts' make_nerf_video.py:21-38 asks imageio
    for an mp4).  frames: uint8 [F][H][W][3]."""
    import io
    import struct
    from PIL import Image
    frames = np.asarray(frames, np.uint8)
    n, h, w = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
    jpgs = []
    for f in frames:
        b = io.BytesIO()
        Image.fromarray(f).save(b, format="JPEG", quality=quality)
        jpgs.append(b.getvalue())

    def chunk(tag, data):
        return tag + struct.pack("<I", len(data)) + data + (b"\0" if len(data) & 1 else b"")

    def lst(tag, data):
        return b"LIST" + struct.pack("<I", len(data) + 4) + tag + data

    biggest = max((len(j) for j in jpgs), default=0)
    avih = struct.pack("<IIIIIIIIII4I", int(1e6 / fps), biggest * fps, 0, 0x10, n, 0, 1, biggest, w, h, 0, 0, 0, 0)
    strh = struct.pack("<4s4sIHHIIIIIIIIhhhh", b"vids", b"MJPG", 0, 0, 0, 0, 1, fps, 0, n, biggest, 0xFFFFFFFF, 0, 0, 0, w, h)
    strf = struct.pack("<IiiHH4sIiiII", 40, w, h, 1, 24, b"MJPG", w * h * 3, 0, 0, 0, 0)
    hdrl = lst(b"hdrl", chunk(b"avih", avih) + lst(b"strl", chunk(b"strh", strh) + chunk(b"strf", strf)))
    movi, idx, off = b"", b"", 4
    for j in jpgs:
        c = chunk(b"00dc", j)
        idx += struct.pack("<4sIII", b"00dc", 0x10, off, len(j))
        movi += c
        off += len(c)
    body = b"AVI " + hdrl + lst(b"movi", movi) + chunk(b"idx1", idx)
    with open(path, "wb") as fh:
        fh.write(b"RIFF" + struct.pack("<I", len(body)) + body)
    return path


def render_video(ctx, dims, ws, bs, height, width, normalized_K, poses, n_samples, pe_bands, out_dir=None, near=2.0, far=6.0,
                 path="tc", ground_truth=None, fps=30, frame_fn=None, dir_bands=None, fine=None, background=None):
    """What make_nerf_video.py is named for but does not do (it stitches ground-truth PNGs): render one frame per
    camera pose with the trained weights, optionally score each against its ground-truth image
    (train_nerf.py:163-183) and write frame_%04d.png, an animated orbit.gif and a Motion-JPEG orbit.avi into out_dir (PIL
    only; an mp4 needs imageio/ffmpeg, which the hosts' environment may not have).  Returns (frames uint8 [F][H][W][3],
    psnr list | None).
    frame_fn(i, pose) -> float image may replace the device render (tests of the host side).  fine: hierarchical
    sampling and background, as in render_frame."""
    frames, psnr = [], ([] if ground_truth is not None else None)
    for i, pose in enumerate(poses):
        img = frame_fn(i, pose) if frame_fn else render_frame(ctx, dims, ws, bs, height, width, normalized_K, np.asarray(pose, np.float64),
                                                            n_samples, pe_bands, near=near, far=far, path=path,
                                                            dir_bands=dir_bands, fine=fine, background=background)
        img = np.clip(np.asarray(img, np.float32), 0.0, 1.0)
        if ground_truth is not None:
            psnr.append(float(compute_psnr(img, ground_truth[i])))
        frames.append((img * 255.0 + 0.5).astype(np.uint8))
    frames = np.stack(frames) if frames else np.zeros((0, height, width, 3), np.uint8)
    if out_dir is not None and len(frames):
        import os
        from PIL import Image
        os.makedirs(out_dir, exist_ok=True)
        pil = [Image.fromarray(f) for f in frames]
        for i, im in enumerate(pil):
            im.save(os.path.join(out_dir, "frame_%04d.png" % i))
        pil[0].save(os.path.join(out_dir, "orbit.gif"), save_all=True, append_images=pil[1:], duration=max(1, int(1000 / fps)), loop=0)
        write_mjpeg_avi(os.path.join(out_dir, "orbit.avi"), frames, fps=fps)
    return frames, psnr
