"""Host-side mirror of the flat API of libloma_nerf_b200.so.

`Context.nerf_step` / `Context.fit_step` evaluate the reference's two loma programs
(/root/reference/scripts/nerf.py:1-306, scripts/mlp_fit.py:1-174) on the GPU: MLP forward,
compositing / loss, and (grad=True) the reverse-mode gradients, with the reference's buffer
layouts (padded weights [L][max_in][max_out], features [N][C_in], dists [R][S] ...).

Inputs are either all torch CUDA tensors (device pointers, asynchronous on the context's stream)
or all numpy / CPU tensors (host pointers: staged through pinned memory, synchronous).  PyTorch is
only used as the owner of device memory; the arithmetic is in the CUDA library.
"""
import ctypes

import numpy as np

from . import _lib as L

try:  # torch is plumbing (device memory / streams); the host-pointer path works without it
    import torch
except Exception:  # pragma: no cover
    torch = None

FWD_OUTPUTS = ("inter", "rgba", "alpha", "cumprod", "weights", "color", "loss")
GRAD_OUTPUTS = ("d_ws", "d_bs", "d_X", "d_target", "d_dists", "d_color", "d_inter")
COMPOSITE_OUTPUTS = ("acc", "depth")   # [R] float32, through lnb_composite


def make_composite(background=None):
    """An lnb_composite: background=None (the reference's compositing) or 3 finite floats.  acc / depth are set by the
    caller."""
    c = L.LnbComposite()
    if background is not None:
        bg = [float(v) for v in np.asarray(background, np.float64).reshape(-1)]
        if len(bg) != 3 or not all(np.isfinite(bg)):
            raise ValueError("background must be 3 finite floats, got %r" % (background,))
        c.background = 1
        for i in range(3):
            c.bg[i] = bg[i]
    return c
PATHS = {"f32": L.PATH_F32, "tc": L.PATH_TC, "f32_layerwise": L.PATH_F32_LAYERWISE}


class LnbError(RuntimeError):
    pass


def make_camera(c2w, normalized_K, width, height=None, near=2.0, far=6.0, first_pixel=0, pixels=None, stratified=False, seed=0):
    """lnb_camera from what the reference hosts hold: the 4x4 (or 3x4) camera-to-world pose and the normalised intrinsics
    K = [[f, 0, .5], [0, f, .5], [0, 0, 1]] (train_nerf.py:265-271), near / far (train_nerf.py:201-202).  `pixels` (int32
    array, on the device for device calls) picks arbitrary pixels; otherwise ray r is pixel first_pixel + r."""
    c = L.LnbCamera()
    m = np.asarray(c2w, np.float64)[:3, :4]
    for i in range(12):
        c.c2w[i] = float(m.flat[i])
    K = np.asarray(normalized_K, np.float64)
    c.fx, c.fy, c.cx, c.cy = float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])
    c.width, c.height = int(width), int(width if height is None else height)
    c.first_pixel, c.near, c.far = int(first_pixel), float(near), float(far)
    c.stratified, c.seed = int(bool(stratified)), int(seed) & 0xFFFFFFFFFFFFFFFF
    if pixels is not None:
        assert str(pixels.dtype).endswith("int32")
        c.pixels = pixels.data_ptr() if torch is not None and isinstance(pixels, torch.Tensor) else pixels.ctypes.data
        c._keep = pixels
    return c


def rays_input_width(pe_bands, dir_bands=None):
    """dims[0] of a net fed in rays or camera mode: 3 + 6E for positions only, (3 + 6E) + (3 + 6E_d) with the view
    direction encoded in E_d = dir_bands bands (include/loma_nerf_b200.h, lnb_step_args.pe_bands)."""
    E = int(pe_bands)
    if E < 0 or (dir_bands is not None and int(dir_bands) < 0):
        raise ValueError("pe_bands and dir_bands must be >= 0")
    return 3 + 6 * E + (0 if dir_bands is None else 3 + 6 * int(dir_bands))


def check_rays_width(dims0, pe_bands, dir_bands=None):
    """ValueError unless dims[0] is the input width of (pe_bands, dir_bands): the library reads the input form off dims[0]
    alone, so the caller states it and a net of the other form is refused before anything is launched."""
    want = rays_input_width(pe_bands, dir_bands)
    if int(dims0) != want:
        form = "positions only" if dir_bands is None else "positions and %d direction bands" % int(dir_bands)
        raise ValueError("dims[0] = %d, but %d position bands with %s need %d inputs%s"
                         % (int(dims0), int(pe_bands), form, want,
                            " (pass dir_bands for a net with view directions)" if dir_bands is None else ""))


def make_mlp(dims, ws_shape, head):
    m = L.LnbMlp()
    dims = [int(d) for d in dims]
    if len(dims) - 1 > L.LNB_MAX_LAYERS:
        raise ValueError("too many layers")
    m.n_layers = len(dims) - 1
    for i, d in enumerate(dims):
        m.dims[i] = d
    m.max_in, m.max_out = int(ws_shape[1]), int(ws_shape[2])
    m.head = head
    return m


def _is_cuda(x):
    return torch is not None and isinstance(x, torch.Tensor) and x.is_cuda


def _ptr(x):
    if x is None:
        return None
    if torch is not None and isinstance(x, torch.Tensor):
        assert x.is_contiguous() and x.dtype in (torch.float32, torch.float64), (x.dtype, x.is_contiguous())
        return x.data_ptr()
    assert x.flags.c_contiguous
    return x.ctypes.data


class Context:
    """One lnb_ctx: a device, a stream and a grow-only workspace.

    Stream rule: the library launches on ONE stream per context.  With torch importable that stream
    defaults to torch's current stream of the device at construction time, so torch-side work on the
    tensors passed in (zero fills, NCCL collectives, allocator reuse) is ordered with the library's
    kernels without further ado.  `set_stream` moves it; buffers this class allocates are then
    filled on that stream, and caller tensors are recorded on it (`Tensor.record_stream`) so the
    caching allocator does not hand their memory out while a kernel still reads it."""

    def __init__(self, device=None, stream=None):
        self.lib = L.load()
        if self.lib.lnb_device_count() <= 0:
            raise LnbError("no CUDA device: libloma_nerf_b200 has no CPU fallback")
        if device is None:
            device = torch.cuda.current_device() if torch is not None and torch.cuda.is_available() else 0
        self.device = int(device)
        h = ctypes.c_void_p()
        rc = self.lib.lnb_create(ctypes.byref(h), self.device)
        if rc != L.LNB_OK:
            raise LnbError("lnb_create failed (%d)" % rc)
        self.h = h
        self._stream_raw = None          # None: the context's own non-blocking stream
        if stream is not None:
            self.set_stream(stream)
        elif torch is not None and torch.cuda.is_available():
            self.use_current_torch_stream()

    def close(self):
        if getattr(self, "h", None):
            self.lib.lnb_destroy(self.h)
            self.h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, stream):
        """stream: a torch.cuda.Stream, a raw cudaStream_t int (0 = the legacy default stream), or
        None (the context's own non-blocking stream)."""
        raw = ctypes.c_void_p(-1) if stream is None else ctypes.c_void_p(getattr(stream, "cuda_stream", stream))
        self._check(self.lib.lnb_set_stream(self.h, raw))
        self._stream_raw = None if stream is None else int(getattr(stream, "cuda_stream", stream))

    def torch_stream(self):
        """The context's stream as a torch stream object (for events / wait_stream), or None when the
        context runs on its own private stream (which torch cannot see: synchronize() orders it)."""
        if torch is None or self._stream_raw is None:
            return None
        cur = torch.cuda.current_stream(self.device)
        if cur.cuda_stream == self._stream_raw:
            return cur
        return torch.cuda.ExternalStream(self._stream_raw, device=torch.device("cuda", self.device))

    def _on_torch_current(self):
        return torch is not None and self._stream_raw is not None and \
            torch.cuda.current_stream(self.device).cuda_stream == self._stream_raw

    def order_after_torch(self):
        """Make the context's stream wait for everything queued on torch's current stream so far."""
        if torch is None or self._on_torch_current():
            return
        ts = self.torch_stream()
        if ts is None:                      # private stream: the only ordering tool is the host
            torch.cuda.current_stream(self.device).synchronize()
        else:
            ts.wait_stream(torch.cuda.current_stream(self.device))

    def order_torch_after(self):
        """Make torch's current stream wait for everything the context has launched so far."""
        if torch is None or self._on_torch_current():
            return
        ts = self.torch_stream()
        if ts is None:
            self.synchronize()
        else:
            torch.cuda.current_stream(self.device).wait_stream(ts)

    def _hold(self, *tensors):
        """Caller tensors read by kernels on a stream that is not torch's current one."""
        if torch is None or self._on_torch_current():
            return
        ts = self.torch_stream()
        for x in tensors:
            if ts is not None and _is_cuda(x):
                x.record_stream(ts)

    def use_current_torch_stream(self):
        self.set_stream(torch.cuda.current_stream(self.device))

    def synchronize(self):
        self._check(self.lib.lnb_synchronize(self.h))

    @property
    def launches(self):
        return int(self.lib.lnb_launch_count(self.h))

    def profile_dominant(self, fn):
        """Run fn() with CUDA events around every launch of the dominant (fused) kernel.
        Returns dict(kernel, launches, ms_per_launch) or None when that kernel never ran."""
        self._check(self.lib.lnb_profile(self.h, 1))
        try:
            fn()
            ms, n = ctypes.c_double(), ctypes.c_longlong()
            name = ctypes.create_string_buffer(128)
            self._check(self.lib.lnb_profile_read(self.h, ctypes.byref(ms), ctypes.byref(n), name, 128))
        finally:
            self.lib.lnb_profile(self.h, 0)
        if n.value == 0:
            return None
        return dict(kernel=name.value.decode(), launches=int(n.value), ms_per_launch=ms.value / n.value)

    def _check(self, rc):
        if rc != L.LNB_OK:
            raise LnbError("libloma_nerf_b200 error %d: %s" % (rc, self.lib.lnb_last_error(self.h).decode()))

    # -------------------------------------------------------------------------------------------
    def _step(self, nerf, dims, X, ws, bs, target, dists, R, S, grad, seed, outputs, out, rows,
              path, inter_accumulate, color_accumulate, head, rays=None, pe_bands=0, camera=None, dir_bands=None,
              background=None, views=None):
        if rays is not None or camera is not None or views is not None:
            check_rays_width(dims[0], pe_bands, dir_bands)
        outputs = tuple(outputs)
        extras = [k for k in COMPOSITE_OUTPUTS if k in outputs]
        if (extras or background is not None) and not nerf:
            raise ValueError("background, acc and depth are nerf-step features")
        if "depth" in extras and rays is None and camera is None and views is None:
            raise ValueError("the depth map needs rays or camera mode: features mode has no sample depths")
        comp = make_composite(background) if (background is not None or extras) else None
        dev = _is_cuda(ws)
        mlp = make_mlp(dims, ws.shape, head)
        Ln, mi, mo = mlp.n_layers, mlp.max_in, mlp.max_out
        N = int(X.shape[0]) if X is not None else int(R) * int(S)
        M = max(int(rows or 0), N)
        Wt = int(target.shape[1]) if target is not None else 3
        a = L.LnbStepArgs()
        a.R, a.S, a.n_rows, a.rows, a.target_w = int(R), int(S), N, M, Wt
        a.X, a.ws, a.bs = _ptr(X), _ptr(ws), _ptr(bs)
        a.target, a.dists = _ptr(target), _ptr(dists)
        if rays is not None:
            ro, rd, tv = rays
            f64 = str(ro.dtype).endswith("float64")
            assert str(rd.dtype) == str(ro.dtype) == str(tv.dtype), "rays_o, rays_d, t must share one dtype"
            assert tuple(ro.shape) == (R, 3) and tuple(rd.shape) == (R, 3) and tuple(tv.shape) == (R, S)
            a.rays_o, a.rays_d, a.t = _ptr(ro), _ptr(rd), _ptr(tv)
            a.ray_dtype, a.pe_bands = (L.RAY_F64 if f64 else L.RAY_F32), int(pe_bands)
        if camera is not None:
            a.cam, a.pe_bands = ctypes.pointer(camera), int(pe_bands)
        if views is not None:
            if not dev:
                raise ValueError("a views step takes device buffers (the scene lives on the device)")
            a.pe_bands = int(pe_bands)
        a.inter_rows, a.inter_ld = M, mo
        a.inter_accumulate, a.color_accumulate = int(inter_accumulate), int(color_accumulate)
        a.want_grad = int(bool(grad))
        if isinstance(seed, str):
            assert seed == "loss"
            a.seed_mode, a.seed = L.SEED_LOSS, 1.0
        else:
            a.seed_mode, a.seed = L.SEED_VALUE, float(seed)
        a.path = PATHS[path]
        shapes = dict(inter=(Ln, M, mo), rgba=(R, S, 4), alpha=(R, S), cumprod=(R, S),
                      weights=(R, S), color=(R, 3), loss=(1,), d_ws=(Ln, mi, mo), d_bs=(Ln, mo),
                      d_X=(N, int(dims[0])), d_target=(R, Wt), d_dists=(R, S),
                      d_color=(R, Wt), d_inter=(Ln, M, mo))
        res = {}
        out = out or {}
        want = [k for k in outputs if k not in COMPOSITE_OUTPUTS]
        if grad:
            want += [k for k in ("d_ws", "d_bs") if k not in want]
        for k in want:
            if k not in shapes:
                raise ValueError("unknown output " + k)
            if not nerf and k in ("rgba", "alpha", "cumprod", "weights", "color", "d_dists"):
                continue
            buf = out.get(k)
            if buf is None:
                if dev:
                    buf = torch.zeros(shapes[k], dtype=torch.float32, device=ws.device)
                else:
                    buf = np.zeros(shapes[k], np.float32)
            else:
                assert tuple(buf.shape) == tuple(shapes[k]), (k, tuple(buf.shape), shapes[k])
            res[k] = buf
            setattr(a, k, _ptr(buf))
        for k in extras:   # acc / depth [R]: through the lnb_composite extras
            buf = out.get(k)
            if buf is None:
                buf = torch.zeros((int(R),), dtype=torch.float32, device=ws.device) if dev else np.zeros((int(R),), np.float32)
            else:
                assert tuple(buf.shape) == (int(R),), (k, tuple(buf.shape), (int(R),))
            res[k] = buf
            setattr(comp, k, _ptr(buf))
        if dev:
            # the zero fills above and whatever produced the inputs ran on torch's current stream
            self.order_after_torch()
            self._hold(X, ws, bs, target, dists, *(rays or ()), *res.values())
        if views is not None:
            self._check(self.lib.lnb_nerf_step_views(self.h, ctypes.byref(mlp), ctypes.byref(a), ctypes.byref(views),
                                                     ctypes.byref(comp) if comp is not None else None))
            return res
        if comp is not None:   # only a step that uses an extra calls the composite entry
            fn = self.lib.lnb_nerf_step_composite if dev else self.lib.lnb_nerf_step_composite_host
            self._check(fn(self.h, ctypes.byref(mlp), ctypes.byref(a), ctypes.byref(comp)))
            return res
        fn = {(True, True): self.lib.lnb_nerf_step, (True, False): self.lib.lnb_nerf_step_host,
              (False, True): self.lib.lnb_fit_step, (False, False): self.lib.lnb_fit_step_host}[(nerf, dev)]
        self._check(fn(self.h, ctypes.byref(mlp), ctypes.byref(a)))
        return res

    def nerf_step(self, dims, X, ws, bs, dists, target=None, R=None, S=None, grad=False, seed=1.0,
                  outputs=("color", "loss"), out=None, rows=None, path="f32",
                  inter_accumulate=False, color_accumulate=False, background=None):
        """MLP -> compositing -> SSE loss [-> gradients] (scripts/nerf.py:67-306).
        X [R*S][C_in] features, dists [R][S], target [R][3]; returns {name: buffer}.  Gradient
        outputs ACCUMULATE into buffers passed through `out` (the reference's += semantics).
        background=(r, g, b) composites onto that colour (colour += (1 - acc) bg; the loss and the gradients follow);
        outputs may also name "acc" ([R] opacity, sum of the compositing weights) and, in rays / camera mode, "depth"
        ([R] sum of weight x sample depth).  See lnb_composite in include/loma_nerf_b200.h."""
        R = int(dists.shape[0]) if R is None else R
        S = int(dists.shape[1]) if S is None else S
        return self._step(True, dims, X, ws, bs, target, dists, R, S, grad, seed, outputs, out,
                          rows, path, inter_accumulate, color_accumulate, L.HEAD_NERF, background=background)

    def nerf_step_rays(self, dims, rays_o, rays_d, t, pe_bands, ws, bs, target=None, grad=False, seed=1.0,
                       outputs=("color", "loss"), out=None, path="f32", dir_bands=None, background=None):
        """The same step starting from rays: the sample positions o + d*t, their positional encoding
        and the dists are computed on the device (train_nerf.py:289-311, pos_encoding.py:38-70) --
        fused into the first layer on the tensor-core path.  rays_o, rays_d [R][3], t [R][S], all
        float64 (the reference's dtype) or all float32.  dir_bands=E_d: the net also takes the unit view
        direction in E_d bands (dims[0] = 3 + 6 pe_bands + 3 + 6 E_d, rays_input_width).  background and the "acc" /
        "depth" outputs as in nerf_step (depth = sum of w_s t_s)."""
        R, S = int(t.shape[0]), int(t.shape[1])
        return self._step(True, dims, None, ws, bs, target, None, R, S, grad, seed, outputs, out, None, path,
                          False, False, L.HEAD_NERF, rays=(rays_o, rays_d, t), pe_bands=pe_bands, dir_bands=dir_bands,
                          background=background)

    def nerf_step_camera(self, dims, camera, R, S, pe_bands, ws, bs, target=None, grad=False, seed=1.0,
                         outputs=("color", "loss"), out=None, path="f32", dir_bands=None, background=None):
        """The same step with rays AND sample depths generated on the device from a pose (`make_camera`): the
        device-side get_rays (train_nerf.py:23-62) and linspace / stratified depths (train_nerf.py:289-311).
        Nothing per ray or per sample is read: R rays of S samples through pixels first_pixel .. (or `pixels`).
        dir_bands, background and the "acc" / "depth" outputs as in nerf_step_rays (the depths are the camera's)."""
        return self._step(True, dims, None, ws, bs, target, None, int(R), int(S), grad, seed, outputs, out, None, path,
                          False, False, L.HEAD_NERF, pe_bands=pe_bands, camera=camera, dir_bands=dir_bands,
                          background=background)

    def nerf_step_views(self, dims, views, S, pe_bands, ws, bs, target=None, grad=False, seed=1.0,
                        outputs=("color", "loss"), out=None, path="f32", dir_bands=None, background=None):
        """The same step on a views batch (`Scene.batch(...)`, lnb_views): ray r is camera mode's ray of pixel
        pixels[r] under the pose of view[r], S samples each.  target defaults to the batch's drawn target.  dir_bands,
        background and the "acc" / "depth" outputs as in nerf_step_camera."""
        target = views.target if target is None else target
        return self._step(True, dims, None, ws, bs, target, None, views.R, int(S), grad, seed, outputs, out, None, path,
                          False, False, L.HEAD_NERF, pe_bands=pe_bands, dir_bands=dir_bands, background=background,
                          views=views.views)

    def views_rays(self, views, S, out=None):
        """(rays_o, rays_d, t) float64 cuda tensors views mode generates for a views batch (NaN for a ray with an
        out-of-range index)."""
        R, dev = views.R, torch.device("cuda", self.device)
        if out is None:
            out = (torch.empty((R, 3), dtype=torch.float64, device=dev), torch.empty((R, 3), dtype=torch.float64, device=dev),
                   torch.empty((R, S), dtype=torch.float64, device=dev))
        o, d, t = out
        if not all(_is_cuda(v) and v.dtype == torch.float64 and v.is_contiguous() and tuple(v.shape) == sh
                   for v, sh in zip(out, ((R, 3), (R, 3), (R, S)))):
            raise ValueError("views_rays: out must be contiguous [R][3], [R][3], [R][S] float64 CUDA tensors")
        self.order_after_torch()
        self._check(self.lib.lnb_views_rays(self.h, ctypes.byref(views.views), int(R), int(S), o.data_ptr(), d.data_ptr(),
                                            t.data_ptr()))
        return o, d, t

    def camera_rays(self, camera, R, S, out=None):
        """(rays_o, rays_d, t) float64 cuda tensors camera mode generates (for checks / hosts that want them).
        out=(rays_o, rays_d, t): contiguous [R][3], [R][3], [R][S] float64 cuda tensors to write instead of new ones."""
        dev = torch.device("cuda", self.device)
        if out is None:
            out = (torch.empty((R, 3), dtype=torch.float64, device=dev), torch.empty((R, 3), dtype=torch.float64, device=dev),
                   torch.empty((R, S), dtype=torch.float64, device=dev))
        o, d, t = out
        if not all(_is_cuda(v) and v.dtype == torch.float64 and v.is_contiguous() and tuple(v.shape) == sh
                   for v, sh in zip(out, ((R, 3), (R, 3), (R, S)))):
            raise ValueError("camera_rays: out must be contiguous [R][3], [R][3], [R][S] float64 CUDA tensors")
        self.order_after_torch()
        self._check(self.lib.lnb_camera_rays(self.h, ctypes.byref(camera), int(R), int(S), o.data_ptr(), d.data_ptr(), t.data_ptr()))
        return o, d, t

    def sample_pdf(self, t, weights, n_fine, stratified=False, seed=0, ray0=0, out=None):
        """Hierarchical sampling (lnb_sample_pdf): n_fine depths per ray drawn by inverse transform from the piecewise-
        constant PDF of a coarse pass's compositing weights, merged with the coarse depths and sorted.  t [R][S] float64,
        weights [R][S] float32, CUDA tensors; returns out [R][S + n_fine] float64.  Row r of a stratified draw uses
        lnb_uniform(seed, ray0 + r, i), so a chunk passed with its first ray's index reproduces the whole-batch call."""
        if not (_is_cuda(t) and t.dtype == torch.float64 and t.dim() == 2 and t.is_contiguous()):
            raise ValueError("t must be a contiguous [R][S] float64 CUDA tensor")
        R, S = int(t.shape[0]), int(t.shape[1])
        if not (_is_cuda(weights) and weights.dtype == torch.float32 and weights.is_contiguous()
                and tuple(weights.shape) == (R, S)):
            raise ValueError("weights must be a contiguous [%d][%d] float32 CUDA tensor" % (R, S))
        n_fine = int(n_fine)
        if out is None:
            out = torch.empty((R, S + max(n_fine, 0)), dtype=torch.float64, device=t.device)
        elif not (_is_cuda(out) and out.dtype == torch.float64 and out.is_contiguous()
                  and tuple(out.shape) == (R, S + n_fine)):
            raise ValueError("out must be a contiguous [%d][%d] float64 CUDA tensor" % (R, S + n_fine))
        self.order_after_torch()
        self._hold(t, weights, out)
        self._check(self.lib.lnb_sample_pdf(self.h, t.data_ptr(), weights.data_ptr(), R, S, n_fine, int(bool(stratified)),
                                            int(seed) & 0xFFFFFFFFFFFFFFFF, int(ray0), out.data_ptr()))
        return out

    def color_to_u8(self, rgb, out=None):
        """uint8 image bytes of float colours, clamp(rgb, 0, 1) * 255 rounded (train_nerf.py:686-700), on the device."""
        assert _is_cuda(rgb) and rgb.dtype == torch.float32 and rgb.is_contiguous()
        if out is None:
            out = torch.empty(rgb.shape, dtype=torch.uint8, device=rgb.device)
        self.order_after_torch()
        self._check(self.lib.lnb_color_to_u8(self.h, rgb.data_ptr(), rgb.numel(), out.data_ptr()))
        return out

    def fit_step(self, dims, X, ws, bs, target, grad=False, seed=1.0, outputs=("loss",), out=None,
                 rows=None, path="f32", inter_accumulate=False):
        """MLP (sigmoid head) -> SSE loss vs target [-> gradients] (scripts/mlp_fit.py:39-174)."""
        return self._step(False, dims, X, ws, bs, target, None, int(target.shape[0]), 1, grad, seed,
                          outputs, out, rows, path, inter_accumulate, False, L.HEAD_SIGMOID)

    # -------------------------------------------------------------------------------------------
    def pos_encoding(self, x, E):
        """pos_encoding.py:4-70 on the device: x (..., F) float64 cuda -> (..., F*(1+2E)) float32."""
        assert _is_cuda(x) and x.dtype == torch.float64 and x.is_contiguous()
        F = int(x.shape[-1])
        n = x.numel() // F
        o = torch.empty(tuple(x.shape[:-1]) + (F * (1 + 2 * E),), dtype=torch.float32, device=x.device)
        self._check(self.lib.lnb_pos_encoding(self.h, x.data_ptr(), n, F, int(E), o.data_ptr()))
        return o

    def sample_encode(self, rays_o, rays_d, t, E, dir_bands=None):
        """train_nerf.py:289-311 + pos_encoding_3d: returns X [R*S][3+6E] f32 and dists [R][S].  dir_bands=E_d appends
        the unit view direction's encoding: X [R*S][rays_input_width(E, E_d)], what rays mode feeds such a net."""
        assert all(_is_cuda(v) and v.dtype == torch.float64 and v.is_contiguous() for v in (rays_o, rays_d, t))
        R, S = int(t.shape[0]), int(t.shape[1])
        X = torch.empty((R * S, rays_input_width(E, dir_bands)), dtype=torch.float32, device=t.device)
        dists = torch.empty((R, S), dtype=torch.float32, device=t.device)
        if dir_bands is None:
            rc = self.lib.lnb_sample_encode(self.h, rays_o.data_ptr(), rays_d.data_ptr(),
                                            t.data_ptr(), R, S, int(E), X.data_ptr(), dists.data_ptr())
        else:
            rc = self.lib.lnb_sample_encode_dirs(self.h, rays_o.data_ptr(), rays_d.data_ptr(), t.data_ptr(), R, S, int(E),
                                                 int(dir_bands), X.data_ptr(), dists.data_ptr())
        self._check(rc)
        return X, dists

    def mult_a_b(self, a, b, c):
        """c += a @ b on the device (scripts/mlp_fit.py:150-172)."""
        self._check(self.lib.lnb_mult_a_b(self.h, a.data_ptr(), int(a.shape[0]), int(a.shape[1]),
                                          b.data_ptr(), int(b.shape[1]), c.data_ptr()))
        return c

    def adam_step(self, param, grad, m, v, t, lr=5e-4, beta1=0.9, beta2=0.999, eps=1e-8):
        """AdamOptimizer.update of train_nerf.py:133-161 (double bias correction kept), in place."""
        self._check(self.lib.lnb_adam_step(self.h, param.data_ptr(), grad.data_ptr(), m.data_ptr(),
                                           v.data_ptr(), param.numel(), int(t), lr, beta1, beta2, eps))

    def adam_step_dev(self, param, grad, m, v, t_dev, lr=5e-4, beta1=0.9, beta2=0.999, eps=1e-8):
        """adam_step with the step counter in device memory (int32 tensor): graph-capturable."""
        self._check(self.lib.lnb_adam_step_dev(self.h, param.data_ptr(), grad.data_ptr(), m.data_ptr(),
                                               v.data_ptr(), param.numel(), t_dev.data_ptr(), lr, beta1, beta2, eps))

    def sgd_step(self, param, grad, lr):
        """ws -= lr * d_ws (fit_img.py:512-513), in place."""
        self._check(self.lib.lnb_sgd_step(self.h, param.data_ptr(), grad.data_ptr(), param.numel(), lr))


class Trainer:
    """Device-resident weights + optimiser state (lnb_trainer): the reference hosts' per-chunk
    "grad call, then Adam / SGD on the padded arrays" loop (train_nerf.py:395-499,
    fit_img.py:468-513) without host round trips.  Batches are torch CUDA tensors.
    background=(r, g, b): every nerf step composites onto that colour (set_background)."""

    def __init__(self, ctx, dims, ws, bs, head=L.HEAD_NERF, optimizer="adam", lr=5e-4, beta1=0.9, beta2=0.999,
                 eps=1e-8, background=None):
        self.ctx, self.lib = ctx, ctx.lib
        ws = np.ascontiguousarray(ws, np.float32)
        bs = np.ascontiguousarray(bs, np.float32)
        self.dims, self.ws_shape, self.bs_shape = [int(d) for d in dims], ws.shape, bs.shape
        self.mlp = make_mlp(dims, ws.shape, head)
        self.head = head
        h = ctypes.c_void_p()
        opt = {"adam": L.OPT_ADAM, "sgd": L.OPT_SGD}[optimizer]
        ctx._check(self.lib.lnb_trainer_create(ctx.h, ctypes.byref(self.mlp), ws.ctypes.data, bs.ctypes.data, opt,
                                               lr, beta1, beta2, eps, ctypes.byref(h)))
        self.h = h
        self.background = None
        if background is not None:
            self.set_background(background)

    def set_background(self, rgb):
        """Composite every later nerf step (step, step_weights, step_host, submit_host, grad) onto the colour rgb
        (3 floats): colour += (1 - acc) rgb before the loss, on whichever path the step runs (lnb_trainer_set_background).
        None restores the reference's compositing.  With the peer all-reduce every rank must set the same colour."""
        if rgb is None:
            self.ctx._check(self.lib.lnb_trainer_set_background(self.h, None))
            self.background = None
            return
        bg = make_composite(rgb).bg
        arr = (ctypes.c_float * 3)(bg[0], bg[1], bg[2])
        self.ctx._check(self.lib.lnb_trainer_set_background(self.h, arr))
        self.background = (float(bg[0]), float(bg[1]), float(bg[2]))

    def set_views(self, batch):
        """Attach a views batch (`Scene.batch(...)`; lnb_trainer_set_views): later nerf steps with no X, rays or camera
        train on it.  step(views=b) attaches b itself; None detaches.  The host-buffer steps refuse such a batch."""
        self.ctx._check(self.lib.lnb_trainer_set_views(self.h, None if batch is None else ctypes.byref(batch.views)))
        self._views_keep = batch

    def close(self):
        if getattr(self, "h", None):
            self.lib.lnb_trainer_destroy(self.h)
            self.h = None

    def _batch(self, X=None, dists=None, target=None, rays=None, pe_bands=0, R=None, S=None, path="tc", seed=1.0, camera=None,
               dir_bands=None, views=None):
        a = L.LnbStepArgs()
        nerf = self.head == L.HEAD_NERF
        if camera is not None or rays is not None or views is not None:
            check_rays_width(self.dims[0], pe_bands, dir_bands)   # dir_bands: the view direction's bands, as in nerf_step_rays
        if views is not None:   # a views batch: no input of its own, the trainer reads the attached lnb_views
            self.set_views(views)
            target = views.target if target is None else target
            R, S = views.R, int(S)
            a.pe_bands = int(pe_bands)
        elif camera is not None:
            R, S = int(target.shape[0]) if R is None else int(R), int(S)
            a.cam, a.pe_bands = ctypes.pointer(camera), int(pe_bands)
            self._cam_keep = camera
        elif rays is not None:
            ro, rd, tv = rays
            R, S = int(tv.shape[0]), int(tv.shape[1])
            a.rays_o, a.rays_d, a.t = _ptr(ro), _ptr(rd), _ptr(tv)
            a.ray_dtype = L.RAY_F64 if str(ro.dtype).endswith("float64") else L.RAY_F32
            a.pe_bands = int(pe_bands)
        else:
            a.X = _ptr(X)
            if nerf:
                R = int(dists.shape[0]) if R is None else R
                S = int(dists.shape[1]) if S is None else S
                a.dists = _ptr(dists)
            else:
                R, S = int(target.shape[0]), 1
        a.R, a.S, a.target_w = R, S, int(target.shape[1])
        a.n_rows = R * S
        a.target = _ptr(target)
        a.path = PATHS[path]
        if isinstance(seed, str):
            a.seed_mode, a.seed = L.SEED_LOSS, 1.0
        else:
            a.seed_mode, a.seed = L.SEED_VALUE, float(seed)
        return a, int(nerf)

    def prepare(self, **batch):
        """A batch marshalled once (the lnb_step_args struct and the buffers it points at), to be handed to step(),
        step_host() or submit_host() any number of times: a hosts' loop that cycles through pre-built batches pays one ctypes
        call per step instead of rebuilding the struct in Python."""
        a, nerf = self._batch(**batch)
        return PreparedBatch(a, nerf, batch)

    def _order(self, batch):
        self.ctx.order_after_torch()
        self.ctx._hold(*[v for v in batch.values() if _is_cuda(v)], *[x for x in (batch.get("rays") or ()) if _is_cuda(x)])

    def step(self, prepared=None, **batch):
        """forward + backward + optimiser update on one batch (keyword arguments, or a prepare()d batch)."""
        if prepared is not None:
            a, nerf, batch = prepared.args, prepared.nerf, prepared.batch
        else:
            a, nerf = self._batch(**batch)
        self._order(batch)
        self.ctx._check(self.lib.lnb_trainer_step(self.h, ctypes.byref(a), nerf))

    def step_weights(self, weights, prepared=None, **batch):
        """step(), and also writes this step's forward compositing weights w_s = alpha_s T_s (at the parameters before
        the update) into weights, a [R][S] float32 CUDA tensor (lnb_trainer_step_weights).  nerf batches only."""
        if prepared is not None:
            a, nerf, batch = prepared.args, prepared.nerf, prepared.batch
        else:
            a, nerf = self._batch(**batch)
        if not (_is_cuda(weights) and weights.dtype == torch.float32 and weights.is_contiguous()
                and tuple(weights.shape) == (a.R, a.S)):
            raise ValueError("weights must be a contiguous [%d][%d] float32 CUDA tensor" % (a.R, a.S))
        self._order(batch)
        self.ctx._hold(weights)
        self.ctx._check(self.lib.lnb_trainer_step_weights(self.h, ctypes.byref(a), nerf, weights.data_ptr()))

    def step_host(self, prepared=None, **batch):
        """step() with the batch in host memory (numpy arrays / pinned CPU tensors): the C library
        stages it to the device, steps, and returns the loss.  Synchronous."""
        a, nerf = (prepared.args, prepared.nerf) if prepared is not None else self._batch(**batch)
        loss = ctypes.c_float()
        self.ctx._check(self.lib.lnb_trainer_step_host(self.h, ctypes.byref(a), nerf, ctypes.byref(loss)))
        return float(loss.value)

    def submit_host(self, prepared=None, **batch):
        """step_host() without the wait: the batch is staged on a copy stream while the previous step still runs
        (lnb_trainer_submit_host).  Pinned host buffers must stay unchanged until the submission after next."""
        if prepared is not None:
            a, nerf, batch = prepared.args, prepared.nerf, prepared
        else:
            a, nerf = self._batch(**batch)
        self._keep = (self.__dict__.get("_keep", []) + [batch])[-3:]
        self.ctx._check(self.lib.lnb_trainer_submit_host(self.h, ctypes.byref(a), nerf))

    def wait(self, max_losses=4096):
        """Block until every submitted step is done; losses of the steps submitted since the last wait (oldest first)."""
        buf = (ctypes.c_float * max_losses)()
        n = ctypes.c_int()
        self.ctx._check(self.lib.lnb_trainer_wait(self.h, buf, max_losses, ctypes.byref(n)))
        return [float(buf[i]) for i in range(n.value)]

    def grad(self, **batch):
        """forward + backward only: gradients (and loss) land in grad_buffer()."""
        a, nerf = self._batch(**batch)
        self._order(batch)
        self.ctx._check(self.lib.lnb_trainer_grad(self.h, ctypes.byref(a), nerf))

    def apply(self):
        self.ctx._check(self.lib.lnb_trainer_apply(self.h))

    def enable_peer_allreduce(self, group=None):
        """Fuse the gradient all-reduce into the step (tensor-core path, GPUs of one box): exchanges
        CUDA IPC handles of the per-rank exchange buffers through torch.distributed and attaches
        them.  Afterwards step()/step_host() sum gradients and loss over all ranks inside the
        reduction kernel (NVLink peer loads) and every rank must step in lockstep."""
        import torch.distributed as dist
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        h = ctypes.create_string_buffer(64)
        self.ctx._check(self.lib.lnb_trainer_comm_export(self.h, h))
        handles = [None] * world
        dist.all_gather_object(handles, bytes(h.raw), group=group)
        blob = ctypes.create_string_buffer(b"".join(handles), 64 * world)
        self.ctx._check(self.lib.lnb_trainer_comm_attach(self.h, rank, world, blob))
        dist.barrier(group)
        return True

    def comm_status(self):
        """0 = fine, 1 = a peer timed out and that step was poisoned with NaN.  Synchronises."""
        return int(self.lib.lnb_trainer_comm_status(self.h))

    def check_comm(self):
        if self.comm_status() != 0:
            raise LnbError("peer all-reduce: a rank did not deliver its gradients in time; the step was poisoned (NaN)")

    def grad_buffer(self):
        """torch view of the flat [d_ws | d_bs | loss] device buffer (for dist.all_reduce).  The
        library writes it on the context's stream: use ctx.order_torch_after() before torch reads it
        and ctx.order_after_torch() before apply() (sharding.data_parallel_step does both)."""
        n = ctypes.c_longlong()
        ptr = self.lib.lnb_trainer_grad_buffer(self.h, ctypes.byref(n))
        return _torch_view(ptr, n.value, self.ctx.device)

    def read(self):
        """(ws, bs, loss) as numpy; synchronises."""
        ws = np.empty(self.ws_shape, np.float32)
        bs = np.empty(self.bs_shape, np.float32)
        loss = np.empty(1, np.float32)
        self.ctx._check(self.lib.lnb_trainer_read(self.h, ws.ctypes.data, bs.ctypes.data, loss.ctypes.data))
        return ws, bs, float(loss[0])


class CoarseFine:
    """Hierarchical sampling in training (the NeRF paper's coarse-to-fine step), on the device.  One step():
      1. camera batch: the rays and the S coarse depths (lnb_camera_rays) into buffers this object owns;
      2. a coarse Trainer.step_weights on the batch (a camera batch stays in camera mode);
      3. sample_pdf: n_fine depths from the coarse weights, merged with the coarse ones (S + n_fine, sorted);
      4. a fine Trainer.step in rays mode on (rays_o, rays_d, t_fine).
    Both nets train on their own colour loss.  Nothing is synchronised with the host and, after the first step of a
    shape, nothing is allocated: a run of steps can be captured in one CUDA graph.  The two nets may differ in shape;
    each runs on the path its shape and sample count select.  Not for a trainer with the peer all-reduce attached.
    Backgrounds need nothing here: each trainer composites onto its own (Trainer(..., background=) / set_background), so a
    white-background run gives both trainers background=(1, 1, 1)."""

    def __init__(self, coarse, fine, n_fine, stratified=True):
        if coarse.head != L.HEAD_NERF or fine.head != L.HEAD_NERF:
            raise ValueError("CoarseFine needs two nerf trainers")
        self.coarse, self.fine, self.n_fine, self.stratified = coarse, fine, int(n_fine), bool(stratified)
        self.ctx = coarse.ctx
        self._buf, self._key = None, None

    def _buffers(self, R, S, device):
        key = (R, S, str(device))
        if self._key != key:
            f64 = dict(dtype=torch.float64, device=device)
            self._buf = dict(o=torch.empty((R, 3), **f64), d=torch.empty((R, 3), **f64), t=torch.empty((R, S), **f64),
                             w=torch.empty((R, S), dtype=torch.float32, device=device),
                             t_fine=torch.empty((R, S + self.n_fine), **f64))
            self._key = key
        return self._buf

    def step(self, camera=None, rays=None, S=None, pe_bands=0, dir_bands=None, target=None, path="tc", seed=None):
        """One coarse-to-fine train step on a camera batch (camera=make_camera(...), S coarse depths, R = len(target))
        or a rays batch (rays=(rays_o, rays_d, t), float64 CUDA tensors).  seed: the stratified fine draw's seed
        (default: the camera's seed; 0 for a rays batch).  Returns the buffers of this step: o, d, t (coarse depths),
        w (coarse weights) and t_fine."""
        if (camera is None) == (rays is None):
            raise ValueError("pass exactly one of camera= and rays=")
        if target is None:
            raise ValueError("a train step needs a target")
        ctx = self.ctx
        R = int(target.shape[0])
        if camera is not None:
            S = int(S)
            b = self._buffers(R, S, target.device)
            o, d, t = ctx.camera_rays(camera, R, S, out=(b["o"], b["d"], b["t"]))
            self.coarse.step_weights(b["w"], camera=camera, R=R, S=S, pe_bands=pe_bands, dir_bands=dir_bands,
                                     target=target, path=path)
            seed = camera.seed if seed is None else seed
            ray0 = camera.first_pixel if not camera.pixels else 0
        else:
            o, d, t = rays
            if not all(_is_cuda(v) and v.dtype == torch.float64 for v in (o, d, t)):
                raise ValueError("a rays batch must be float64 CUDA tensors (the sampler bins float64 depths)")
            S = int(t.shape[1])
            b = self._buffers(R, S, target.device)
            self.coarse.step_weights(b["w"], rays=(o, d, t), pe_bands=pe_bands, dir_bands=dir_bands, target=target, path=path)
            seed, ray0 = (0 if seed is None else seed), 0
        ctx.sample_pdf(t, b["w"], self.n_fine, stratified=self.stratified, seed=seed, ray0=ray0, out=b["t_fine"])
        self.fine.step(rays=(o, d, b["t_fine"]), pe_bands=pe_bands, dir_bands=dir_bands, target=target, path=path)
        return dict(o=o, d=d, t=t, w=b["w"], t_fine=b["t_fine"])


class Scene:
    """A training scene held on the device: poses [n_views][12] float64 (the 3 x 4 camera-to-world rows) and images
    [n_views][P][3] float32, P = width * height, uploaded once.  batch() makes the per-step views batches drawn from it."""

    def __init__(self, ctx, poses, images, normalized_K, near=2.0, far=6.0):
        self.ctx = ctx
        dev = torch.device("cuda", ctx.device)
        images = torch.as_tensor(np.asarray(images, np.float32) if not isinstance(images, torch.Tensor) else images)
        if images.dim() != 4 or images.shape[3] != 3:
            raise ValueError("images must be [n_views][height][width][3], got %r" % (tuple(images.shape),))
        self.n_views, self.height, self.width = int(images.shape[0]), int(images.shape[1]), int(images.shape[2])
        pz = np.asarray(poses.cpu() if isinstance(poses, torch.Tensor) else poses, np.float64)
        if pz.shape[0] != self.n_views or pz.shape[1:] not in ((3, 4), (4, 4)):
            raise ValueError("poses must be [n_views][3 or 4][4], got %r" % (pz.shape,))
        self.poses = torch.as_tensor(np.ascontiguousarray(pz[:, :3, :4].reshape(self.n_views, 12))).to(dev)
        self.images = images.to(device=dev, dtype=torch.float32).reshape(self.n_views, self.width * self.height, 3).contiguous()
        K = np.asarray(normalized_K, np.float64)
        self.fx, self.fy, self.cx, self.cy = float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])
        self.near, self.far = float(near), float(far)

    @property
    def P(self):
        return self.width * self.height

    @classmethod
    def from_blender(cls, ctx, scene, near=2.0, far=6.0):
        """Every frame of a dataset.BlenderScene (its white_background compositing included)."""
        frames = [scene[i] for i in range(len(scene))]
        return cls(ctx, np.stack([f["pose"] for f in frames]), np.stack([f["image"] for f in frames]), scene.normalized_K,
                   near=near, far=far)

    def batch(self, R, stratified=False, one_view=False, seed=0):
        """A views batch of R rays drawn from this scene (ViewsBatch).  one_view=True: every ray of a step from one view
        (the paper's Blender protocol); else from all views.  seed: the draw's seed."""
        return ViewsBatch(self, R, stratified, one_view, seed)


class ViewsBatch:
    """The buffers of one step's views batch (view, pixels [R] int32, target [R][3] float32, the step's jitter seed and
    the draw counter [2] int64 (counter[0] = the next draw's k), all on the device) and the lnb_views that points at them.
    draw() writes a new batch and advances the counter (lnb_views_draw), so a captured graph of draw() + a step trains on a
    new batch at every replay.  The stratified jitter seed is the drawn step seed (views.seed_dev)."""

    def __init__(self, scene, R, stratified=False, one_view=False, seed=0):
        self.scene, self.ctx, self.R = scene, scene.ctx, int(R)
        self.one_view, self.seed = bool(one_view), int(seed) & 0xFFFFFFFFFFFFFFFF
        dev = scene.images.device
        self.view = torch.zeros(self.R, dtype=torch.int32, device=dev)
        self.pixels = torch.zeros(self.R, dtype=torch.int32, device=dev)
        self.target = torch.zeros((self.R, 3), dtype=torch.float32, device=dev)
        self.step_seed = torch.zeros(1, dtype=torch.int64, device=dev)
        self.counter = torch.zeros(2, dtype=torch.int64, device=dev)
        v = L.LnbViews()
        v.poses, v.n_views, v.width, v.height = scene.poses.data_ptr(), scene.n_views, scene.width, scene.height
        v.fx, v.fy, v.cx, v.cy, v.near, v.far = scene.fx, scene.fy, scene.cx, scene.cy, scene.near, scene.far
        v.stratified, v.seed, v.seed_dev = int(bool(stratified)), 0, self.step_seed.data_ptr()
        v.view, v.pixels = self.view.data_ptr(), self.pixels.data_ptr()
        self.views = v

    def draw(self):
        """Launch the draw on the context's stream."""
        ctx, sc = self.ctx, self.scene
        ctx.order_after_torch()
        ctx._check(ctx.lib.lnb_views_draw(ctx.h, sc.images.data_ptr(), sc.n_views, sc.P, self.R, int(self.one_view), self.seed,
                                          self.counter.data_ptr(), self.view.data_ptr(), self.pixels.data_ptr(),
                                          self.target.data_ptr(), self.step_seed.data_ptr()))


class PreparedBatch:
    """Trainer.prepare(): the marshalled lnb_step_args of one batch plus references that keep its buffers alive."""
    __slots__ = ("args", "nerf", "batch")

    def __init__(self, args, nerf, batch):
        self.args, self.nerf, self.batch = args, nerf, batch


def _torch_view(ptr, n_floats, device):
    """float32 torch tensor aliasing n_floats of device memory at ptr (no copy, no ownership)."""
    class _Arr:
        __cuda_array_interface__ = {"shape": (int(n_floats),), "typestr": "<f4", "data": (int(ptr), False), "version": 3,
                                    "strides": None}
    return torch.as_tensor(_Arr(), device=torch.device("cuda", device))
