"""ctypes binding of libloma_nerf_b200.so (include/loma_nerf_b200.h).

The CUDA library IS the product: importing this module fails loudly when the library has not been
built, and nothing here (or anywhere in the package) falls back to a CPU implementation.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_longlong, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libloma_nerf_b200.so")

LNB_MAX_LAYERS = 16
LNB_OK, LNB_ERR_CUDA, LNB_ERR_ARG, LNB_ERR_UNSUPPORTED = 0, 1, 2, 3
HEAD_NERF, HEAD_SIGMOID = 0, 1
SEED_VALUE, SEED_LOSS = 0, 1
PATH_F32, PATH_TC, PATH_F32_LAYERWISE = 0, 1, 2
RAY_F64, RAY_F32 = 0, 1
OPT_ADAM, OPT_SGD = 0, 1

c_float_p = POINTER(c_float)


class LnbMlp(Structure):
    _fields_ = [("n_layers", c_int), ("dims", c_int * (LNB_MAX_LAYERS + 1)), ("max_in", c_int),
                ("max_out", c_int), ("head", c_int)]


class LnbCamera(Structure):
    """Mirror of lnb_camera (camera mode: rays and sample depths generated on the device from a pose)."""
    _fields_ = [("c2w", c_double * 12), ("fx", c_double), ("fy", c_double), ("cx", c_double), ("cy", c_double),
                ("width", c_int), ("height", c_int), ("first_pixel", c_longlong), ("pixels", c_void_p),
                ("near", c_double), ("far", c_double), ("stratified", c_int), ("seed", ctypes.c_ulonglong)]


class LnbStepArgs(Structure):
    """Mirror of lnb_step_args; field order and types must match the header exactly
    (tests/test_abi.py compares sizeof and offsets with the values the library reports)."""
    _fields_ = [
        ("R", c_int), ("S", c_int), ("n_rows", c_int), ("rows", c_int), ("target_w", c_int),
        ("X", c_void_p), ("ws", c_void_p), ("bs", c_void_p), ("target", c_void_p),
        ("dists", c_void_p),
        ("inter", c_void_p), ("inter_rows", c_int), ("inter_ld", c_int),
        ("inter_accumulate", c_int),
        ("rgba", c_void_p), ("alpha", c_void_p), ("cumprod", c_void_p), ("weights", c_void_p),
        ("color", c_void_p), ("color_accumulate", c_int),
        ("loss", c_void_p),
        ("want_grad", c_int), ("seed_mode", c_int), ("seed", c_float),
        ("d_ws", c_void_p), ("d_bs", c_void_p), ("d_X", c_void_p), ("d_target", c_void_p),
        ("d_dists", c_void_p), ("d_color", c_void_p), ("d_inter", c_void_p),
        ("path", c_int),
        ("rays_o", c_void_p), ("rays_d", c_void_p), ("t", c_void_p), ("ray_dtype", c_int),
        ("pe_bands", c_int),
        ("cam", POINTER(LnbCamera)),
    ]


class LnbComposite(Structure):
    """Mirror of lnb_composite (compositing extras: background colour, opacity and depth maps); checked against
    lnb_composite_layout."""
    _fields_ = [("background", c_int), ("bg", c_float * 3), ("acc", c_void_p), ("depth", c_void_p)]


class LnbViews(Structure):
    """Mirror of lnb_views (views mode: camera mode with a pose per ray); checked against lnb_views_layout."""
    _fields_ = [("poses", c_void_p), ("n_views", c_int), ("width", c_int), ("height", c_int),
                ("fx", c_double), ("fy", c_double), ("cx", c_double), ("cy", c_double), ("near", c_double), ("far", c_double),
                ("stratified", c_int), ("seed", ctypes.c_ulonglong), ("seed_dev", c_void_p), ("view", c_void_p),
                ("pixels", c_void_p)]


class LibraryMissing(RuntimeError):
    pass


_lib = None


def load():
    """Load the library (once) and set argtypes for the flat API."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryMissing(
            "%s not found: build it with `python -m loma_nerf_b200.build` (nvcc, sm_100a). "
            "There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    P = POINTER
    lib.lnb_abi_version.restype = c_int
    lib.lnb_device_count.restype = c_int
    lib.lnb_create.argtypes = [P(c_void_p), c_int]
    lib.lnb_create.restype = c_int
    lib.lnb_destroy.argtypes = [c_void_p]
    lib.lnb_destroy.restype = None
    lib.lnb_set_stream.argtypes = [c_void_p, c_void_p]
    lib.lnb_synchronize.argtypes = [c_void_p]
    lib.lnb_last_error.argtypes = [c_void_p]
    lib.lnb_last_error.restype = c_char_p
    lib.lnb_launch_count.argtypes = [c_void_p]
    lib.lnb_launch_count.restype = c_longlong
    lib.lnb_profile.argtypes = [c_void_p, c_int]
    lib.lnb_profile_read.argtypes = [c_void_p, P(c_double), P(c_longlong), c_char_p, c_int]
    lib.lnb_host_alloc.argtypes = [c_size_t]
    lib.lnb_host_alloc.restype = c_void_p
    lib.lnb_host_free.argtypes = [c_void_p]
    lib.lnb_host_free.restype = None
    for name in ("lnb_nerf_step", "lnb_fit_step", "lnb_nerf_step_host", "lnb_fit_step_host"):
        fn = getattr(lib, name)
        fn.argtypes = [c_void_p, P(LnbMlp), P(LnbStepArgs)]
        fn.restype = c_int
    for name in ("lnb_nerf_step_composite", "lnb_nerf_step_composite_host"):
        fn = getattr(lib, name)
        fn.argtypes = [c_void_p, P(LnbMlp), P(LnbStepArgs), P(LnbComposite)]
        fn.restype = c_int
    lib.lnb_nerf_step_views.argtypes = [c_void_p, P(LnbMlp), P(LnbStepArgs), P(LnbViews), P(LnbComposite)]
    lib.lnb_nerf_step_views.restype = c_int
    lib.lnb_views_layout.argtypes = [P(c_int), c_int]
    lib.lnb_views_layout.restype = c_int
    lib.lnb_views_rays.argtypes = [c_void_p, P(LnbViews), c_int, c_int, c_void_p, c_void_p, c_void_p]
    lib.lnb_views_draw.argtypes = [c_void_p, c_void_p, c_int, c_longlong, c_int, c_int, ctypes.c_ulonglong, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p]
    lib.lnb_views_pick.argtypes = [ctypes.c_ulonglong, ctypes.c_ulonglong, ctypes.c_ulonglong, ctypes.c_ulonglong]
    lib.lnb_views_pick.restype = ctypes.c_ulonglong
    lib.lnb_trainer_set_views.argtypes = [c_void_p, P(LnbViews)]
    lib.lnb_trainer_set_views.restype = c_int
    lib.lnb_composite_layout.argtypes = [P(c_int), c_int]
    lib.lnb_composite_layout.restype = c_int
    lib.lnb_pos_encoding.argtypes = [c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p]
    lib.lnb_sample_encode.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                      c_void_p, c_void_p]
    lib.lnb_sample_encode_dirs.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                           c_void_p, c_void_p]
    lib.lnb_camera_rays.argtypes = [c_void_p, P(LnbCamera), c_int, c_int, c_void_p, c_void_p, c_void_p]
    lib.lnb_color_to_u8.argtypes = [c_void_p, c_void_p, c_longlong, c_void_p]
    lib.lnb_uniform.argtypes = [ctypes.c_ulonglong, c_longlong, c_int]
    lib.lnb_uniform.restype = c_double
    lib.lnb_sample_pdf.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.c_ulonglong,
                                   c_longlong, c_void_p]
    lib.lnb_mult_a_b.argtypes = [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]
    lib.lnb_adam_step.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_longlong,
                                  c_int, c_double, c_double, c_double, c_double]
    lib.lnb_adam_step_dev.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_longlong,
                                      c_void_p, c_double, c_double, c_double, c_double]
    lib.lnb_sgd_step.argtypes = [c_void_p, c_void_p, c_void_p, c_longlong, c_double]
    lib.lnb_trainer_create.argtypes = [c_void_p, P(LnbMlp), c_void_p, c_void_p, c_int, c_double, c_double,
                                       c_double, c_double, P(c_void_p)]
    lib.lnb_trainer_destroy.argtypes = [c_void_p]
    lib.lnb_trainer_destroy.restype = None
    for name in ("lnb_trainer_step", "lnb_trainer_grad"):
        getattr(lib, name).argtypes = [c_void_p, P(LnbStepArgs), c_int]
    lib.lnb_trainer_set_background.argtypes = [c_void_p, P(c_float)]
    lib.lnb_trainer_set_background.restype = c_int
    lib.lnb_trainer_step_weights.argtypes = [c_void_p, P(LnbStepArgs), c_int, c_void_p]
    lib.lnb_trainer_step_host.argtypes = [c_void_p, P(LnbStepArgs), c_int, P(c_float)]
    lib.lnb_trainer_submit_host.argtypes = [c_void_p, P(LnbStepArgs), c_int]
    lib.lnb_trainer_wait.argtypes = [c_void_p, P(c_float), c_int, P(c_int)]
    lib.lnb_trainer_comm_export.argtypes = [c_void_p, c_void_p]
    lib.lnb_trainer_comm_attach.argtypes = [c_void_p, c_int, c_int, c_void_p]
    lib.lnb_trainer_comm_status.argtypes = [c_void_p]
    lib.lnb_trainer_apply.argtypes = [c_void_p]
    lib.lnb_trainer_grad_buffer.argtypes = [c_void_p, P(c_longlong)]
    lib.lnb_trainer_grad_buffer.restype = c_void_p
    lib.lnb_trainer_params.argtypes = [c_void_p, P(c_longlong), P(c_longlong)]
    lib.lnb_trainer_params.restype = c_void_p
    lib.lnb_trainer_read.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p]
    lib.lnb_default_ctx.restype = c_void_p
    lib.lnb_struct_layout.argtypes = [P(c_int), c_int]
    lib.lnb_struct_layout.restype = c_int
    _lib = lib
    return lib
