"""Compositing extras without a GPU: the float64 model with a background (tests/composite_model.py) against finite
differences of its own loss, its agreement with the oracle when nothing is asked for, the bf16 model's exact mode, the
white-background Blender reader and the lnb_composite mirror."""
import json
import os

import numpy as np
import pytest

import composite_model as CM
from oracle import oracle as O

BG = np.array([1.0, 0.25, 0.6])


def _rgba_case(seed, R=3, S=7):
    rng = np.random.default_rng(seed)
    rgba = np.concatenate([rng.uniform(0.05, 0.95, (R * S, 3)), rng.uniform(0.2, 3.0, (R * S, 1))], 1)
    t = np.sort(rng.uniform(2.0, 6.0, (R, S)), 1)
    dists = np.concatenate([t[:, 1:] - t[:, :-1], np.full((R, 1), 0.5)], 1)
    target = rng.uniform(0, 1, (R, 3))
    return rgba, dists, target, t, R, S


@pytest.mark.parametrize("g", [1.0, "loss"])
def test_background_adjoint_against_finite_differences(g):
    rgba, dists, target, t, R, S = _rgba_case(1)
    res = CM.composite_f64(rgba, dists, target, R, S, g, bg=BG)
    scale = res["g"]

    def loss(rg, di):
        return CM.composite_f64(rg, di, target, R, S, bg=BG)["loss"]

    h = 1e-6
    for idx in [(0, 0), (4, 1), (10, 2), (2, 3), (13, 3), (20, 3)]:
        a, b = rgba.copy(), rgba.copy()
        a[idx] += h
        b[idx] -= h
        fd = (loss(a, dists) - loss(b, dists)) / (2 * h)
        assert abs(scale * fd - res["dY"][idx]) <= 1e-6 * max(1.0, abs(res["dY"][idx])), (idx, fd, res["dY"][idx])
    for idx in [(0, 0), (1, 3), (2, 5)]:
        a, b = dists.copy(), dists.copy()
        a[idx] += h
        b[idx] -= h
        fd = (loss(rgba, a) - loss(rgba, b)) / (2 * h)
        assert abs(scale * fd - res["d_dists"][idx]) <= 1e-6 * max(1.0, abs(res["d_dists"][idx])), (idx, fd)


def test_no_background_is_the_oracle_exactly():
    rgba, dists, target, t, R, S = _rgba_case(2)
    for g in (None, 1.0, "loss"):
        ref = O.composite_f64(rgba, dists, target, R, S, g)
        res = CM.composite_f64(rgba, dists, target, R, S, g, t=t)
        for k, v in ref.items():
            assert np.array_equal(np.asarray(res[k]), np.asarray(v)), k


def test_zero_background_changes_nothing_but_the_extras():
    rgba, dists, target, t, R, S = _rgba_case(3)
    ref = O.composite_f64(rgba, dists, target, R, S, 1.0)
    res = CM.composite_f64(rgba, dists, target, R, S, 1.0, bg=np.zeros(3))
    for k in ("loss", "color", "dY", "d_dists"):
        np.testing.assert_allclose(res[k], ref[k], rtol=0, atol=1e-15)


def test_acc_and_depth_are_sums_of_the_weights():
    rgba, dists, target, t, R, S = _rgba_case(4)
    res = CM.composite_f64(rgba, dists, target, R, S, bg=BG, t=t)
    assert np.array_equal(res["acc"], res["weights"].sum(1))
    assert np.array_equal(res["depth"], (res["weights"] * t).sum(1))
    assert (res["acc"] <= 1.0 + 1e-9).all()
    # the background fills exactly what the samples leave
    np.testing.assert_allclose(res["color"], (res["weights"][..., None] * rgba.reshape(R, S, 4)[..., :3]).sum(1)
                               + (1 - res["acc"])[:, None] * BG, rtol=0, atol=1e-15)


def test_tc_model_exact_mode_with_background_is_the_f64_model():
    case = O.make_nerf_case(7, 33, 9, E=3, width=12, n_layers=3)
    args = (case["X"], case["ws"], case["bs"], case["dims"], case["target"], case["dists"], 33, 9)
    for g in (None, 1.0, "loss"):
        m = CM.nerf_tc_model(*args, g=g, bg=BG, t=case["t"], _exact=True)
        f = CM.nerf_f64(*args, g=g, bg=BG, t=case["t"])
        for k in ("loss", "color", "acc", "depth") + (("d_ws", "d_bs") if g is not None else ()):
            np.testing.assert_allclose(m[k], f[k], rtol=1e-12, atol=1e-12 * max(1.0, np.abs(f[k]).max()))


def test_blender_white_background(tmp_path):
    from PIL import Image
    from loma_nerf_b200.dataset import BlenderScene
    rgba = np.zeros((4, 4, 4), np.uint8)
    rgba[..., 0] = 200
    rgba[..., 1] = 40
    rgba[..., 2] = 100
    rgba[..., 3] = np.arange(16).reshape(4, 4) * 17
    os.makedirs(tmp_path / "train")
    Image.fromarray(rgba, "RGBA").save(tmp_path / "train" / "r_0.png")
    with open(tmp_path / "transforms_train.json", "w") as fh:
        json.dump({"camera_angle_x": 0.69, "frames": [{"file_path": "./train/r_0", "transform_matrix": np.eye(4).tolist()}]}, fh)
    white = BlenderScene(str(tmp_path), img_size=4, white_background=True)[0]["image"]
    a = rgba[..., 3:].astype(np.float32) / 255.0
    want = rgba[..., :3].astype(np.float32) / 255.0 * a + (1.0 - a)
    np.testing.assert_allclose(white, want, rtol=0, atol=1e-6)
    assert white.dtype == np.float32 and white.shape == (4, 4, 3)
    plain = BlenderScene(str(tmp_path), img_size=4)[0]["image"]     # the default drops alpha, as before
    np.testing.assert_array_equal(plain, np.asarray(Image.fromarray(rgba, "RGBA").convert("RGB"), np.float32) / 255.0)


def test_composite_mirror_matches_the_library():
    import ctypes
    from loma_nerf_b200 import _lib as L
    lib = L.load()
    out = (ctypes.c_int * 8)()
    n = lib.lnb_composite_layout(out, 8)
    C = L.LnbComposite
    assert n == 5
    assert list(out[:n]) == [ctypes.sizeof(C), C.background.offset, C.bg.offset, C.acc.offset, C.depth.offset]
