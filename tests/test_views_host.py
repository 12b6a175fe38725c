"""Views mode without a GPU: the draw's pick rule (lnb_views_pick) against a Python-integer restatement, and the ctypes
mirror of lnb_views against the library's layout."""
import ctypes

import pytest

from loma_nerf_b200 import _lib as L

M64 = (1 << 64) - 1


def mix(z):
    z ^= z >> 30
    z = (z * 0xBF58476D1CE4E5B9) & M64
    z ^= z >> 27
    z = (z * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def z_of(seed, k, i):
    return mix((seed + 0x9E3779B97F4A7C15 * ((k << 32) + i + 1)) & M64)


def pick(seed, k, i, n):
    return (z_of(seed, k, i) * n) >> 64


@pytest.fixture(scope="module")
def lib():
    return L.load()


@pytest.mark.parametrize("seed", [0, 1, 12345, M64, 0x9E3779B97F4A7C15])
def test_views_pick_matches_rule(lib, seed):
    ns = [1, 2, 3, 800 * 800, 100 * 800 * 800, (1 << 31) - 1, (1 << 32) + 7, 5 * (1 << 40) + 3, M64]
    for k in (0, 1, 7, (1 << 32) - 1, 1 << 40):
        for i in (0, 1, 255, 4095, (1 << 32) - 2, (1 << 32) - 1):
            for n in ns:
                got = lib.lnb_views_pick(seed, k, i, n)
                assert got == pick(seed, k, i, n), (seed, k, i, n)
                assert 0 <= got < n


def test_views_pick_spreads_views_and_pixels(lib):
    # all-views mode splits g = pick(n_views * P) into (view, pixel); every view should appear in a modest draw
    n_views, P = 5, 37
    seen = {pick(3, 2, r, n_views * P) // P for r in range(400)}
    assert seen == set(range(n_views))
    assert [lib.lnb_views_pick(3, 2, r, n_views * P) for r in range(50)] == [pick(3, 2, r, n_views * P) for r in range(50)]


def test_views_layout_matches_mirror(lib):
    out = (ctypes.c_int * 16)()
    n = lib.lnb_views_layout(out, 16)
    V = L.LnbViews
    want = [ctypes.sizeof(V), V.poses.offset, V.n_views.offset, V.fx.offset, V.near.offset, V.stratified.offset,
            V.seed.offset, V.seed_dev.offset, V.view.offset, V.pixels.offset]
    assert n == len(want)
    assert list(out[:n]) == want
