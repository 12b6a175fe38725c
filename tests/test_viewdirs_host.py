"""View directions in rays and camera mode, host side: the float64 restatement of the direction input
(oracle/viewdirs.py) and the Python rule that ties dims[0] to (pe_bands, dir_bands).  No GPU."""
import numpy as np
import pytest

from oracle import oracle as O
from oracle import viewdirs as V


def test_view_encoding_is_the_unit_direction_per_ray():
    rng = np.random.default_rng(3)
    R, S = 17, 5
    _, d = O.synthetic_rays(rng, R)
    d = d * rng.uniform(0.2, 5.0, (R, 1))                       # lengths must not matter
    for E_d in (0, 1, 4):
        enc = V.view_encoding(d, E_d, S)
        assert enc.shape == (R * S, 3 + 6 * E_d) and enc.dtype == np.float32
        u = enc[:, :3].astype(np.float64)
        assert np.abs(np.linalg.norm(u, axis=1) - 1.0).max() <= 4e-7
        per_ray = enc.reshape(R, S, -1)
        assert (per_ray == per_ray[:, :1]).all()                 # the same columns for every sample of a ray
        assert np.array_equal(per_ray[:, 0], O.positional_encoding(V.unit_directions(d), E_d))
    assert V.view_encoding(d, 0, S).shape[1] == 3


def test_features_append_the_direction_after_the_positions():
    case = O.make_nerf_case(4, 6, 7, E=3)
    X, dists = V.features(case["rays_o"], case["rays_d"], case["t"], 3, 2)
    assert X.shape == (42, 21 + 15)
    assert np.array_equal(X[:, :21], case["X"]) and np.array_equal(dists, case["dists"])
    assert np.array_equal(X[:, 21:], V.view_encoding(case["rays_d"], 2, 7))


@pytest.mark.parametrize("args", [(11, 8, 16), (5, 4, 64), (3, 9, 1)])
def test_make_nerf_case_without_directions_is_unchanged(args):
    a, b = O.make_nerf_case(*args), V.make_nerf_case(*args)
    assert sorted(a) == sorted(b)
    for k in a:
        assert np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes(), k


def test_make_nerf_case_with_directions():
    case = V.make_nerf_case(12, 9, 8, E=10, E_dir=4)
    assert case["X"].shape == (72, 90) and list(case["dims"]) == [90, 30, 30, 4]
    assert case["ws"].shape == (3, 90, 30)
    base = O.make_nerf_case(12, 9, 8, E=10)
    assert np.array_equal(case["X"][:, :63], base["X"]) and np.array_equal(case["dists"], base["dists"])


@pytest.mark.parametrize("dims0,E,E_d", [(33, 5, None), (63, 10, None), (3, 0, None), (60, 5, 4), (90, 10, 4),
                                         (36, 5, 0), (6, 0, 0), (42, 5, 1)])
def test_width_rule_accepts(dims0, E, E_d):
    from loma_nerf_b200 import api
    assert api.rays_input_width(E, E_d) == dims0
    api.check_rays_width(dims0, E, E_d)


@pytest.mark.parametrize("dims0,E,E_d", [
    (60, 5, None),      # a direction-form width without dir_bands
    (90, 10, None),
    (33, 5, 0),         # dir_bands for a positions-only width
    (60, 5, 3),         # dir_bands that disagree with dims[0]
    (34, 5, None),      # neither form
    (64, 10, None),
    (33, 4, None),      # wrong position bands
    (60, 5, -1),
    (33, -1, None),
])
def test_width_rule_refuses(dims0, E, E_d):
    from loma_nerf_b200 import api
    with pytest.raises(ValueError):
        api.check_rays_width(dims0, E, E_d)
