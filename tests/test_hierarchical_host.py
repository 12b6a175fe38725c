"""Hierarchical sampling's float64 restatement (oracle/hierarchical.py) against an independent transcription of the NeRF
paper's sample_pdf, and the properties every output row has.  No GPU needed."""
import numpy as np
import pytest

from oracle import hierarchical as Hs


def paper_sample_pdf(bins, weights, u):
    """The paper's sample_pdf line by line (normalise, cumsum, searchsorted, gather), one ray at a time, with the sample
    positions u given.  bins [S-1] midpoints, weights [S-2] interior weights."""
    weights = weights + 1e-5
    pdf = weights / np.sum(weights)
    cdf = np.concatenate([[0.0], np.cumsum(pdf)])
    inds = np.searchsorted(cdf, u, side="right")
    below = np.maximum(0, inds - 1)
    above = np.minimum(len(cdf) - 1, inds)
    cdf_g = np.stack([cdf[below], cdf[above]], -1)
    bins_g = np.stack([bins[below], bins[above]], -1)
    denom = cdf_g[:, 1] - cdf_g[:, 0]
    denom = np.where(denom < 1e-5, np.ones_like(denom), denom)
    tt = (u - cdf_g[:, 0]) / denom
    return bins_g[:, 0] + tt * (bins_g[:, 1] - bins_g[:, 0])


def _case(seed, R, S, kind="random"):
    rng = np.random.default_rng(seed)
    t = np.sort(rng.uniform(2.0, 6.0, (R, S)), axis=1)
    if kind == "random":
        w = rng.uniform(0, 1, (R, S)).astype(np.float32) ** 3
    elif kind == "zero":
        w = np.zeros((R, S), np.float32)
    else:
        w = np.full((R, S), 0.25, np.float32)
    return t, w


def test_linspace_is_the_stated_form():
    for n in range(1, 300):
        want = np.array([i * (1.0 / (n - 1)) for i in range(n)]) if n > 1 else np.array([0.0])
        if n > 1:
            want[-1] = 1.0
        assert np.array_equal(np.linspace(0.0, 1.0, n), want), n


def test_uniform_matches_the_library():
    from loma_nerf_b200 import _lib
    lib = _lib.load()
    for seed, q, s in [(0, 0, 0), (7, 123456, 4095), (2 ** 64 - 1, 2 ** 40, 17), (99, 640000 - 1, 191)]:
        assert Hs.uniform(seed, q, s) == lib.lnb_uniform(seed, q, s)


@pytest.mark.parametrize("S", [3, 4, 33, 64])
@pytest.mark.parametrize("n_fine", [1, 2, 31, 64])
@pytest.mark.parametrize("stratified", [False, True])
def test_against_the_paper_transcription(S, n_fine, stratified):
    # Every bin carries more than 1e-5 of the mass here.  The clamp d < 1e-5 -> 1 is discontinuous: with a lighter bin
    # next to u = 1 the paper's cdf, normalised before the sum, may end a rounding step above 1 and put u = 1 into that
    # bin instead of onto m_{S-2}; the rule's cdf ends at exactly 1.
    R = 12
    rng = np.random.default_rng(S * 100 + n_fine)
    t = np.sort(rng.uniform(2.0, 6.0, (R, S)), axis=1)
    w = rng.uniform(0.05, 1.0, (R, S)).astype(np.float32)
    got = Hs.sample_pdf_f64(t, w, n_fine, stratified=stratified, seed=5, ray0=40)
    u = Hs.sample_positions(R, n_fine, stratified, 5, 40)
    for r in range(R):
        x = paper_sample_pdf(0.5 * (t[r, 1:] + t[r, :-1]), w[r, 1:-1].astype(np.float64), u[r])
        want = np.sort(np.concatenate([t[r], x]))
        assert np.abs(got[r] - want).max() <= 1e-12


@pytest.mark.parametrize("kind", ["random", "zero", "uniform"])
@pytest.mark.parametrize("stratified", [False, True])
def test_rows_are_sorted_contain_t_and_stay_inside_the_bins(kind, stratified):
    R, S, n = 20, 64, 128
    t, w = _case(3, R, S, kind)
    out = Hs.sample_pdf_f64(t, w, n, stratified=stratified, seed=9)
    assert out.shape == (R, S + n)
    assert (np.diff(out, axis=1) >= 0).all()
    mids = 0.5 * (t[:, 1:] + t[:, :-1])
    for r in range(R):
        rest = list(out[r])
        for v in t[r]:
            rest.remove(v)                      # every coarse depth is in the row, once per occurrence
        x = np.array(rest)
        assert x.shape == (n,) and (x >= mids[r, 0]).all() and (x <= mids[r, -1]).all()


@pytest.mark.parametrize("kind", ["zero", "uniform"])
def test_flat_weights_space_samples_evenly(kind):
    R, S, n = 4, 33, 31
    t = np.broadcast_to(np.linspace(2.0, 6.0, S), (R, S)).copy()
    w = np.zeros((R, S), np.float32) if kind == "zero" else np.full((R, S), 0.3, np.float32)
    out = Hs.sample_pdf_f64(t, w, n)
    m0, m1 = 0.5 * (t[0, 0] + t[0, 1]), 0.5 * (t[0, -2] + t[0, -1])
    want = np.sort(np.concatenate([t[0], m0 + np.linspace(0, 1, n) * (m1 - m0)]))
    for r in range(R):
        assert np.abs(out[r] - want).max() <= 1e-12


@pytest.mark.parametrize("j", [0, 5, 30])
def test_one_hot_weight_pulls_the_samples_into_its_bin(j):
    R, S, n = 3, 33, 128
    t = np.broadcast_to(np.linspace(2.0, 6.0, S), (R, S)).copy()
    w = np.zeros((R, S), np.float32)
    w[:, j + 1] = 1.0                           # interior weight v_j: bin [m_j, m_{j+1}]
    out = Hs.sample_pdf_f64(t, w, n)
    mids = 0.5 * (t[0, 1:] + t[0, :-1])
    x = out[0][~np.isin(out[0], t[0])]
    outside = int(((x < mids[j]) | (x > mids[j + 1])).sum())
    # the other S-3 bins hold (S-3) 1e-5 / (1 + (S-2) 1e-5) of the mass; u = 0 and u = 1 land on m_0 and m_{S-2}
    assert outside <= 2 + int(np.ceil(n * (S - 3) * 1e-5)), outside


def test_u_one_gives_the_last_midpoint():
    R, S = 6, 17
    t, w = _case(11, R, S)
    out = Hs.sample_pdf_f64(t, w, 1, u=np.ones((R, 1)))
    mids_last = 0.5 * (t[:, -1] + t[:, -2])
    for r in range(R):
        x = out[r][~np.isin(out[r], t[r])]
        assert x.shape == (1,) and x[0] == mids_last[r]
