"""JetNet's W1-M, W1-P and W1-EFP (DESIGN.md §4.6e) on the CPU: a numpy statement of the drawn sample (expansion, duplicates,
mask order) and of W1 per draw against scipy, hand cases, and the aggregation over the draws (``observables.w1_summary``)."""
import numpy as np
import pytest
import scipy.stats

from multimodal_particles_b200.observables import PARTICLE_COLUMNS, w1_summary


def drawn_sample(x, mask, idx):
    """The sample of one draw: the used slots of the jets x[idx] ([n, P, F]; mask [n, P] or None), in draw order and slot order."""
    F = x.shape[-1]
    parts = [x[j][mask[j] != 0] if mask is not None else x[j] for j in idx]
    return np.concatenate(parts).reshape(-1, F) if parts else np.zeros((0, F), x.dtype)


def merged_w1(x, y):
    """W1 = sum_k |i_k m' - j_k n'| (z_{k+1} - z_k) / (n' m') over the finite values, in fp64 (DESIGN.md §4.6c)."""
    x = np.sort(np.asarray(x, np.float64)[np.isfinite(x)])
    y = np.sort(np.asarray(y, np.float64)[np.isfinite(y)])
    n, m = len(x), len(y)
    if n == 0 or m == 0:
        return float("nan")
    z = np.sort(np.concatenate([x, y]))
    i = np.searchsorted(x, z[:-1], side="right").astype(np.int64)
    j = np.searchsorted(y, z[:-1], side="right").astype(np.int64)
    return float(np.sum(np.abs(i * m - j * n) * np.diff(z)) / (n * m))


def drawn_w1(x, idx_x, y, idx_y, mask_x=None, mask_y=None):
    """[draws, F]: W1 per draw and feature between the drawn samples."""
    out = np.empty((len(idx_x), x.shape[-1]))
    for t in range(len(idx_x)):
        a, b = drawn_sample(x, mask_x, idx_x[t]), drawn_sample(y, mask_y, idx_y[t])
        out[t] = [merged_w1(a[:, c], b[:, c]) for c in range(x.shape[-1])]
    return out


def _clouds(g, n, P, F):
    x = g.normal(0, 1, (n, P, F)).astype(np.float32)
    mask = (np.arange(P)[None, :] < g.integers(0, P + 1, n)[:, None]).astype(np.uint8)
    return x, mask


def test_drawn_sample_expansion_order_and_duplicates():
    x = np.arange(3 * 4 * 2, dtype=np.float32).reshape(3, 4, 2)
    mask = np.array([[1, 0, 1, 0], [0, 0, 0, 0], [0, 1, 1, 1]], np.uint8)
    got = drawn_sample(x, mask, [2, 0, 1, 2])
    want = np.concatenate([x[2, [1, 2, 3]], x[0, [0, 2]], x[2, [1, 2, 3]]])
    np.testing.assert_array_equal(got, want)
    assert drawn_sample(x, None, [1]).shape == (4, 2)
    assert drawn_sample(x, mask, [1, 1]).shape == (0, 2)


def test_drawn_w1_matches_scipy():
    g = np.random.default_rng(3)
    x, mx = _clouds(g, 300, 16, 3)
    y, my = _clouds(g, 200, 16, 3)
    y[..., 0] += 0.25
    ix, iy = g.integers(0, 300, (4, 120)), g.integers(0, 200, (4, 120))
    got = drawn_w1(x, ix, y, iy, mx, my)
    for t in range(4):
        a, b = drawn_sample(x, mx, ix[t]).astype(np.float64), drawn_sample(y, my, iy[t]).astype(np.float64)
        for c in range(3):
            assert got[t, c] == pytest.approx(scipy.stats.wasserstein_distance(a[:, c], b[:, c]), rel=1e-12, abs=1e-14)


def test_constant_shift_gives_the_shift():
    g = np.random.default_rng(4)
    x, mx = _clouds(g, 100, 8, 3)
    x = np.round(x * 64) / 64                                   # dyadic values and shift: x + 0.5 and every difference are exact
    idx = g.integers(0, 100, (3, 50))
    got = drawn_w1(x, idx, x + np.float32(0.5), idx, mx, mx)
    assert np.all(got == 0.5)


def test_sample_against_itself_is_zero():
    g = np.random.default_rng(5)
    x, mx = _clouds(g, 100, 8, 2)
    idx = g.integers(0, 100, (3, 40))
    assert np.all(drawn_w1(x, idx, x, idx, mx, mx) == 0.0)


def test_jet_drawn_twice_counts_twice():
    x = np.array([[[0.0]], [[1.0]]], np.float32)     # two one-particle jets
    y = np.array([[[0.0]]], np.float32)
    assert drawn_w1(x, [[0, 0, 1]], y, [[0, 0, 0]])[0, 0] == pytest.approx(1 / 3, rel=1e-15)
    assert drawn_w1(x, [[0, 1, 1]], y, [[0, 0, 0]])[0, 0] == pytest.approx(2 / 3, rel=1e-15)


def test_no_used_particle_is_nan():
    x = np.zeros((2, 3, 1), np.float32)
    mask = np.array([[0, 0, 0], [1, 1, 0]], np.uint8)
    got = drawn_w1(x, [[0, 0], [1, 0]], x, [[1, 1], [1, 1]], mask, mask)
    assert np.isnan(got[0, 0]) and got[1, 0] == 0.0


def test_aggregation_rules():
    vals = np.array([[1.0, 2.0], [3.0, 4.0], [5.0, 9.0]])
    mean, std = w1_summary(vals)
    means, stds = vals.mean(0), np.sqrt(((vals - vals.mean(0)) ** 2).mean(0))   # np.std with ddof = 0
    assert mean == pytest.approx(means.mean(), rel=1e-15)
    assert std == pytest.approx(np.sqrt((stds ** 2).sum()), rel=1e-15)   # np.linalg.norm of the per-feature stds
    m, s = w1_summary(vals, average=False)
    np.testing.assert_allclose(m, means, rtol=1e-15)
    np.testing.assert_allclose(s, stds, rtol=1e-15)
    one = w1_summary(vals[:, :1])
    assert one == (pytest.approx(3.0), pytest.approx(np.sqrt(8 / 3)))
    nan = w1_summary(np.array([[1.0, 2.0], [np.nan, 4.0]]), average=False)   # a draw with no used particle poisons its feature
    assert np.isnan(nan[0][0]) and np.isnan(nan[1][0]) and nan[0][1] == 3.0 and nan[1][1] == 1.0
    assert PARTICLE_COLUMNS == ("pt", "eta_rel", "phi_rel")
