"""CPU: the numpy statements of tests/efp_oracle.py — EFP closed forms against the literal sum over index tuples and worked jets,
their symmetries and pt selection, efp1 = 2 e2, and the FPD / KPD statements against scipy's sqrtm and an explicit Gram sum."""
import numpy as np
import pytest
import scipy.linalg

import efp_oracle as eo
import substructure_oracle as so


def random_jet(g, n):
    return g.uniform(0.1, 5.0, n), g.normal(0, 0.4, n), g.normal(0, 0.4, n)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 12])
@pytest.mark.parametrize("beta", [1.0, 2.0, 0.5])
def test_closed_forms_equal_brute_force(n, beta):
    g = np.random.default_rng(n * 10 + int(beta * 2))
    jet = random_jet(g, n)
    np.testing.assert_allclose(eo.closed_forms(*jet, beta), eo.brute_force(*jet, beta), rtol=1e-12, atol=1e-15)


def test_two_particle_jet():
    # z = (1/4, 3/4), theta = 0.5: efp1 = 2 z1 z2 t, paw = 0 (no triangle), square = mid2 = end2 = 2 z1^2 z2^2 t^4,
    # star2 = z1 z2 t^4 (z1^2 + z2^2)
    z1, z2, t = 0.25, 0.75, 0.5
    got = eo.closed_forms(np.array([1.0, 3.0]), np.array([0.1, 0.6]), np.array([-0.2, -0.2]))
    c = 2 * z1 ** 2 * z2 ** 2 * t ** 4
    np.testing.assert_allclose(got, [2 * z1 * z2 * t, c, 0.0, c, c, z1 * z2 * t ** 4 * (z1 ** 2 + z2 ** 2)], rtol=1e-12, atol=1e-16)


def test_equilateral_three_particle_jet():
    # three equal-pt particles at mutual distance L: efp1 = 2L/3, square = 2L^4/9, paw = 4L^4/27, mid2 = end2 = star2 = 8L^4/27
    L = 0.3
    got = eo.closed_forms(np.ones(3) * 2.0, np.array([0.0, L, L / 2]), np.array([0.0, 0.0, L * np.sqrt(3) / 2]))
    np.testing.assert_allclose(got, [2 * L / 3, 2 * L ** 4 / 9, 4 * L ** 4 / 27, 8 * L ** 4 / 27, 8 * L ** 4 / 27, 8 * L ** 4 / 27],
                               rtol=1e-12)


def test_empty_and_single_particle():
    assert np.isnan(eo.closed_forms(np.zeros(0), np.zeros(0), np.zeros(0))).all()
    assert eo.closed_forms(np.array([2.0]), np.array([0.3]), np.array([1.0])).tolist() == [0.0] * 6


def test_permutation_eta_shift_and_phi_wrap():
    g = np.random.default_rng(7)
    pt, eta, phi = random_jet(g, 40)
    phi = np.clip(phi, -0.9, 0.9)
    base = eo.closed_forms(pt, eta, phi)
    p = g.permutation(40)
    np.testing.assert_allclose(eo.closed_forms(pt[p], eta[p], phi[p]), base, rtol=1e-12)
    np.testing.assert_allclose(eo.closed_forms(pt, eta + 1.7, phi), base, rtol=1e-10)
    rot = phi + 2.8                                            # straddles +pi: wrapped differences are unchanged
    rot = np.where(rot > np.pi, rot - 2 * np.pi, rot)
    assert (rot > 0).any() and (rot < 0).any()
    np.testing.assert_allclose(eo.closed_forms(pt, eta, rot), base, rtol=1e-10)


def test_non_positive_pt_is_ignored():
    g = np.random.default_rng(8)
    B, N = 6, 20
    x = np.stack([g.uniform(0.1, 3, (B, N)), g.normal(0, 0.3, (B, N)), g.normal(0, 0.3, (B, N))], -1).astype(np.float32)
    mask = np.ones((B, N), np.uint8)
    mask[:, 15:] = 0
    x2 = x.copy()
    x2[:, 10:12, 0] = np.array([0.0, -1.0], np.float32)          # pt <= 0: not used
    x2[:, 15:, :] = 9.0                                         # masked: not used
    keep = np.ones(N, bool)
    keep[10:12] = False
    keep[15:] = False
    want = np.array([eo.closed_forms(*[c.astype(np.float64) for c in (x[b, keep, 0], x[b, keep, 1], x[b, keep, 2])]) for b in range(B)])
    np.testing.assert_allclose(eo.numpy_batch(x2, mask), want, rtol=1e-12)


def test_efp1_is_twice_e2():
    g = np.random.default_rng(9)
    for n in (3, 17, 60):
        for beta in (1.0, 2.0):
            pt, eta, phi = random_jet(g, n)
            row, _ = so.numpy_jet(pt, eta, phi, np.arange(n), beta=beta, fp32_params=False)
            assert eo.closed_forms(pt, eta, phi, beta)[0] == pytest.approx(2 * row[5], rel=1e-12)


def test_frechet_statement_matches_sqrtm():
    g = np.random.default_rng(10)
    for d in (1, 5, 12):
        a = g.normal(0, 1, (400, d)) @ g.normal(0, 1, (d, d))
        b = g.normal(0.2, 1, (300, d)) @ g.normal(0, 1, (d, d))
        (m1, s1), (m2, s2) = eo.gaussian(a), eo.gaussian(b)
        covmean = scipy.linalg.sqrtm(s1 @ s2).real
        want = (m1 - m2) @ (m1 - m2) + np.trace(s1) + np.trace(s2) - 2 * np.trace(covmean)
        assert eo.frechet_distance(m1, s1, m2, s2) == pytest.approx(want, rel=1e-8, abs=1e-10)
        assert eo.frechet_distance(m1, s1, m1, s1) == pytest.approx(0.0, abs=1e-9)


def test_mmd_statement_matches_explicit_sum():
    g = np.random.default_rng(11)
    B, d = 25, 4
    X, Y = g.normal(0, 1, (B, d)), g.normal(0.3, 1, (B, d))
    k = lambda u, v: (u @ v / d + 1.0) ** 3
    sxx = sum(k(X[i], X[j]) for i in range(B) for j in range(B) if i != j)
    syy = sum(k(Y[i], Y[j]) for i in range(B) for j in range(B) if i != j)
    sxy = sum(k(X[i], Y[j]) for i in range(B) for j in range(B))
    want = (sxx + syy) / (B * (B - 1)) - 2 * sxy / B ** 2
    assert eo.mmd_unbiased(X, Y, degree=3) == pytest.approx(want, rel=1e-12)
