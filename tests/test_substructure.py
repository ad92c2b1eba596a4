"""CPU: the oracle of mmb_jet_substructure (N-subjettiness on exclusive kt / WTA_pt axes, energy correlation functions) on a
worked case, on the undefined cases, against a numpy fp64 brute-force statement of the definitions, and under the
symmetries the observables have."""
import numpy as np
import pytest

import substructure_oracle as so

WORKED = np.array([[[10.0, 0.0, 0.0], [9.0, 0.1, 0.0], [1.0, 1.5, 0.0]]], np.float32)   # A, B, C


def random_jets(g, B, N, lo=3, hi=128, straddle=True):
    """JetClass-like clouds: pt > 0 falling with the slot, eta / phi spread ~0.3 around the jet axis; some jets sit on
    phi = +-pi so that their particles straddle the wrap."""
    mult = g.integers(lo, hi + 1, B)
    mask = (np.arange(N)[None] < mult[:, None]).astype(np.uint8)
    x = np.empty((B, N, 3), np.float32)
    x[..., 0] = g.exponential(1.0, (B, N)) * 20.0 / (1.0 + np.arange(N)[None] * 0.1) + 0.01
    x[..., 1] = g.normal(0.0, 0.3, (B, N)) + g.uniform(-1.5, 1.5, (B, 1))
    centre = np.where(g.random((B, 1)) < (0.3 if straddle else 0.0), np.pi, g.uniform(-2.5, 2.5, (B, 1)))
    phi = g.normal(0.0, 0.3, (B, N)) + centre
    x[..., 2] = (phi + np.pi) % (2 * np.pi) - np.pi
    perm = np.argsort(g.random((B, N)), axis=1)   # used slots not a prefix
    return np.take_along_axis(x, perm[..., None], 1), np.take_along_axis(mask, perm, 1)


WORKED_ROW = [0.15, 0.0875, 0.0, 0.0875 / 0.15, 0.0, 0.0915, 0.0023625, 0.0023625 / 0.0915 ** 3]


def test_worked_case():
    # C goes to the beam first (d_CB = 1 < d_AB = 1.2656 < d_BC = 3.0625), so tau2 uses {A, B}; A and B then merge with A's
    # direction, so tau1 uses A.  R = 0.8, beta = 1.
    # the fp64 statement on the exact inputs and R (0.1 and 0.8 have no fp32 form) gives the worked numbers to 1e-12 ...
    exact = np.array([[10.0, 0.0, 0.0], [9.0, 0.1, 0.0], [1.0, 1.5, 0.0]])
    row, ax = so.numpy_jet(exact[:, 0], exact[:, 1], exact[:, 2], np.arange(3), fp32_params=False)
    np.testing.assert_allclose(row, WORKED_ROW, rtol=0, atol=1e-12)
    assert abs(row[3] - 0.58333) < 1e-5 and abs(row[7] - 3.08396) < 1e-5
    assert abs(row[1] - 0.05625) > 1e-3   # what tau2 would be without the beam step
    assert ax.tolist() == [0, 0, 1, 0, 1, 2]
    out, axes = so.jet_substructure(WORKED, np.ones((1, 3), np.uint8))
    assert axes[0].tolist() == [0, 0, 1, 0, 1, 2]
    # ... and the oracle, fed the fp32 inputs, returns them rounded to fp32 (eta_B and R move by ~1.5e-8 on the way in)
    np.testing.assert_allclose(out[0].astype(np.float64), WORKED_ROW, rtol=2e-7, atol=1e-12)


def test_undefined_jets():
    x = np.zeros((3, 8, 3), np.float32)
    mask = np.zeros((3, 8), np.uint8)
    x[0, :2] = WORKED[0, :2]
    mask[0, :2] = 1                         # two used particles
    x[1, :3] = WORKED[0]                    # three particles, none live
    x[2, :3] = WORKED[0]
    x[2, :3, 0] = [0.0, -1.0, 0.0]          # live but pt <= 0: none used
    mask[2, :3] = 1
    out, axes = so.jet_substructure(x, mask)
    assert np.isnan(out).all() and (axes == -1).all()


def test_live_particles_without_pt_change_nothing():
    g = np.random.default_rng(3)
    x, mask = random_jets(g, 40, 64, 3, 40)
    out, axes = so.jet_substructure(x, mask)
    x2, m2 = x.copy(), mask.copy()
    dead = (mask == 0)
    x2[..., 0] = np.where(dead, -np.abs(x2[..., 0]) * g.integers(0, 2, dead.shape), x2[..., 0])   # pt <= 0 ...
    m2[dead] = 1                                                                                  # ... on live slots
    out2, axes2 = so.jet_substructure(x2, m2)
    assert np.array_equal(axes, axes2)
    np.testing.assert_array_equal(out, out2)


@pytest.mark.parametrize("beta", [1.0, 2.0])
def test_oracle_matches_numpy_statement(beta):
    g = np.random.default_rng(7 + int(beta))
    B, N = 200, 128
    x, mask = random_jets(g, B, N)
    mult = (mask != 0).sum(1)
    assert mult.min() >= 3 and mult.max() > 100
    out, axes = so.jet_substructure(x, mask, beta=beta)
    want, wax = so.numpy_batch(x, mask, beta=beta)
    assert np.array_equal(axes, wax)
    # the oracle rounds its fp64 results to fp32 once
    np.testing.assert_allclose(out, want.astype(np.float32), rtol=1e-12 if beta == 1.0 else 2e-7, atol=1e-12)
    assert np.array_equal(np.isnan(out), np.isnan(want))


def _wrap(phi):
    return ((phi + np.pi) % (2 * np.pi) - np.pi).astype(np.float32)


def test_symmetries():
    g = np.random.default_rng(11)
    B, N = 60, 48
    x, mask = random_jets(g, B, N, 3, 48)
    out, axes = so.jet_substructure(x, mask)

    def same(o2, a2, slot_map=None, rtol=1e-5):
        mapped = axes if slot_map is None else np.take_along_axis(slot_map, axes.astype(np.int64), 1)
        for lo, hi in ((0, 1), (1, 3), (3, 6)):     # each axis set as a set of slots
            assert np.array_equal(np.sort(mapped[:, lo:hi], 1), np.sort(a2[:, lo:hi], 1))
        np.testing.assert_allclose(o2, out, rtol=rtol, atol=1e-6)

    shifted = x.copy()
    shifted[..., 1] += 0.75                                          # eta shift: dR unchanged
    same(*so.jet_substructure(shifted, mask))
    rotated = x.copy()
    rotated[..., 2] = _wrap(rotated[..., 2].astype(np.float64) + 2.9)   # phi rotation across +-pi
    same(*so.jet_substructure(rotated, mask))
    doubled = x.copy()
    doubled[..., 0] *= 2.0                                           # pt x 2: every d scales by 4, ratios stay
    same(*so.jet_substructure(doubled, mask), rtol=1e-6)
    perm = np.argsort(g.random((B, N)), axis=1)                      # slot permutation: axes follow their particles
    inv = np.argsort(perm, axis=1)
    same(*so.jet_substructure(np.take_along_axis(x, perm[..., None], 1), np.take_along_axis(mask, perm, 1)), slot_map=inv)
