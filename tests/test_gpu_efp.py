"""Energy flow polynomials on the device (mmb_energy_flow_polynomials): the kernel against the fp64 closed forms of
tests/efp_oracle.py, special jets, the stats path, efp1 = 2 e2 against jet_substructure, determinism, argument errors and the
JetClassHighLevelFeatures mirror (compute_efps, W1-EFP)."""
import numpy as np
import pytest
import torch

import efp_oracle as eo

DEV = "cuda:0"
REL = 1e-5
STATS = {"mean": [1.2, 0.0, 0.0], "std": [0.35, 0.2, 0.2]}


def batch(seed, B, N, mult=None, stats=True):
    """Standardised JetClass-like clouds: multiplicities ``mult`` (default normal(45, 18) clipped to [1, N]), live slots first."""
    g = np.random.default_rng(seed)
    if mult is None:
        mult = np.clip(np.rint(g.normal(45, 18, B)), 1, N).astype(int)
    mask = (np.arange(N)[None] < np.asarray(mult)[:, None]).astype(np.uint8)
    x = g.normal(0, 1, (B, N, 3)).astype(np.float32)
    if not stats:
        x = x * np.float32(STATS["std"]) + np.float32(STATS["mean"])
    return x, mask


def efps(x, mask, stats=None, beta=1.0):
    from multimodal_particles_b200.observables import energy_flow_polynomials
    return energy_flow_polynomials(torch.from_numpy(x).to(DEV), torch.from_numpy(mask).to(DEV), stats, beta).cpu().numpy()


def check(x, mask, stats=STATS, beta=1.0):
    got = efps(x, mask, stats, beta)
    want = eo.numpy_batch(x, mask, stats, beta)
    np.testing.assert_allclose(got, want, rtol=REL, atol=0)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["jetclass_4096x128", "n30", "n200", "n256_all_live", "beta2"])
def test_kernel_matches_closed_forms(case):
    if case == "jetclass_4096x128":
        check(*batch(1, 4096, 128))
    elif case == "n30":
        check(*batch(2, 512, 30))
    elif case == "n200":
        check(*batch(3, 96, 200, mult=np.random.default_rng(3).integers(150, 201, 96)))
    elif case == "n256_all_live":
        check(*batch(4, 24, 256, mult=[256] * 24))
    else:
        check(*batch(5, 1024, 128), beta=2.0)


@pytest.mark.gpu
def test_empty_and_single_particle_jets():
    x, mask = batch(6, 8, 64, mult=[0, 1, 1, 2, 3, 64, 0, 33], stats=False)
    x[7, :, 0] = -1.0                                  # every particle of jet 7 has pt <= 0: no used particle
    x[7, 5, 0] = 2.0                                   # ... but one
    got = efps(x, mask)
    assert np.isnan(got[[0, 6]]).all()
    assert (got[[1, 2, 7]] == 0.0).all()
    np.testing.assert_allclose(got, eo.numpy_batch(x, mask), rtol=REL, atol=0)


@pytest.mark.gpu
def test_stats_path_equals_physical_input():
    x, mask = batch(7, 300, 128)
    phys = x * np.float32(STATS["std"]) + np.float32(STATS["mean"])
    assert efps(x, mask, STATS).tobytes() == efps(phys, mask, None).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("beta", [1.0, 2.0])
def test_efp1_is_twice_e2_of_jet_substructure(beta):
    from multimodal_particles_b200.observables import jet_substructure
    x, mask = batch(8, 2048, 128)
    sub = jet_substructure(torch.from_numpy(x).to(DEV), torch.from_numpy(mask).to(DEV), STATS, beta=beta).cpu().numpy()
    got = efps(x, mask, STATS, beta)
    defined = ~np.isnan(sub[:, 5])
    assert defined.sum() > 1900
    np.testing.assert_allclose(got[defined, 0], 2 * sub[defined, 5].astype(np.float64), rtol=1e-5)


@pytest.mark.gpu
def test_bit_identical_across_calls():
    x, mask = batch(9, 4096, 128)
    a, b = efps(x, mask, STATS), efps(x, mask, STATS)
    assert a.tobytes() == b.tobytes()


@pytest.mark.gpu
def test_argument_errors_are_codes():
    from multimodal_particles_b200 import _native
    from multimodal_particles_b200.observables import energy_flow_polynomials
    with pytest.raises(_native.MmbError):
        energy_flow_polynomials(torch.zeros(2, 8, 3), torch.ones(2, 8, dtype=torch.uint8))            # host tensors
    with pytest.raises(_native.MmbError):
        energy_flow_polynomials(torch.zeros(2, 257, 3, device=DEV), torch.ones(2, 257, dtype=torch.uint8, device=DEV))   # N > 256
    with pytest.raises(_native.MmbError):
        energy_flow_polynomials(torch.zeros(2, 8, 3, device=DEV), torch.ones(2, 8, dtype=torch.uint8, device=DEV), beta=0.0)
    lib = _native.load()
    assert lib.mmb_energy_flow_polynomials(None, None, None, None, 1, 8, 1.0, None, None) == -1


def _clouds(seed, B=768, N=128):
    from multimodal_particles_b200 import HybridState
    from multimodal_particles_b200.observables import JetClassHighLevelFeatures, ParticleClouds
    g = np.random.default_rng(seed)
    mult = np.clip(np.rint(g.normal(45, 18, B)), 0, N).astype(int)
    mask = (np.arange(N)[None] < mult[:, None]).astype(np.int64)
    xs = g.normal(0, 1, (B, N, 3)).astype(np.float32) * mask[..., None]
    k = g.integers(0, 8, (B, N)) * mask
    state = HybridState(None, torch.from_numpy(xs), torch.from_numpy(k)[..., None], torch.from_numpy(mask)[..., None])
    pc = ParticleClouds(dataset=state)
    pc.postprocess(input_continuous="standardize", input_discrete="tokens", stats=STATS)
    jets = JetClassHighLevelFeatures(pc)
    jets.compute_efps()
    return jets, pc


@pytest.mark.gpu
def test_mirror_class_compute_efps_and_w1_efp():
    from multimodal_particles_b200.observables import EFP_COLUMNS
    (a, pa), (b, _) = _clouds(1), _clouds(2, B=640)
    x = pa.continuous.cpu().numpy()
    m = pa.mask.cpu().numpy().reshape(x.shape[0], -1)
    want = eo.numpy_batch(x, m)
    want = want[~np.isnan(want[:, 0])]
    for i, name in enumerate(EFP_COLUMNS):
        np.testing.assert_allclose(getattr(a, name).cpu().numpy(), want[:, i], rtol=REL, atol=0)
    got = a.wasserstein1d(b, EFP_COLUMNS[1:])                                   # W1-EFP
    assert list(got) == list(EFP_COLUMNS[1:])
    for f in EFP_COLUMNS[1:]:
        assert got[f] == pytest.approx(a.Wassertein1D(f, b), rel=1e-9, abs=1e-12), f
    with pytest.raises(NotImplementedError):
        a.substructure()
