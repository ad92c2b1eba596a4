"""Every EFP of degree <= 4 on the device (mmb_energy_flow_polynomials_d4): the kernel against the fp64 closed forms of
tests/efp_d4_oracle.py, bit-identity of the columns it shares with mmb_energy_flow_polynomials, special jets, the stats path,
determinism, argument errors, and JetNet's FPD / KPD on these features in the sharded generation run."""
import ctypes

import numpy as np
import pytest
import torch

import efp_d4_oracle as do
from pipeline_lib import one_gpu_run, two_gpu_run

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


def run(fn, x, mask, stats=None, beta=1.0):
    return fn(torch.from_numpy(x).to(DEV), torch.from_numpy(mask).to(DEV), stats, beta).cpu().numpy()


def efps_d4(x, mask, stats=None, beta=1.0):
    from multimodal_particles_b200.observables import energy_flow_polynomials_d4
    return run(energy_flow_polynomials_d4, x, mask, stats, beta)


CASES = {"jetclass_4096x128": lambda: batch(1, 4096, 128),
         "n30": lambda: batch(2, 512, 30),
         "n200": lambda: batch(3, 96, 200, mult=np.random.default_rng(3).integers(150, 201, 96)),
         "n256_all_live": lambda: batch(4, 24, 256, mult=[256] * 24),
         "beta2": lambda: batch(5, 1024, 128)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_kernel_matches_closed_forms_and_shares_columns_bit_for_bit(case):
    from multimodal_particles_b200.observables import EFP_COLUMNS, EFP_D4_COLUMNS, energy_flow_polynomials
    x, mask = CASES[case]()
    beta = 2.0 if case == "beta2" else 1.0
    got = efps_d4(x, mask, STATS, beta)
    assert got.shape == (x.shape[0], 36) and got.dtype == np.float32
    np.testing.assert_allclose(got, do.numpy_batch(x, mask, STATS, beta), rtol=REL, atol=0)
    old = run(energy_flow_polynomials, x, mask, STATS, beta)
    shared = [EFP_D4_COLUMNS.index(c) for c in EFP_COLUMNS]
    assert np.ascontiguousarray(got[:, shared]).tobytes() == old.tobytes()


@pytest.mark.gpu
def test_empty_and_single_particle_jets():
    x, mask = batch(6, 8, 64, mult=[0, 1, 1, 2, 3, 64, 0, 33], stats=False)
    x[7, :, 0] = -1.0                                  # every particle of jet 7 has pt <= 0: no used particle
    x[7, 5, 0] = 2.0                                   # ... but one
    got = efps_d4(x, mask)
    assert np.isnan(got[[0, 6]]).all()
    for b in (1, 2, 7):
        assert got[b].tolist() == [1.0] + [0.0] * 35
    np.testing.assert_allclose(got, do.numpy_batch(x, mask), rtol=REL, atol=0)


@pytest.mark.gpu
def test_stats_path_equals_physical_input_and_calls_are_bit_identical():
    x, mask = batch(7, 300, 128)
    phys = x * np.float32(STATS["std"]) + np.float32(STATS["mean"])
    assert efps_d4(x, mask, STATS).tobytes() == efps_d4(phys, mask, None).tobytes()
    x, mask = batch(9, 4096, 128)
    assert efps_d4(x, mask, STATS).tobytes() == efps_d4(x, mask, STATS).tobytes()


@pytest.mark.gpu
def test_fpd_features_are_the_named_columns():
    from multimodal_particles_b200.observables import EFP_D4_COLUMNS, FPD_EFP_COLUMNS, jetnet_fpd_features
    x, mask = batch(10, 500, 128)
    xd, md = torch.from_numpy(x).to(DEV), torch.from_numpy(mask).to(DEV)
    got = jetnet_fpd_features(xd, md, STATS).cpu().numpy()
    assert got.shape == (500, len(FPD_EFP_COLUMNS))
    pick = [EFP_D4_COLUMNS.index(c) for c in FPD_EFP_COLUMNS]
    assert got.tobytes() == np.ascontiguousarray(efps_d4(x, mask, STATS)[:, pick]).tobytes()


@pytest.mark.gpu
def test_argument_errors_are_codes():
    from multimodal_particles_b200 import _native
    from multimodal_particles_b200.observables import energy_flow_polynomials_d4
    with pytest.raises(_native.MmbError):
        energy_flow_polynomials_d4(torch.zeros(2, 8, 3), torch.ones(2, 8, dtype=torch.uint8))            # host tensors
    with pytest.raises(_native.MmbError):
        energy_flow_polynomials_d4(torch.zeros(2, 257, 3, device=DEV), torch.ones(2, 257, dtype=torch.uint8, device=DEV))   # N > 256
    with pytest.raises(_native.MmbError):
        energy_flow_polynomials_d4(torch.zeros(2, 8, 3, device=DEV), torch.ones(2, 8, dtype=torch.uint8, device=DEV), beta=0.0)
    lib = _native.load()
    assert lib.mmb_energy_flow_polynomials_d4(None, None, None, None, 1, 8, 1.0, None, None) == -1
    x, m = torch.zeros(2, 8, 3, device=DEV), torch.ones(2, 8, dtype=torch.uint8, device=DEV)
    out = torch.empty(2, 36, device=DEV)
    mean = (ctypes.c_float * 3)(0.0, 0.0, 0.0)
    assert lib.mmb_energy_flow_polynomials_d4(x.data_ptr(), m.data_ptr(), mean, None, 2, 8, 1.0, out.data_ptr(), None) == -1
    assert lib.mmb_energy_flow_polynomials_d4(x.data_ptr(), m.data_ptr(), None, None, -1, 8, 1.0, out.data_ptr(), None) == -1


# ---- pipeline ----------------------------------------------------------------------------------------------------------------
TOTAL, REF_JETS = 3 * 16384, 20000
NEW_KEYS = {"jetnet_fpd", "jetnet_kpd", "jetnet_fpd_reference_jets", "jetnet_fpd_seconds"}


def _same_except_time(a, b):
    assert set(a) == set(b)
    for key, val in a.items():
        if key != "value" and not key.endswith("seconds"):
            assert b[key] == val, key


@pytest.mark.gpu
def test_sharded_run_jetnet_fpd_kpd():
    import bench
    from multimodal_particles_b200.observables import FPD_EFP_COLUMNS, fpd, kpd
    from multimodal_particles_b200.pipeline import STATS as PIPE_STATS
    from multimodal_particles_b200.pipeline import reference_fpd_features, reference_observables
    dev_ = torch.device(DEV)
    cfg, model = bench.build_model(dev_)
    ref = reference_fpd_features(model, cfg, REF_JETS, dev_, n_particles=bench.N_PART)
    assert ref.shape == (REF_JETS, len(FPD_EFP_COLUMNS)) and ref.dtype == torch.float32
    base = one_gpu_run(model, cfg, TOTAL, 16384)
    big = one_gpu_run(model, cfg, TOTAL, 16384, fpd_reference=ref)
    small = one_gpu_run(model, cfg, TOTAL, 4096, fpd_reference=ref)
    assert set(big) - set(base) == NEW_KEYS
    _same_except_time(base, {k: v for k, v in big.items() if k not in NEW_KEYS})      # the d <= 4 pass changes nothing else
    for key in ("jetnet_fpd", "jetnet_kpd"):
        assert big[key] == small[key], key                                            # bit-identical for any micro-batch
    assert big["jetnet_fpd_reference_jets"] == REF_JETS and big["jetnet_fpd_seconds"] > 0
    # the same jets, collected outside the pipeline
    same = reference_fpd_features(model, cfg, TOTAL, dev_, n_particles=bench.N_PART, jet_offset=0)
    assert list(fpd(ref, same)) == big["jetnet_fpd"] and list(kpd(ref, same)) == big["jetnet_kpd"]
    # the existing EFP metrics are the same with and without the d <= 4 features
    w1_ref = reference_observables(model, cfg, REF_JETS, dev_, n_particles=bench.N_PART, efp=True)
    efp_plain = one_gpu_run(model, cfg, TOTAL, 16384, w1_reference=w1_ref, efp=True)
    efp_both = one_gpu_run(model, cfg, TOTAL, 16384, w1_reference=w1_ref, efp=True, fpd_reference=ref)
    _same_except_time(efp_plain, {k: v for k, v in efp_both.items() if k not in NEW_KEYS})
    assert efp_both["jetnet_fpd"] == big["jetnet_fpd"] and efp_both["jetnet_kpd"] == big["jetnet_kpd"]
    # an independent reference of the same model is within a few errors of 0; one with 25 % wider jets is far
    (fv, fe), (kv, ke) = big["jetnet_fpd"], big["jetnet_kpd"]
    assert fv <= 5 * fe + 1e-9 and abs(kv) <= 5 * ke + 1e-9, (big["jetnet_fpd"], big["jetnet_kpd"])
    shifted = dict(PIPE_STATS, std=[PIPE_STATS["std"][0], 0.25, 0.25])
    ref_shift = reference_fpd_features(model, cfg, REF_JETS, dev_, n_particles=bench.N_PART, stats=shifted)
    far = one_gpu_run(model, cfg, TOTAL, 16384, fpd_reference=ref_shift)
    assert far["jetnet_fpd"][0] > 10 * (fv + fe), (far["jetnet_fpd"], big["jetnet_fpd"])
    assert far["jetnet_kpd"][0] > 10 * (abs(kv) + ke), (far["jetnet_kpd"], big["jetnet_kpd"])


def _two_gpu_kwargs(model, cfg, dev_):
    import bench
    from multimodal_particles_b200.pipeline import reference_fpd_features
    return dict(fpd_reference=reference_fpd_features(model, cfg, REF_JETS, dev_, n_particles=bench.N_PART))


@pytest.mark.gpu
def test_two_gpu_jetnet_fpd_kpd_equal_one_gpu(tmp_path):
    """FPD and KPD on the d <= 4 EFPs of a two-GPU run (uneven shards) are bit-identical to the one-GPU run; needs two GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import bench
    two = two_gpu_run(tmp_path, TOTAL + 5, _two_gpu_kwargs, ("jetnet_fpd", "jetnet_kpd"))
    dev_ = torch.device(DEV)
    cfg, model = bench.build_model(dev_)
    one = one_gpu_run(model, cfg, TOTAL + 5, 16384, **_two_gpu_kwargs(model, cfg, dev_))
    assert two["jetnet_fpd"] == one["jetnet_fpd"] and two["jetnet_kpd"] == one["jetnet_kpd"]
