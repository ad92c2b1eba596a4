"""FPD and KPD on the device: mmb_sampled_moments / mmb_kpd_mmd against the numpy statements of tests/efp_oracle.py on the same
injected draws, determinism, the metrics' sensitivity, and the EFP metrics of the sharded generation run."""
import numpy as np
import pytest
import torch

import efp_oracle as eo
from pipeline_lib import one_gpu_run, two_gpu_run

DEV = "cuda:0"


def law(g, n, d=5):
    """Positive, correlated, skewed features of a few units (EFP-like after the max normalisation)."""
    base = g.normal(0, 1, (n, d))
    base[:, 1] = 0.8 * base[:, 0] + 0.6 * base[:, 1]
    return (np.abs(np.linspace(1.0, 3.0, d) + 0.1 * base) + 0.02 * g.gamma(2.0, 1.0, (n, d))).astype(np.float32)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [5, 40, 64])
def test_sampled_moments_and_frechet_match_numpy(d):
    from multimodal_particles_b200.observables import frechet_distances, sampled_moments
    g = np.random.default_rng(d)
    wide = law(g, 30000, d + 3)
    real = wide[:, :d]                                        # strided rows: the kernel reads a view with ldx = d + 3
    gen = law(g, 25000, d) * np.float32(1.02)
    scale = (1.0 / np.abs(real).max(0)).astype(np.float32)
    draws, rows = 4, 3001
    ir, ig = g.integers(0, len(real), (draws, rows)), g.integers(0, len(gen), (draws, rows))
    sums, sumsq = sampled_moments(dev(wide)[:, :d], dev(ir), dev(scale))
    for t in range(draws):
        r = eo.draw_rows(real, ir[t], scale)
        np.testing.assert_allclose(sums[t].cpu().numpy(), r.sum(0), rtol=1e-12)
        np.testing.assert_allclose(sumsq[t].cpu().numpy(), r.T @ r, rtol=1e-12)
    fd = frechet_distances(dev(wide)[:, :d], dev(gen), dev(ir), dev(ig), dev(scale)).cpu().numpy()
    for t in range(draws):
        want = eo.frechet_distance(*eo.gaussian(eo.draw_rows(real, ir[t], scale)), *eo.gaussian(eo.draw_rows(gen, ig[t], scale)))
        assert fd[t] == pytest.approx(want, rel=1e-9), t
    again = frechet_distances(dev(wide)[:, :d], dev(gen), dev(ir), dev(ig), dev(scale)).cpu().numpy()
    assert again.tobytes() == fd.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("d,B,degree", [(5, 700, 4), (5, 64, 4), (64, 300, 3), (2, 2, 4)])
def test_kpd_mmd_matches_numpy(d, B, degree):
    from multimodal_particles_b200.observables import kpd_mmd
    g = np.random.default_rng(B + d)
    real, gen = law(g, 5000, d), law(g, 4000, d) * np.float32(1.03)
    scale = (1.0 / np.abs(real).max(0)).astype(np.float32)
    batches = 3
    ir, ig = g.integers(0, len(real), (batches, B)), g.integers(0, len(gen), (batches, B))
    got = kpd_mmd(dev(real), dev(gen), dev(ir), dev(ig), dev(scale), degree).cpu().numpy()
    for t in range(batches):
        want = eo.mmd_unbiased(eo.draw_rows(real, ir[t], scale), eo.draw_rows(gen, ig[t], scale), degree)
        assert got[t] == pytest.approx(want, abs=1e-10), t
    again = kpd_mmd(dev(real), dev(gen), dev(ir), dev(ig), dev(scale), degree).cpu().numpy()
    assert again.tobytes() == got.tobytes()


@pytest.mark.gpu
def test_argument_errors_are_codes():
    from multimodal_particles_b200 import _native
    from multimodal_particles_b200.observables import fpd, kpd_mmd, sampled_moments
    lib = _native.load()
    assert lib.mmb_kpd_mmd_workspace_bytes(1, 1, 5) == 0 and lib.mmb_kpd_mmd_workspace_bytes(1, 100, 65) == 0
    assert lib.mmb_kpd_mmd_workspace_bytes(2, 100, 5) > 0
    x = torch.zeros(10, 5, device=DEV)
    i = torch.zeros(2, 4, dtype=torch.int32, device=DEV)
    with pytest.raises(_native.MmbError):
        sampled_moments(torch.zeros(10, 5), i)                                     # host tensor
    with pytest.raises(_native.MmbError):
        sampled_moments(torch.zeros(10, 65, device=DEV), i)                        # d > 64
    with pytest.raises(_native.MmbError):
        kpd_mmd(x, x, i[:, :1], i[:, :1])                                          # B < 2
    with pytest.raises(_native.MmbError):
        kpd_mmd(x, x, i, i, degree=0)
    ws = torch.empty(lib.mmb_kpd_mmd_workspace_bytes(2, 4, 5), dtype=torch.uint8, device=DEV)
    out = torch.empty(2, dtype=torch.float64, device=DEV)
    p = lambda t: None if t is None else t.data_ptr()
    s = torch.cuda.current_stream().cuda_stream
    assert lib.mmb_kpd_mmd(p(x), 5, 10, p(x), 5, 10, 5, None, p(i), p(i), 2, 4, 4, p(out), p(ws), ws.numel() - 1, s) == -3
    assert lib.mmb_kpd_mmd(p(x), 4, 10, p(x), 5, 10, 5, None, p(i), p(i), 2, 4, 4, p(out), p(ws), ws.numel(), s) == -1
    assert lib.mmb_sampled_moments(p(x), 5, 10, 5, None, p(i), 2, 0, p(out), p(out), s) == -1
    with pytest.raises(ValueError):
        fpd(torch.full((10, 5), float("nan"), device=DEV), x)


def _metrics(g_real, g_gen, transform=None, seed=42):
    from multimodal_particles_b200.observables import fpd, kpd
    real, gen = law(g_real, 60000), law(g_gen, 60000)
    if transform is not None:
        gen = transform(gen)
    return fpd(dev(real), dev(gen), seed=seed), kpd(dev(real), dev(gen), seed=seed)


@pytest.mark.gpu
def test_metrics_have_teeth():
    same = [_metrics(np.random.default_rng(100 + s), np.random.default_rng(200 + s), seed=s) for s in range(3)]
    f_floor = max(f[0] + f[1] for f, _ in same)
    k_floor = max(abs(k[0]) + k[1] for _, k in same)

    def shift(a):
        a = a.copy()
        a[:, 0] *= np.float32(1.05)
        return a

    def swap(a):
        return np.ascontiguousarray(a[:, [0, 2, 1, 3, 4]])

    for name, tr in (("shift", shift), ("swap", swap)):
        (fv, fe), (kv, ke) = _metrics(np.random.default_rng(100), np.random.default_rng(200), tr)
        assert fv > 10 * f_floor and fv > 5 * fe, (name, fv, fe, f_floor)
        assert kv > 10 * k_floor and kv > 5 * ke, (name, kv, ke, k_floor)


# ---- pipeline ----------------------------------------------------------------------------------------------------------------
TOTAL, REF_JETS = 3 * 16384, 20000
METRIC_KEYS = ("w1", "w1_used", "fpd", "kpd")


@pytest.mark.gpu
def test_sharded_run_efp_metrics():
    import bench
    from multimodal_particles_b200.observables import EFP_COLUMNS, fpd, kpd
    from multimodal_particles_b200.pipeline import reference_observables, w1_columns
    dev_ = torch.device(DEV)
    cfg, model = bench.build_model(dev_)
    ref = reference_observables(model, cfg, REF_JETS, dev_, n_particles=bench.N_PART, efp=True)
    cols = w1_columns(False, True)
    assert ref.shape == (REF_JETS, len(cols)) and cols[-6:] == EFP_COLUMNS
    base = one_gpu_run(model, cfg, TOTAL, 16384)
    plain = one_gpu_run(model, cfg, TOTAL, 16384, w1_reference=ref[:, :len(w1_columns())])
    big = one_gpu_run(model, cfg, TOTAL, 16384, w1_reference=ref, efp=True)
    small = one_gpu_run(model, cfg, TOTAL, 4096, w1_reference=ref, efp=True)
    for key, val in base.items():                                    # the EFP pass changes nothing else
        if key not in ("seconds", "value"):
            assert big[key] == val, key
    assert "fpd" not in plain and "mean_efp1" not in base and set(plain["w1"]) == set(w1_columns())
    for key in METRIC_KEYS:
        assert big[key] == small[key], key                           # bit-identical for any micro-batch
    assert [big["w1"][c] for c in w1_columns()] == [plain["w1"][c] for c in w1_columns()]
    assert big["jet_metrics_seconds"] > 0 and big["mean_efp1"] > 0
    # the same jets, collected outside the pipeline
    same = reference_observables(model, cfg, TOTAL, dev_, n_particles=bench.N_PART, efp=True, jet_offset=0)
    pick = [cols.index(c) for c in EFP_COLUMNS[1:]]
    assert list(fpd(ref[:, pick], same[:, pick])) == big["fpd"] and list(kpd(ref[:, pick], same[:, pick])) == big["kpd"]
    # an independent reference of the same model is close; one with 25 % wider jets is not (the EFPs do not see the pT scale)
    from multimodal_particles_b200.pipeline import STATS
    shifted = dict(STATS, std=[STATS["std"][0], 0.25, 0.25])
    ref_shift = reference_observables(model, cfg, REF_JETS, dev_, n_particles=bench.N_PART, stats=shifted, efp=True)
    far = one_gpu_run(model, cfg, TOTAL, 16384, w1_reference=ref_shift, efp=True)
    assert far["fpd"][0] > 10 * (big["fpd"][0] + big["fpd"][1]), (far["fpd"], big["fpd"])
    assert far["kpd"][0] > 10 * (abs(big["kpd"][0]) + big["kpd"][1]), (far["kpd"], big["kpd"])


def _two_gpu_kwargs(model, cfg, dev_):
    import bench
    from multimodal_particles_b200.pipeline import reference_observables
    return dict(w1_reference=reference_observables(model, cfg, REF_JETS, dev_, n_particles=bench.N_PART, efp=True), efp=True)


@pytest.mark.gpu
def test_two_gpu_efp_metrics_equal_one_gpu(tmp_path):
    """W1, FPD and KPD of a two-GPU run (uneven shards) are bit-identical to the one-GPU run; needs two GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import bench
    two = two_gpu_run(tmp_path, TOTAL + 5, _two_gpu_kwargs, METRIC_KEYS)
    dev_ = torch.device(DEV)
    cfg, model = bench.build_model(dev_)
    one = one_gpu_run(model, cfg, TOTAL + 5, 16384, **_two_gpu_kwargs(model, cfg, dev_))
    assert two["w1"] == one["w1"] and two["w1_used"] == {c: list(v) for c, v in one["w1_used"].items()}
    assert two["fpd"] == one["fpd"] and two["kpd"] == one["kpd"]
