"""1-D Wasserstein distance (mmb_wasserstein1d): a numpy statement of the merged-sequence formula against scipy (CPU); the kernel
against scipy on the same float32 data, determinism, argument errors, the JetClassHighLevelFeatures mirror and the W1 of the
sharded generation run (GPU)."""
import ctypes

import numpy as np
import pytest
import scipy.stats
import torch

from pipeline_lib import one_gpu_run, two_gpu_run

DEV = "cuda:0"
REL, ABS = 1e-9, 1e-12


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


def scipy_w1(x, y):
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    return scipy.stats.wasserstein_distance(x[np.isfinite(x)], y[np.isfinite(y)])


@pytest.mark.parametrize("case", ["normal", "ties", "n_ne_m", "single", "single_vs_many", "nonfinite"])
def test_merged_formula_matches_scipy(case):
    g = np.random.default_rng(sum(map(ord, case)))
    x, y = {
        "normal": lambda: (g.normal(0, 1, 5000), g.normal(0.1, 1.2, 5000)),
        "ties": lambda: (g.integers(0, 6, 3000).astype(float), g.integers(1, 8, 2500).astype(float)),
        "n_ne_m": lambda: (g.exponential(2.0, 1001), g.exponential(2.5, 77)),
        "single": lambda: (np.array([0.5]), np.array([-1.25])),
        "single_vs_many": lambda: (np.array([3.0]), g.normal(0, 1, 999)),
        "nonfinite": lambda: (np.concatenate([g.normal(0, 1, 300), [np.nan, np.inf]]), np.concatenate([g.normal(0, 1, 200), [-np.inf]])),
    }[case]()
    assert merged_w1(x, y) == pytest.approx(scipy_w1(x, y), rel=1e-12, abs=1e-14)
    assert merged_w1(x, x) == 0.0


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
def w1(x, y, return_counts=False):
    from multimodal_particles_b200.observables import wasserstein1d
    return wasserstein1d(torch.from_numpy(np.ascontiguousarray(x)).to(DEV), torch.from_numpy(np.ascontiguousarray(y)).to(DEV),
                         return_counts)


def check_columns(got, x, y):
    got = np.atleast_1d(got.cpu().numpy())
    for c in range(x.shape[1]):
        assert got[c] == pytest.approx(scipy_w1(x[:, c], y[:, c]), rel=REL, abs=ABS), c


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 5, 64])
def test_normals_n_ne_m(K):
    g = np.random.default_rng(K)
    scale = g.uniform(0.1, 10.0, K).astype(np.float32)
    x = (g.normal(0, 1, (100003, K)) * scale).astype(np.float32)
    y = (g.normal(0.05, 1.1, (77777, K)) * scale).astype(np.float32)
    check_columns(w1(x, y), x, y)


@pytest.mark.gpu
def test_heavy_ties():
    g = np.random.default_rng(3)
    x = np.stack([np.clip(np.rint(g.normal(45, 18, 200000)), 1, 128), g.integers(-6, 7, 200000), g.integers(-1, 2, 200000)], 1)
    y = np.stack([np.clip(np.rint(g.normal(47, 17, 150001)), 1, 128), g.integers(-5, 7, 150001), g.integers(-1, 2, 150001)], 1)
    x, y = x.astype(np.float32), y.astype(np.float32)
    check_columns(w1(x, y), x, y)


@pytest.mark.gpu
def test_self_is_zero_and_dyadic_shift():
    g = np.random.default_rng(4)
    x = (np.rint(g.normal(0, 1, (65537, 3)) * 1024) / 1024).astype(np.float32)   # multiples of 2^-10 in (-8, 8): x + 0.25 is exact
    assert w1(x, x).cpu().numpy().tolist() == [0.0, 0.0, 0.0]
    shifted = w1(x, x + np.float32(0.25)).cpu().numpy()
    np.testing.assert_allclose(shifted, 0.25, rtol=REL, atol=ABS)
    check_columns(torch.from_numpy(shifted), x, x + np.float32(0.25))


@pytest.mark.gpu
def test_one_row_samples_and_vectors():
    x, y = np.array([[0.5, -2.0]], np.float32), np.array([[-1.25, 7.0]], np.float32)
    check_columns(w1(x, y), x, y)
    many = np.random.default_rng(5).normal(0, 1, (999, 2)).astype(np.float32)
    check_columns(w1(x, many), x, many)
    check_columns(w1(many, y), many, y)
    d, used = w1(many[:, 0], many[:, 1], return_counts=True)       # 1-D inputs: a 0-d result
    assert d.dim() == 0 and d.dtype == torch.float64 and used.tolist() == [999, 999]
    assert float(d) == pytest.approx(scipy_w1(many[:, 0], many[:, 1]), rel=REL, abs=ABS)


@pytest.mark.gpu
def test_nonfinite_values_are_dropped_and_counted():
    g = np.random.default_rng(6)
    n, m, K = 50000, 40000, 4
    x, y = g.normal(0, 1, (n, K)).astype(np.float32), g.normal(0, 1, (m, K)).astype(np.float32)
    x[g.random(n) < 0.1, 0] = np.nan
    x[g.random(n) < 0.02, 1] = np.inf
    y[g.random(m) < 0.05, 1] = -np.inf
    y[g.random(m) < 0.3, 2] = np.nan
    x[:, 3] = np.nan                                                # no finite value: NaN
    out, used = w1(x, y, return_counts=True)
    out = out.cpu().numpy()
    assert np.isnan(out[3])
    check_columns(torch.from_numpy(out[:3]), x[:, :3], y[:, :3])
    assert used.tolist() == [np.isfinite(x).sum(0).tolist(), np.isfinite(y).sum(0).tolist()]


@pytest.mark.gpu
def test_many_tiles():
    g = np.random.default_rng(8)
    x = g.normal(0, 1, (1 << 23, 1)).astype(np.float32)
    y = g.normal(0.01, 1, ((1 << 23) - 3, 1)).astype(np.float32)
    check_columns(w1(x, y), x, y)


@pytest.mark.gpu
def test_bit_identical_across_calls_and_row_order():
    g = np.random.default_rng(9)
    x = g.normal(0, 1, (300001, 6)).astype(np.float32)
    x[g.random(300001) < 0.01, 2] = np.nan
    x[:1000, 4] = 0.0
    x[1000:2000, 4] = -0.0
    y = g.gamma(2.0, 1.0, (200000, 6)).astype(np.float32)
    a, b = w1(x, y).cpu().numpy(), w1(x, y).cpu().numpy()
    c = w1(x[g.permutation(len(x))], y[g.permutation(len(y))]).cpu().numpy()
    assert a.tobytes() == b.tobytes() == c.tobytes()


@pytest.mark.gpu
def test_argument_errors_are_codes():
    from multimodal_particles_b200 import _native
    from multimodal_particles_b200.observables import wasserstein1d
    with pytest.raises(_native.MmbError):
        wasserstein1d(torch.zeros(8), torch.zeros(8))                                # host tensors
    lib = _native.load()
    n, m, K = 100, 90, 4
    x, y = torch.zeros(n, K, device=DEV), torch.zeros(m, K, device=DEV)
    out, used = torch.empty(K, dtype=torch.float64, device=DEV), torch.empty(2 * K, dtype=torch.int64, device=DEV)
    need = lib.mmb_wasserstein1d_workspace_bytes(n, m, K)
    assert need > 0 and lib.mmb_wasserstein1d_workspace_bytes(n, m, 0) == 0 and lib.mmb_wasserstein1d_workspace_bytes(n, m, 65) == 0
    ws = torch.empty(need, dtype=torch.uint8, device=DEV)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    call = lambda X, ldx, Y, ldy, k, O, W, nb: lib.mmb_wasserstein1d(X, ldx, n, Y, ldy, m, k, O, p(used), W, nb, s)
    assert call(p(x), K, p(y), K, 0, p(out), p(ws), need) == -1             # K = 0
    assert call(p(x), K, p(y), K, 65, p(out), p(ws), need) == -1            # K > 64
    assert call(p(x), K - 1, p(y), K, K, p(out), p(ws), need) == -1        # ldx < K
    assert call(p(x), K, p(y), K - 1, K, p(out), p(ws), need) == -1        # ldy < K
    assert call(None, K, p(y), K, K, p(out), p(ws), need) == -1             # null x
    assert call(p(x), K, None, K, K, p(out), p(ws), need) == -1             # null y
    assert call(p(x), K, p(y), K, K, None, p(ws), need) == -1               # null out
    assert call(p(x), K, p(y), K, K, p(out), None, need) == -1              # null workspace
    assert call(p(x), K, p(y), K, K, p(out), p(ws), need - 1) == -3        # workspace one byte short
    assert lib.mmb_wasserstein1d(p(x), K, -1, p(y), K, m, K, p(out), None, p(ws), need, s) == -1   # negative size
    assert call(p(x), K, p(y), K, K, p(out), p(ws), need) == 0
    torch.cuda.synchronize()
    assert out.cpu().tolist() == [0.0] * K and used.cpu().tolist() == [n] * K + [m] * K


def _clouds(seed, B=768, N=128):
    from multimodal_particles_b200 import HybridState
    from multimodal_particles_b200.observables import JetClassHighLevelFeatures, ParticleClouds
    g = np.random.default_rng(seed)
    mult = np.clip(np.rint(g.normal(45, 18, B)), 1, N).astype(int)
    mask = (np.arange(N)[None] < mult[:, None]).astype(np.int64)
    xs = g.normal(0, 1, (B, N, 3)).astype(np.float32) * mask[..., None]
    k = g.integers(0, 8, (B, N)) * mask
    state = HybridState(None, torch.from_numpy(xs), torch.from_numpy(k)[..., None], torch.from_numpy(mask)[..., None])
    pc = ParticleClouds(dataset=state)
    pc.postprocess(input_continuous="standardize", input_discrete="tokens", stats={"mean": [1.2, 0.0, 0.0], "std": [0.35, 0.2, 0.2]})
    jets = JetClassHighLevelFeatures(pc)
    jets.compute_substructure()
    return jets


@pytest.mark.gpu
def test_mirror_class_equals_wassertein1d():
    a, b = _clouds(1), _clouds(2, B=640)
    features = ("pt", "m", "eta", "phi", "multiplicity", "Q_total", "Q_jet", "tau1", "tau2", "tau3", "tau21", "tau32", "d2")
    got = a.wasserstein1d(b, features)
    assert list(got) == list(features)
    for f in features:
        assert got[f] == pytest.approx(a.Wassertein1D(f, b), rel=REL, abs=ABS), f
    assert set(a.wasserstein1d(b)) == {"pt", "m", "eta", "phi", "multiplicity", "Q_total", "Q_jet"}
    assert a.wasserstein1d(a, ("pt", "tau21")) == {"pt": 0.0, "tau21": 0.0}


TOTAL, REF_JETS = 3 * 16384, 20000


@pytest.mark.gpu
def test_sharded_run_w1():
    import bench
    from multimodal_particles_b200.observables import wasserstein1d
    from multimodal_particles_b200.pipeline import STATS, reference_observables, w1_columns
    dev = torch.device(DEV)
    cfg, model = bench.build_model(dev)
    ref = reference_observables(model, cfg, REF_JETS, dev, n_particles=bench.N_PART, substructure=True)
    cols = w1_columns(True)
    assert ref.shape == (REF_JETS, len(cols))
    base = one_gpu_run(model, cfg, TOTAL, 16384, substructure=True)
    big = one_gpu_run(model, cfg, TOTAL, 16384, substructure=True, w1_reference=ref)
    small = one_gpu_run(model, cfg, TOTAL, 4096, substructure=True, w1_reference=ref)
    for key, val in base.items():                                   # the W1 collection changes nothing else
        if key not in ("seconds", "value"):
            assert big[key] == val, key
    assert "w1" not in base
    assert big["w1"] == small["w1"] and big["w1_used"] == small["w1_used"]   # bit-identical for any micro-batch
    assert list(big["w1"]) == list(cols) and big["w1_reference_jets"] == REF_JETS and big["w1_seconds"] > 0
    # the same jets, collected outside the pipeline
    same = reference_observables(model, cfg, TOTAL, dev, n_particles=bench.N_PART, substructure=True, jet_offset=0)
    direct = wasserstein1d(same, ref).cpu().tolist()
    assert [big["w1"][c] for c in cols] == direct
    # an independent reference of the same model: W1 is a small fraction of each column's spread
    r = ref.cpu().numpy()
    for i, c in enumerate(cols):
        v = r[:, i][np.isfinite(r[:, i])]
        spread = np.quantile(v, 0.9) - np.quantile(v, 0.1)
        assert big["w1"][c] < 0.05 * spread, (c, big["w1"][c], spread)
        assert big["w1_used"][c][0] > TOTAL // 2 and big["w1_used"][c][1] > REF_JETS // 2
    # a reference with a harder particle pT scale is far away in jet pT
    shifted = dict(STATS, mean=[STATS["mean"][0] + 0.3] + STATS["mean"][1:])
    ref_shift = reference_observables(model, cfg, REF_JETS, dev, n_particles=bench.N_PART, stats=shifted)
    far = one_gpu_run(model, cfg, TOTAL, 16384, w1_reference=ref_shift)
    assert far["w1"]["pt"] > 10 * big["w1"]["pt"]


def _two_gpu_kwargs(model, cfg, dev):
    import bench
    from multimodal_particles_b200.pipeline import reference_observables
    return dict(substructure=True, w1_reference=reference_observables(model, cfg, REF_JETS, dev, n_particles=bench.N_PART, substructure=True))


@pytest.mark.gpu
def test_two_gpu_w1_equals_one_gpu(tmp_path):
    """The gathered W1 of a two-GPU run (uneven shards) is bit-identical to the one-GPU run; needs two GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import bench
    two = two_gpu_run(tmp_path, TOTAL + 5, _two_gpu_kwargs, ("w1", "w1_used"))
    dev = torch.device(DEV)
    cfg, model = bench.build_model(dev)
    one = one_gpu_run(model, cfg, TOTAL + 5, 16384, **_two_gpu_kwargs(model, cfg, dev))
    assert two["w1"] == one["w1"] and two["w1_used"] == {c: list(v) for c, v in one["w1_used"].items()}
