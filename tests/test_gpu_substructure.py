"""GPU: mmb_jet_substructure against its oracle (axes bit-exact), the stats path, the JetClassHighLevelFeatures mirror, argument
errors, and the substructure histograms of the sharded generation run."""
import ctypes

import numpy as np
import pytest
import torch

import substructure_oracle as so
from multimodal_particles_b200 import HybridState, _native
from multimodal_particles_b200.observables import JetClassHighLevelFeatures, ParticleClouds, jet_substructure
from test_substructure import random_jets

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def jetclass_like(g, B, N, all_full=False):
    mult = np.full(B, N) if all_full else np.clip(np.rint(g.normal(45, 18, B)), 1, N).astype(int)
    mask = (np.arange(N)[None] < mult[:, None]).astype(np.uint8)
    x, _ = random_jets(g, B, N, 3, 3)
    return (x * mask[..., None]).astype(np.float32), mask


def check(out, axes, want, wax):
    assert np.array_equal(axes, wax)
    assert np.array_equal(np.isnan(out), np.isnan(want))
    ok = ~np.isnan(want)
    rel = lambda c: np.abs(out[:, c] - want[:, c])[ok[:, c]] / np.maximum(np.abs(want[:, c]), 1e-30)[ok[:, c]]
    for c in range(5):   # tau_N and their ratios
        assert np.all((rel(c) <= 1e-6) | (np.abs(out[:, c] - want[:, c])[ok[:, c]] <= 1e-7)), c
    for c in (5, 6):
        assert np.all(rel(c) <= 1e-5), c
    assert np.all(rel(7) <= 1e-4)


@pytest.mark.parametrize("B,N,full", [(4096, 128, False), (4096, 128, True), (4096, 30, False), (512, 200, True)])
def test_kernel_matches_oracle(B, N, full):
    g = np.random.default_rng(N + full)
    x, mask = jetclass_like(g, B, N, full)
    mask[:7, 2:] = 0   # a few jets with fewer than 3 particles
    want, wax = so.jet_substructure(x, mask)
    out, axes = jet_substructure(torch.from_numpy(x).to(DEV), torch.from_numpy(mask).to(DEV), want_axes=True)
    check(out.cpu().numpy(), axes.cpu().numpy(), want, wax)


def test_beta_two_matches_oracle():
    g = np.random.default_rng(5)
    x, mask = jetclass_like(g, 1024, 128)
    want, wax = so.jet_substructure(x, mask, R=0.4, beta=2.0)
    out, axes = jet_substructure(torch.from_numpy(x).to(DEV), torch.from_numpy(mask).to(DEV), R=0.4, beta=2.0, want_axes=True)
    check(out.cpu().numpy(), axes.cpu().numpy(), want, wax)


def test_stats_path():
    g = np.random.default_rng(9)
    B, N = 2048, 128
    x, mask = jetclass_like(g, B, N)
    stats = {"mean": [1.2, 0.0, 0.0], "std": [0.35, 0.2, 0.2]}
    xs = ((x - np.float32(1.2) * mask[..., None]) / np.array([0.35, 0.2, 0.2], np.float32)).astype(np.float32)
    xs[..., 0] += g.normal(0, 2.0, (B, N)).astype(np.float32) * (g.random((B, N)) < 0.05)   # some pt <= 0 after de-standardising
    phys = xs * np.array(stats["std"], np.float32) + np.array(stats["mean"], np.float32)   # the kernel's fp32 de-standardisation
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    a, aa = jet_substructure(dev(xs), dev(mask), stats, want_axes=True)
    b, ba = jet_substructure(dev(phys), dev(mask), None, want_axes=True)
    assert np.array_equal(aa.cpu().numpy(), ba.cpu().numpy())
    np.testing.assert_array_equal(a.cpu().numpy(), b.cpu().numpy())
    want, wax = so.jet_substructure(xs, mask, stats)
    check(a.cpu().numpy(), aa.cpu().numpy(), want, wax)


def test_mirror_class():
    g = np.random.default_rng(13)
    B, N = 512, 128
    x, mask = jetclass_like(g, B, N)
    mask[:4, 1:] = 0
    stats = {"mean": [1.2, 0.0, 0.0], "std": [0.35, 0.2, 0.2]}
    xs = ((x - np.float32(1.2) * mask[..., None]) / np.array([0.35, 0.2, 0.2], np.float32)).astype(np.float32)
    k = (g.integers(0, 8, (B, N)) * mask).astype(np.int64)
    state = HybridState(None, torch.from_numpy(xs), torch.from_numpy(k)[..., None], torch.from_numpy(mask.astype(np.int64))[..., None])
    pc = ParticleClouds(dataset=state)
    pc.postprocess(input_continuous="standardize", input_discrete="tokens", stats=stats)
    jets = JetClassHighLevelFeatures(pc)
    jets.compute_substructure()
    direct = jet_substructure(torch.from_numpy(xs).to(DEV), torch.from_numpy(mask).to(DEV), stats).cpu().numpy()
    keep = ~np.isnan(direct[:, 0])
    used = ((mask != 0) & (xs[..., 0] * np.float32(0.35) + np.float32(1.2) > 0)).sum(1)
    assert np.array_equal(keep, used >= 3) and not keep[:4].any()
    assert jets.tau21.shape == (keep.sum(),) and jets.tau21.device.type == "cpu"
    for name, col in (("tau1", 0), ("tau2", 1), ("tau3", 2), ("tau21", 3), ("tau32", 4), ("d2", 7)):
        np.testing.assert_allclose(getattr(jets, name).numpy(), direct[keep, col], rtol=1e-4, atol=1e-6)
    assert jets.Wassertein1D("tau21", jets) == 0.0
    with pytest.raises(NotImplementedError):
        jets.substructure()


def test_host_tensors_and_bad_arguments():
    with pytest.raises(_native.MmbError):
        jet_substructure(torch.zeros(2, 8, 3), torch.ones(2, 8, dtype=torch.uint8))
    lib = _native.load()
    x = torch.zeros(2, 300, 3, device=DEV)
    m = torch.ones(2, 300, dtype=torch.uint8, device=DEV)
    out = torch.empty(2, 8, device=DEV)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.mmb_jet_substructure(p(x), p(m), None, None, 2, 300, 0.8, 1.0, p(out), None, s) == -1    # N > 256
    assert lib.mmb_jet_substructure(p(x), p(m), None, None, -1, 8, 0.8, 1.0, p(out), None, s) == -1     # negative size
    assert lib.mmb_jet_substructure(p(x), p(m), None, None, 2, 8, 0.0, 1.0, p(out), None, s) == -1      # R <= 0
    assert lib.mmb_jet_substructure(p(x), p(m), None, None, 2, 8, 0.8, -1.0, p(out), None, s) == -1     # beta <= 0
    assert lib.mmb_jet_substructure(None, p(m), None, None, 2, 8, 0.8, 1.0, p(out), None, s) == -1      # null input
    assert lib.mmb_jet_substructure(p(x), p(m), None, None, 0, 8, 0.8, 1.0, p(out), None, s) == 0       # nothing to do
    torch.cuda.synchronize()


def test_sharded_run_histograms():
    import bench
    from multimodal_particles_b200.pipeline import SUBSTRUCTURE_BINS, sharded_generation_run
    dev = torch.device(DEV)
    cfg, model = bench.build_model(dev)
    total = 3 * 16384
    base = sharded_generation_run(model, cfg, total, 0, 1, dev, micro_batch=16384, n_particles=bench.N_PART, warmup_batches=1)
    with_sub = sharded_generation_run(model, cfg, total, 0, 1, dev, micro_batch=16384, n_particles=bench.N_PART, warmup_batches=1,
                                      substructure=True)
    small = sharded_generation_run(model, cfg, total, 0, 1, dev, micro_batch=4096, n_particles=bench.N_PART, warmup_batches=1,
                                   substructure=True)
    for key, val in base.items():
        if key not in ("seconds", "value"):
            assert with_sub[key] == val, key
    assert with_sub["substructure_sha1"] == small["substructure_sha1"]
    assert with_sub["substructure_counts"] == small["substructure_counts"]
    for name, counts in with_sub["substructure_counts"].items():
        assert len(counts) == SUBSTRUCTURE_BINS + 1 and sum(counts) == total, name
        assert sum(counts[:SUBSTRUCTURE_BINS]) > total // 2, name
    assert 0.0 < with_sub["mean_tau21"] < 1.0 and 0.0 < with_sub["mean_tau32"] < 1.0 and with_sub["mean_d2"] > 0.0
