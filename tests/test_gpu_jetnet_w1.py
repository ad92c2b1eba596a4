"""W1 of drawn jets (mmb_wasserstein1d_drawn, DESIGN.md §4.6e) on the GPU: bit-identity with mmb_wasserstein1d on the gathered
drawn sample, agreement with scipy, determinism under repeats and permutations, argument errors, JetNet's w1m / w1efp / w1p,
and W1-P, W1-M and W1-EFP of the sharded generation run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.stats
import torch

from pipeline_lib import one_gpu_run, two_gpu_run

DEV = "cuda:0"


def _multiplicities(g, n, P, kind):
    if kind == "jetclass":
        return np.clip(np.rint(g.normal(45, 18, n)), 1, P).astype(int)
    if kind == "all":
        return np.full(n, P)
    return g.integers(0, P + 1, n)   # "random": includes jets with no used slot


def _sample(g, n, P, F, kind="random", nonfinite=False, scattered=False):
    x = g.normal(0, 1, (n, P, F)).astype(np.float32) * g.uniform(0.1, 10, F).astype(np.float32)
    mult = _multiplicities(g, n, P, kind)
    mask = (np.arange(P)[None, :] < mult[:, None])
    if scattered:   # used slots anywhere in the jet, not a prefix
        mask = np.take_along_axis(mask, g.permuted(np.tile(np.arange(P), (n, 1)), axis=1), 1)
    if nonfinite:
        hit = g.random(x.shape) < 0.02
        x[hit] = g.choice(np.array([np.nan, np.inf, -np.inf], np.float32), hit.sum())
    return torch.from_numpy(x).to(DEV), torch.from_numpy(mask.astype(np.uint8)).to(DEV)


def drawn(x, ix, y, iy, mx=None, my=None):
    from multimodal_particles_b200.observables import wasserstein1d_drawn
    return wasserstein1d_drawn(x, ix, y, iy, mx, my, return_counts=True)


def gathered(x, ix, y, iy, mx=None, my=None):
    """Per draw: mmb_wasserstein1d on the used slots of the drawn jets gathered into rows -> ([draws, F], [2, draws, F])."""
    from multimodal_particles_b200.observables import wasserstein1d
    x3, y3 = (x if x.dim() == 3 else x[:, None]), (y if y.dim() == 3 else y[:, None])
    outs, counts = [], []
    for t in range(ix.shape[0]):
        a, b = x3[ix[t].long()], y3[iy[t].long()]
        a = a[mx[ix[t].long()].bool()] if mx is not None else a.reshape(-1, a.shape[-1])
        b = b[my[iy[t].long()].bool()] if my is not None else b.reshape(-1, b.shape[-1])
        o, c = wasserstein1d(a.contiguous(), b.contiguous(), return_counts=True)
        outs.append(o)
        counts.append(c)
    return torch.stack(outs), torch.stack(counts, 1)


def assert_bits(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    assert torch.equal(a.view(torch.int64) if a.dtype == torch.float64 else a, b.view(torch.int64) if b.dtype == torch.float64 else b)


CASES = {   # name: (n, m, P, F, draws, rows, multiplicities, non-finite values, scattered masks)
    "jetclass_n128": (20000, 15000, 128, 3, 3, 5000, "jetclass", False, False),
    "all_n128": (3000, 2000, 128, 3, 2, 2000, "all", False, False),
    "n256": (3000, 2500, 256, 3, 2, 1500, "random", False, True),
    "f1": (5000, 4000, 128, 1, 4, 3000, "jetclass", False, False),
    "f64": (3000, 3000, 8, 64, 2, 2000, "random", False, True),
    "repeats": (40, 30, 16, 3, 3, 4000, "random", False, False),
    "nonfinite": (4000, 3000, 64, 3, 3, 2000, "random", True, True),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_bit_identical_to_gathered_sample(case):
    n, m, P, F, draws, rows, kind, nonfinite, scattered = CASES[case]
    g = np.random.default_rng(sum(map(ord, case)))
    x, mx = _sample(g, n, P, F, kind, nonfinite, scattered)
    y, my = _sample(g, m, P, F, kind, nonfinite, scattered)
    y[..., 0] += 0.3
    ix = torch.randint(n, (draws, rows), generator=torch.Generator(DEV).manual_seed(1), device=DEV, dtype=torch.int32)
    iy = torch.randint(m, (draws, rows), generator=torch.Generator(DEV).manual_seed(2), device=DEV, dtype=torch.int32)
    out, used = drawn(x, ix, y, iy, mx, my)
    ref, ref_used = gathered(x, ix, y, iy, mx, my)
    assert_bits(out, ref)
    assert torch.equal(used, ref_used)
    if case == "all_n128":   # no mask is the same as an all-ones mask
        o2, u2 = drawn(x, ix, y, iy)
        assert_bits(o2, out)
        assert torch.equal(u2, used)


@pytest.mark.gpu
def test_jet_level_bit_identical():
    g = np.random.default_rng(7)
    x = torch.from_numpy(g.exponential(50, (30000, 5)).astype(np.float32)).to(DEV)
    y = torch.from_numpy(g.exponential(55, (20000, 5)).astype(np.float32)).to(DEV)
    x[::97, 2] = float("nan")
    ix = torch.randint(30000, (5, 50000), device=DEV, dtype=torch.int32)
    iy = torch.randint(20000, (5, 50000), device=DEV, dtype=torch.int32)
    out, used = drawn(x, ix, y, iy)
    ref, ref_used = gathered(x, ix, y, iy)
    assert_bits(out, ref)
    assert torch.equal(used, ref_used)
    o1, _ = drawn(x[:, 1:2], ix, y[:, 1:2], iy)   # a column alone: the same bits
    assert_bits(o1[:, 0], out[:, 1])


@pytest.mark.gpu
def test_side_without_finite_value_is_nan():
    g = np.random.default_rng(8)
    x, mx = _sample(g, 100, 16, 3)
    y, my = _sample(g, 100, 16, 3)
    y[:10] = float("nan")   # draw 0 of y: only the all-NaN jets 0..9
    my[10:20] = 0           # draw 1 of y: only jets with no used slot
    ix = torch.randint(100, (3, 50), device=DEV, dtype=torch.int32)
    iy = torch.stack([torch.arange(50, device=DEV) % 10, 10 + torch.arange(50, device=DEV) % 10, torch.arange(50, device=DEV)]).int()
    out, used = drawn(x, ix, y, iy, mx, my)
    assert torch.isnan(out[:2]).all() and torch.equal(used[1, :2], torch.zeros(2, 3, dtype=torch.int64, device=DEV))
    assert torch.isfinite(out[2]).all()
    ref, ref_used = gathered(x, ix, y, iy, mx, my)
    assert_bits(out, ref)
    assert torch.equal(used, ref_used)


@pytest.mark.gpu
def test_agrees_with_scipy():
    g = np.random.default_rng(9)
    x, mx = _sample(g, 2000, 64, 3, "jetclass")
    y, my = _sample(g, 1500, 64, 3, "jetclass")
    y[..., 1] *= 1.1
    ix = torch.randint(2000, (3, 1000), device=DEV, dtype=torch.int32)
    iy = torch.randint(1500, (3, 1000), device=DEV, dtype=torch.int32)
    out = drawn(x, ix, y, iy, mx, my)[0].cpu().numpy()
    xn, yn, mxn, myn = x.cpu().numpy(), y.cpu().numpy(), mx.cpu().numpy().astype(bool), my.cpu().numpy().astype(bool)
    for t in range(3):
        a, b = xn[ix[t].cpu().numpy()][mxn[ix[t].cpu().numpy()]], yn[iy[t].cpu().numpy()][myn[iy[t].cpu().numpy()]]
        for c in range(3):
            want = scipy.stats.wasserstein_distance(a[:, c].astype(np.float64), b[:, c].astype(np.float64))
            assert out[t, c] == pytest.approx(want, rel=1e-9, abs=1e-12), (t, c)


@pytest.mark.gpu
def test_same_bits_on_repeat_and_under_permutations():
    g = np.random.default_rng(10)
    x, mx = _sample(g, 3000, 128, 3, "jetclass", nonfinite=True)
    y, my = _sample(g, 2000, 128, 3, "jetclass")
    ix = torch.randint(3000, (3, 4000), device=DEV, dtype=torch.int32)
    iy = torch.randint(2000, (3, 4000), device=DEV, dtype=torch.int32)
    out, used = drawn(x, ix, y, iy, mx, my)
    again, _ = drawn(x, ix, y, iy, mx, my)
    assert_bits(again, out)
    slots = torch.from_numpy(g.permuted(np.tile(np.arange(128), (3000, 1)), axis=1)).to(DEV)   # slots within each jet
    xp, mxp = torch.gather(x, 1, slots[..., None].expand(-1, -1, 3)), torch.gather(mx, 1, slots)
    assert_bits(drawn(xp, ix, y, iy, mxp, my)[0], out)
    perm = torch.from_numpy(g.permutation(3000)).to(DEV)                                          # jets, indices remapped
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(3000, device=DEV)
    po, pu = drawn(x[perm], inv[ix.long()].int(), y, iy, mx[perm], my)
    assert_bits(po, out)
    assert torch.equal(pu, used)


@pytest.mark.gpu
def test_argument_errors():
    from multimodal_particles_b200 import _native
    from multimodal_particles_b200.observables import wasserstein1d_drawn
    lib = _native.load()
    x = torch.zeros(10, 4, 3, device=DEV)
    idx = torch.zeros(2, 5, dtype=torch.int32, device=DEV)
    out = torch.empty(2, 3, dtype=torch.float64, device=DEV)
    ws = torch.empty(lib.mmb_wasserstein1d_drawn_workspace_bytes(2, 5, 4, 3), dtype=torch.uint8, device=DEV)
    p = _native._ptr

    def call(P=4, F=3, draws=2, rows=5, nbytes=None):
        return lib.mmb_wasserstein1d_drawn(p(x), 12, 3, None, 0, 10, p(x), 12, 3, None, 0, 10, P, F, p(idx), p(idx), draws, rows,
                                           p(out), None, p(ws), ws.numel() if nbytes is None else nbytes, _native._stream())
    assert call() == 0
    torch.cuda.synchronize()
    assert torch.equal(out, torch.zeros_like(out))
    EINVAL, ENOMEM = -1, -3
    for kw in (dict(F=0), dict(F=65), dict(draws=0), dict(rows=0), dict(P=0), dict(rows=1 << 24, P=128), dict(draws=1 << 25, F=64)):
        assert call(**kw) == EINVAL, kw
        assert lib.mmb_wasserstein1d_drawn_workspace_bytes(kw.get("draws", 2), kw.get("rows", 5), kw.get("P", 4), kw.get("F", 3)) == 0
    assert call(nbytes=ws.numel() - 1) == ENOMEM
    with pytest.raises(_native.MmbError):
        wasserstein1d_drawn(x.cpu(), idx, x, idx)
    with pytest.raises(_native.MmbError):
        wasserstein1d_drawn(x, idx.cpu(), x, idx.cpu())
    with pytest.raises(_native.MmbError):
        wasserstein1d_drawn(x, idx, x[:, :2], idx)


def _numpy_summary(vals, average=True):
    means, stds = vals.mean(0), vals.std(0)
    return (means.mean(), np.linalg.norm(stds)) if average else (means, stds)


@pytest.mark.gpu
def test_jetnet_functions_aggregate_the_draws():
    from multimodal_particles_b200.observables import jetnet_draws, w1efp, w1m, w1p, wasserstein1d_drawn
    g = np.random.default_rng(11)
    real, mr = _sample(g, 6000, 128, 3, "jetclass")
    gen, mg = _sample(g, 5000, 128, 3, "jetclass")
    ir, ig = jetnet_draws(6000, 5000, 2000, 4, seed=3, device=real.device)
    vals = wasserstein1d_drawn(real, ir, gen, ig, mr, mg).cpu().numpy()
    assert w1p(real, gen, mr, mg, num_eval_samples=2000, num_batches=4, seed=3) == pytest.approx(_numpy_summary(vals), rel=1e-15)
    per = w1p(real, gen, mr, mg, num_eval_samples=2000, num_batches=4, seed=3, average_over_features=False)
    np.testing.assert_array_equal(per[0], vals.mean(0))
    np.testing.assert_array_equal(per[1], vals.std(0))
    jr = torch.from_numpy(g.exponential(1, (6000, 5)).astype(np.float32)).to(DEV)
    jg = torch.from_numpy(g.exponential(1.1, (5000, 5)).astype(np.float32)).to(DEV)
    ir, ig = jetnet_draws(6000, 5000, seed=42, device=jr.device)   # JetNet's defaults: 5 x 50 000
    vals = wasserstein1d_drawn(jr, ir, jg, ig).cpu().numpy()
    assert w1efp(jr, jg) == pytest.approx(_numpy_summary(vals), rel=1e-15)
    m, s = w1efp(jr, jg, average_over_efps=False)
    np.testing.assert_array_equal(m, vals.mean(0))
    vals_m = wasserstein1d_drawn(jr[:, :1], ir, jg[:, :1], ig).cpu().numpy()
    assert w1m(jr[:, 0], jg[:, 0]) == pytest.approx(_numpy_summary(vals_m), rel=1e-15)
    assert w1m(jr[:, 0], jr[:, 0], num_eval_samples=1000)[0] > 0     # different draws of the same sample


# ---- sharded generation run --------------------------------------------------------------------------------------------------
TOTAL, REF_JETS = 3 * 16384, 20000


def _references(model, cfg, dev):
    import bench
    from multimodal_particles_b200.pipeline import reference_observables, reference_particles
    return (reference_observables(model, cfg, REF_JETS, dev, n_particles=bench.N_PART, efp=True),
            reference_particles(model, cfg, REF_JETS, dev, n_particles=bench.N_PART))


@pytest.mark.gpu
def test_sharded_run_jetnet_w1():
    import bench
    from multimodal_particles_b200.observables import EFP_COLUMNS, PARTICLE_COLUMNS, w1efp, w1m, w1p
    from multimodal_particles_b200.pipeline import reference_observables, reference_particles, w1_columns
    dev = torch.device(DEV)
    cfg, model = bench.build_model(dev)
    ref_jets, ref_parts = _references(model, cfg, dev)
    assert ref_parts[0].shape == (REF_JETS, bench.N_PART, 3) and ref_parts[1].shape == (REF_JETS, bench.N_PART)
    base = one_gpu_run(model, cfg, TOTAL, 16384, efp=True, w1_reference=ref_jets)
    big = one_gpu_run(model, cfg, TOTAL, 16384, efp=True, w1_reference=ref_jets, particle_reference=ref_parts)
    small = one_gpu_run(model, cfg, TOTAL, 4096, efp=True, w1_reference=ref_jets, particle_reference=ref_parts)
    new = {"w1p", "w1p_features", "w1m", "w1efp", "jetnet_w1_seconds"}
    assert set(big) == set(base) | new and not new & set(base)
    for key, val in base.items():                                   # the particle collection changes nothing else
        if key not in ("seconds", "value", "w1_seconds", "jet_metrics_seconds"):
            assert big[key] == val, key
    for key in ("w1p", "w1p_features", "w1m", "w1efp"):              # bit-identical for any micro-batch
        assert big[key] == small[key], key
    assert list(big["w1p_features"]) == list(PARTICLE_COLUMNS) and big["jetnet_w1_seconds"] > 0
    # the same jets, made outside the pipeline
    own_x, own_m = reference_particles(model, cfg, TOTAL, dev, n_particles=bench.N_PART, jet_offset=0)
    assert list(w1p(ref_parts[0], own_x, ref_parts[1], own_m)) == big["w1p"]
    per = w1p(ref_parts[0], own_x, ref_parts[1], own_m, average_over_features=False)
    assert {c: [float(a), float(b)] for c, a, b in zip(PARTICLE_COLUMNS, *per)} == big["w1p_features"]
    cols = w1_columns(False, True)
    own_jets = reference_observables(model, cfg, TOTAL, dev, n_particles=bench.N_PART, efp=True, jet_offset=0)
    mi, pick = cols.index("m"), [cols.index(c) for c in EFP_COLUMNS[1:]]
    assert list(w1m(ref_jets[:, mi], own_jets[:, mi])) == big["w1m"]
    assert list(w1efp(ref_jets[:, pick], own_jets[:, pick])) == big["w1efp"]
    # an independent reference of the same model: W1-P is a small fraction of each feature's spread
    x, msk = ref_parts[0].cpu().numpy(), ref_parts[1].cpu().numpy().astype(bool)
    for i, c in enumerate(PARTICLE_COLUMNS):
        v = x[..., i][msk]
        assert big["w1p_features"][c][0] < 0.05 * (np.quantile(v, 0.9) - np.quantile(v, 0.1)), c
    # without a W1 reference only W1-P joins
    only = one_gpu_run(model, cfg, TOTAL, 16384, particle_reference=ref_parts)
    assert "w1m" not in only and "w1efp" not in only and only["w1p"] == big["w1p"]


@pytest.mark.gpu
def test_million_jets_tool_with_both_references(tmp_path):
    """tools/million_jets.py with a W1 reference and a W1-P reference together (the only way it reports W1-M and W1-EFP)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "rec.json"
    proc = subprocess.run([sys.executable, os.path.join(root, "tools", "million_jets.py"), "--jets", "32768", "--efp",
                           "--w1-reference-jets", "20000", "--w1p-reference-jets", "20000", "--out", str(out)],
                          capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stderr[-3000:]
    rec = json.loads(out.read_text())
    assert {"w1", "fpd", "kpd", "w1p", "w1p_features", "w1m", "w1efp", "jetnet_w1_seconds"} <= set(rec)
    assert all(np.isfinite(rec[k]).all() for k in ("w1p", "w1m", "w1efp"))


def _two_gpu_kwargs(model, cfg, dev):
    ref_jets, ref_parts = _references(model, cfg, dev)
    return dict(efp=True, w1_reference=ref_jets, particle_reference=ref_parts)


@pytest.mark.gpu
def test_two_gpu_jetnet_w1_equals_one_gpu(tmp_path):
    """W1-P, W1-M and W1-EFP of a two-GPU run (uneven shards) are bit-identical to the one-GPU run; needs two GPUs."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import bench
    keys = ("w1p", "w1p_features", "w1m", "w1efp")
    two = two_gpu_run(tmp_path, TOTAL + 5, _two_gpu_kwargs, keys)
    dev = torch.device(DEV)
    cfg, model = bench.build_model(dev)
    one = one_gpu_run(model, cfg, TOTAL + 5, 16384, **_two_gpu_kwargs(model, cfg, dev))
    assert two == json.loads(json.dumps({k: one[k] for k in keys}))
