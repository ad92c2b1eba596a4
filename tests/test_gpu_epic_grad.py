"""GPU: the native losses and gradients of MultiModalBridgeMatching.bridge_matching_losses (epic_grad.cu) against float64
autograd of the torch restatement (tests/grad_lib.py, pinned to the reference's heads and losses by test_epic_grad.py), and the
properties a training loop relies on: values, determinism, normalisation, empty jets, AdamW steps, trained weights in generation."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import grad_lib
from multimodal_particles_b200 import HybridState, MultiModalBridgeMatching, _native
from multimodal_particles_b200.config_classes.multimodal_bridge_matching_config import MultimodalBridgeMatchingConfig
from multimodal_particles_b200.databatch import jetclass_like_databatch
from multimodal_particles_b200.epic import as_u8

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
GRAD_BAR = 1e-4   # max|g - g64| <= GRAD_BAR * max|g64| per state-dict key and loss

SHAPES = {
    "c2": {},                                                                                      # the C2 widths, discrete head
    "odd": dict(dim_hidden_glob=19, num_blocks=3, add_discrete_head=False, dim_emb_time=14),      # test_abi's odd shape
    "noskip": dict(skip_connection=False),
    "default": dict(dim_hidden_local=128, num_blocks=6, dim_hidden_glob=10),                      # the class defaults (epic.py:99-101)
    "ctx": "context",                                                                             # Linear-embedded context
}


def make_config(shape):
    cfg = MultimodalBridgeMatchingConfig()
    tweak = SHAPES[shape]
    if tweak == "context":
        cfg.data.dim_context_continuous = 2
        cfg.encoder.embedding_context_continuous, cfg.encoder.dim_emb_context_continuous = "Embedding", 3
    else:
        for key, val in tweak.items():
            setattr(cfg.encoder, key, val)
    return cfg


def make_model(shape, seed=0):
    cfg = make_config(shape)
    torch.manual_seed(seed)
    return MultiModalBridgeMatching(cfg).to(DEV)


def make_batch(cfg, B, N, seed, special=False):
    """Bridge state and batch.  ``special``: jet 0 empty, jet 1 one particle, jet 2 full, the rest uniform multiplicities;
    otherwise JetClass-like multiplicities (bench.source_batch's distribution)."""
    g = torch.Generator().manual_seed(seed)
    S, Dc = cfg.data.vocab_size_features, cfg.data.dim_features_continuous
    if special:
        mult = torch.randint(1, N + 1, (B,), generator=g)
        mult[:3] = torch.tensor([0, 1, N])
        mask = (torch.arange(N)[None] < mult[:, None]).long().unsqueeze(-1)
    else:
        mask = jetclass_like_databatch(B, N, generator=g).source_mask
    rnd = lambda: torch.randn(B, N, Dc, generator=g) * mask
    tok = lambda: torch.randint(0, S, (B, N, 1), generator=g) * mask
    batch = SimpleNamespace(source_continuous=rnd(), target_continuous=rnd(), target_discrete=tok(), target_mask=mask)
    if cfg.data.dim_context_continuous:
        batch.context_continuous = torch.randn(B, cfg.data.dim_context_continuous, generator=g)
    state = HybridState(torch.rand(B, 1, 1, generator=g), rnd().to(DEV), tok().to(DEV), mask.to(DEV))
    return state, batch


def native_grads(model, state, batch):
    names = [n for n, _ in model.named_parameters() if n.startswith("encoder.")]
    params = [dict(model.named_parameters())[n] for n in names]
    l0, l1 = model.bridge_matching_losses(state, batch)
    out = []
    for i, loss in enumerate((l0, l1)):
        gs = torch.autograd.grad(loss, params, retain_graph=i == 0, allow_unused=True)
        out.append({n: torch.zeros_like(p) if g is None else g for n, p, g in zip(names, params, gs)})
    return (l0, l1), out


def reference_grads(model, state, batch, ref):
    params = ref.encoder_parameters()
    l0, l1 = ref.bridge_matching_losses(state, batch)
    out = []
    for i, loss in enumerate((l0, l1)):
        gs = torch.autograd.grad(loss, list(params.values()), retain_graph=i == 0, allow_unused=True)
        out.append({n: torch.zeros_like(p) if g is None else g for (n, p), g in zip(params.items(), gs)})
    return (l0, l1), out


def worst_ratio(got, want):
    """(largest max|g - g64| / max|g64| over keys and losses, first key above GRAD_BAR or None)"""
    worst, bad = 0.0, None
    for which in range(2):
        assert set(got[which]) == set(want[which])
        for key, g64 in want[which].items():
            g = got[which][key].double()
            assert torch.isfinite(g).all(), key
            scale, err = float(g64.abs().max()), float((g - g64).abs().max())
            if err > GRAD_BAR * scale and bad is None:
                bad = (which, key, err, scale)
            if scale > 0:
                worst = max(worst, err / scale)
    return worst, bad


@pytest.mark.parametrize("batch_kind", ["b64_n30_special", "b1024_n128_jetclass"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_gradients_match_float64_autograd(shape, batch_kind):
    """Per state-dict key and loss, against float64 autograd on the branches of the float32 forward: float64's own leaky-ReLU
    branches, or those with one or two units flipped whose pre-activation is within float32 rounding of zero
    (grad_lib.float64_branch_choices).  The plain float64 ratio of the kernel and of torch float32 autograd is printed beside."""
    model = make_model(shape, seed=3)
    B, N, special = (64, 30, True) if batch_kind.startswith("b64") else (1024, 128, False)
    state, batch = make_batch(model.config, B, N, seed=11, special=special)
    (n0, n1), got = native_grads(model, state, batch)
    tried = []
    for flips, ref in grad_lib.float64_branch_choices(model, state, batch, DEV):
        (r0, r1), want = reference_grads(model, state, batch, ref)
        if not flips:
            np.testing.assert_allclose([float(n0.detach()), float(n1.detach())], [float(r0.detach()), float(r1.detach())], rtol=1e-5)
            plain = want
        worst, bad = worst_ratio(got, want)
        tried.append((flips, worst, bad))
        if bad is None:
            break
    assert bad is None, tried
    _, eager = reference_grads(model, state, batch, grad_lib.Restatement(model, torch.float32, DEV))
    print(f"grad[{shape},{batch_kind}]: worst max|g - g64| / max|g64| = {worst:.3e} with {len(flips)} near-zero unit(s) flipped; "
          f"against plain float64: kernel {worst_ratio(got, plain)[0]:.3e}, torch float32 autograd {worst_ratio(eager, plain)[0]:.3e}")


def test_values_equal_fp32_forward_and_no_jacobian_without_grad(monkeypatch):
    model = make_model("c2", seed=1)
    state, batch = make_batch(model.config, 512, 128, seed=2)
    l0, l1 = model.bridge_matching_losses(state, batch)
    assert l0.grad_fn is not None and l1.grad_fn is not None
    heads = model(state, batch)
    w0, w1 = model.loss_continuous(heads, state, batch), model.loss_discrete(heads, state, batch)
    np.testing.assert_allclose([float(l0), float(l1)], [float(w0), float(w1)], rtol=1e-6)
    calls = []
    real = _native.epic_loss_grad

    def spy(*args, **kwargs):
        calls.append(kwargs.get("jacobian", True))
        return real(*args, **kwargs)

    monkeypatch.setattr(_native, "epic_loss_grad", spy)
    with torch.no_grad():
        m0, m1 = model.bridge_matching_losses(state, batch)
    assert calls == [False] and m0.grad_fn is None
    assert torch.equal(m0, l0.detach()) and torch.equal(m1, l1.detach())


def test_gradients_are_deterministic():
    model = make_model("c2", seed=4)
    state, batch = make_batch(model.config, 1024, 128, seed=5)
    runs = []
    for _ in range(2):
        model.zero_grad(set_to_none=True)
        l0, l1 = model.bridge_matching_losses(state, batch)
        (l0 + 0.5 * l1).backward()
        runs.append({n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None})
    assert runs[0].keys() == runs[1].keys() and len(runs[0]) > 10
    for key in runs[0]:
        assert torch.equal(runs[0][key], runs[1][key]), key


def _split(state, batch, idx):
    sub = SimpleNamespace(**{k: v[idx] for k, v in vars(batch).items()})
    return HybridState(state.time[idx], state.continuous[idx], state.discrete[idx], state.absorbing[idx]), sub


def _blob_jacobian(model, state, batch):
    """jac [2][total] of mmb_epic_loss_grad, split into the blob's tensors (mmb_epic_layout order), and the live count."""
    epic, head = model.encoder.epic, model.encoder.fc_layer
    with torch.no_grad():
        W = epic.packed_parameters(head).to(DEV).contiguous()
        rows = epic.context_rows(state.time, None, None, DEV)
        u8 = lambda a: as_u8(a.to(DEV))
        f32 = lambda a: a.to(DEV, torch.float32).contiguous()
        losses, jac, _ = _native.epic_loss_grad(epic.epic_dims(head[0].out_features), W, f32(state.continuous), u8(state.discrete),
                                                u8(state.absorbing), rows, f32(batch.source_continuous), f32(batch.target_continuous),
                                                u8(batch.target_discrete))
    sizes = [p.numel() for p in epic._blob_parts(head, lambda layer: layer.weight_v)]
    return [row.double().split(sizes) for row in jac], float(losses[2])


def test_batch_gradient_is_live_weighted_mean_of_halves():
    """The kernel's Jacobian of a batch == the live-count-weighted combination of the Jacobians of its halves (partitioning and
    normalisation), per tensor of the blob."""
    model = make_model("c2", seed=6)
    state, batch = make_batch(model.config, 256, 128, seed=7)
    whole, live = _blob_jacobian(model, state, batch)
    halves = [_blob_jacobian(model, *_split(state, batch, idx)) for idx in (slice(0, 128), slice(128, 256))]
    assert live == halves[0][1] + halves[1][1]
    for which in range(2):
        for i, g in enumerate(whole[which]):
            want = (halves[0][1] * halves[0][0][which][i] + halves[1][1] * halves[1][0][which][i]) / live
            assert float((g - want).abs().max()) <= 1e-6 * float(want.abs().max()), (which, i)


def test_empty_jets_change_no_gradient_bit():
    model = make_model("c2", seed=8)
    state, batch = make_batch(model.config, 1024, 128, seed=9)
    (a0, a1), base = native_grads(model, state, batch)
    pad = 64
    grow = lambda t: torch.cat([t, torch.zeros((pad,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)])
    state2 = HybridState(grow(state.time), grow(state.continuous), grow(state.discrete), grow(state.absorbing))
    batch2 = SimpleNamespace(**{k: grow(v) for k, v in vars(batch).items()})
    (b0, b1), padded = native_grads(model, state2, batch2)
    assert torch.equal(a0, b0) and torch.equal(a1, b1)
    for which in range(2):
        for key, g in base[which].items():
            assert torch.isfinite(padded[which][key]).all() and torch.equal(g, padded[which][key]), key


def test_adamw_training_matches_float64_and_trained_weights_reach_generation():
    cfg = make_config("c2")
    cfg.bridge.num_timesteps = 20
    torch.manual_seed(12)
    model = MultiModalBridgeMatching(cfg).to(DEV)
    g = torch.Generator().manual_seed(13)
    src = jetclass_like_databatch(256, 64, generator=g)
    batch = SimpleNamespace(source_continuous=src.source_continuous, source_discrete=src.source_discrete, source_mask=src.source_mask,
                            target_continuous=torch.randn(256, 64, 3, generator=g) * src.source_mask,
                            target_discrete=torch.randint(0, 8, (256, 64, 1), generator=g) * src.source_mask, target_mask=src.source_mask)
    t, z, u = torch.rand(256, generator=g), torch.randn(256, 64, 3, generator=g), torch.rand(256, 64, generator=g)
    u_gen = torch.rand(cfg.bridge.num_timesteps - 1, 256, 64, generator=g)
    fresh_state = lambda: HybridState(None, batch.source_continuous.clone(), batch.source_discrete.clone(), batch.source_mask.clone())
    before = model.simulate_dynamics(fresh_state(), batch, uniforms=u_gen, precision="fp32")

    tr = cfg.train
    opt_args = dict(lr=tr.lr, betas=tuple(tr.betas), eps=tr.eps, weight_decay=tr.weight_decay)
    ref = grad_lib.Restatement(model, torch.float64, DEV)
    opt = torch.optim.AdamW(model.parameters(), **opt_args)
    ref_opt = torch.optim.AdamW(list(ref.params.values()), **opt_args)
    worst = 0.0
    for step in range(20):
        state = model.sample_bridges(batch, t=t, z=z, u=u)
        l0, l1 = model.bridge_matching_losses(state, batch)
        loss, _ = model.loss_multihead([l0, l1])
        opt.zero_grad()
        loss.backward()
        opt.step()
        r0, r1 = ref.bridge_matching_losses(state, batch)
        ref_loss = ref.multihead(r0, r1)
        ref_opt.zero_grad()
        ref_loss.backward()
        ref_opt.step()
        rel = abs(float(loss) - float(ref_loss)) / abs(float(ref_loss))
        worst = max(worst, rel)
        assert rel <= 1e-4, (step, float(loss), float(ref_loss))
    print(f"adamw: worst per-step relative loss difference over 20 steps = {worst:.3e}")

    after = model.simulate_dynamics(fresh_state(), batch, uniforms=u_gen, precision="fp32")
    loaded = MultiModalBridgeMatching(cfg).to(DEV)
    loaded.load_state_dict(model.state_dict())
    again = loaded.simulate_dynamics(fresh_state(), batch, uniforms=u_gen, precision="fp32")
    assert torch.equal(after.continuous, again.continuous) and torch.equal(after.discrete, again.discrete)
    assert not torch.equal(after.continuous, before.continuous)
