"""A torch restatement of MultiModalEPiC and the two bridge-matching losses, used as the yardstick of the native gradients.

Built from the mirror modules' parameters with the weight norm *unfolded* (``torch._weight_norm`` of each ``weight_v`` /
``weight_g`` leaf), so autograd reaches every state-dict key.  The op sequence is the reference's (utils.py:112-172,
epic.py:136-241, mbm.py:102-113, 167-197), as in tools/torch_eager_baseline.py.  One deliberate difference: a jet without a live
particle pools over a count clamped to one, so its heads are finite and the masked losses exclude it, as the native losses do
(the reference's heads are NaN there, epic.py:141)."""
import torch
import torch.nn.functional as F
from torch import nn


class Restatement:
    """``branches``: None; an empty list, which the next evaluation fills with every leaky-ReLU pre-activation (detached); or a
    list of boolean masks (one per leaky ReLU, in evaluation order) that choose the positive branch instead of the sign."""

    def __init__(self, model, dtype=torch.float64, device="cpu", branches=None):
        self.branches = branches
        self._replay = iter(branches) if branches else None
        self._record = branches is not None and not branches
        enc = model.encoder
        self.params = {k: p.detach().to(device, dtype).clone().requires_grad_(True) for k, p in model.named_parameters()}
        self.dtype, self.device = dtype, torch.device(device)
        self.skip = bool(enc.epic.epic.use_skip_connection)
        self.L = enc.epic.epic.num_blocks
        self.head = bool(enc.add_discrete_head)
        self.Dc, self.S, self.T = enc.dim_features_continuous, enc.vocab_size, model.config.encoder.dim_emb_time
        emb = enc.epic.embedding
        self.context_kind = None
        if hasattr(emb, "embedding_continuous_context"):
            self.context_kind = "linear" if isinstance(emb.embedding_continuous_context, nn.Linear) else "identity"

    def encoder_parameters(self):
        return {k: v for k, v in self.params.items() if k.startswith("encoder.")}

    def _p(self, name):
        return self.params["encoder." + name]

    def _lrelu(self, a):
        if self._replay is not None:
            return torch.where(next(self._replay), a, 0.01 * a)
        if self._record:
            self.branches.append(a.detach())
        return F.leaky_relu(a)

    def _lin(self, name, inp):
        w = torch._weight_norm(self._p(name + ".weight_v"), self._p(name + ".weight_g"), 0)
        return F.linear(inp, w, self._p(name + ".bias"))

    def heads(self, temb, x, k, mask, context_continuous=None):
        """temb [B,T] (or [1,T]), x [B,N,Dc], k [B,N] int, mask [B,N] -> (v [B,N,Dc], logits [B,N,S])"""
        f = lambda a: torch.as_tensor(a).to(self.device, self.dtype)
        x, m = f(x), f(mask).reshape(x.shape[0], x.shape[1])[..., None]
        k = torch.as_tensor(k).to(self.device).long().reshape(x.shape[0], x.shape[1])
        B, N, _ = x.shape
        ctx = f(temb).expand(B, -1)
        if self.context_kind is not None:
            c = f(context_continuous).reshape(B, -1)
            if self.context_kind == "linear":
                c = F.linear(c, self._p("epic.embedding.embedding_continuous_context.weight"),
                             self._p("epic.embedding.embedding_continuous_context.bias"))
            ctx = torch.cat([ctx, c], -1)
        T = temb.shape[-1]
        lrelu = self._lrelu
        if self.branches and not self._record:
            self._replay = iter(self.branches)
        e = F.linear(x, self._p("epic.embedding.embedding_continuous.weight"), self._p("epic.embedding.embedding_continuous.bias"))
        feat = torch.cat([ctx[:, None, :T].expand(B, N, T), e, self._p("epic.embedding.embedding_discrete.weight")[k]], -1) * m
        cnt = m.sum(1).clamp(min=1.0)

        def pool(xl, *glob):
            s = (xl * m).sum(1)
            return torch.cat([s / cnt, s, *glob], 1)

        net = "epic.epic."
        xl = lrelu(self._lin(net + "epic_proj.local_0", feat))
        xg = lrelu(self._lin(net + "epic_proj.global_0", pool(xl, ctx)))
        xg = lrelu(self._lin(net + "epic_proj.global_1", xg))
        xg = lrelu(self._lin(net + "epic_proj.global_2", xg))
        xl = xl * m
        skl, skg = xl, xg
        for i in range(self.L):
            pre = f"{net}epic_layers.{i}."
            h = lrelu(self._lin(pre + "fc_global1", pool(xl, xg, ctx)))
            xg = lrelu(self._lin(pre + "fc_global2", h) + xg)
            loc = torch.cat([xl, xg[:, None, :].expand(B, N, -1), ctx[:, None, :].expand(B, N, -1)], -1)
            xl = lrelu(self._lin(pre + "fc_local2", lrelu(self._lin(pre + "fc_local1", loc))) + xl) * m
            if self.skip:
                xl, xg = xl + skl, xg + skg
        h = self._lin(net + "output_layer", xl) * m
        v, z = h[..., :self.Dc], h[..., self.Dc:]
        if self.head:
            z = F.linear(F.selu(F.linear(z, self._p("fc_layer.0.weight"), self._p("fc_layer.0.bias"))),
                         self._p("fc_layer.2.weight"), self._p("fc_layer.2.bias"))
        return v, z

    def losses(self, v, logits, x0, x1, k1, mask):
        return bridge_losses(v, logits, x0, x1, k1, mask, self.dtype, self.device)

    def bridge_matching_losses(self, state, batch):
        """The pair MultiModalBridgeMatching.bridge_matching_losses returns, from the same state and batch."""
        temb = sinusoidal(state.time, self.T)
        v, logits = self.heads(temb, state.continuous, state.discrete, state.absorbing, getattr(batch, "context_continuous", None))
        return self.losses(v, logits, batch.source_continuous, batch.target_continuous, batch.target_discrete, state.absorbing)

    def multihead(self, l0, l1):
        w = self.params["loss_multihead.weights"]
        return torch.exp(-w[0]) * l0 + w[0] + torch.exp(-w[1]) * l1 + w[1]


def sinusoidal(t, dim):
    """The time embedding the model uses (evaluated on the host in fp32, as EPiCWrapper.time_embedding does)."""
    from multimodal_particles_b200.steptable import sinusoidal_time_embedding
    t = torch.as_tensor(t)
    return sinusoidal_time_embedding(t.detach().reshape(t.shape[0]).float().cpu(), dim, 10000)


def bridge_losses(v, logits, x0, x1, k1, mask, dtype=torch.float64, device="cpu"):
    """Masked MSE of the drift and masked cross entropy, each over the live particles (mbm.py:167-197)."""
    f = lambda a: torch.as_tensor(a).to(device, dtype)
    v, logits = f(v), f(logits)
    B, N, S = logits.shape
    m = f(mask).reshape(B, N)
    k1 = torch.as_tensor(k1).to(device).long().reshape(B, N)
    live = m.sum()
    mse = (((v - (f(x1) - f(x0))) ** 2).sum(-1) * m).sum() / live
    ce = (F.cross_entropy(logits.reshape(-1, S), k1.reshape(-1), reduction="none").reshape(B, N) * m).sum() / live
    return mse, ce


def float64_branch_choices(model, state, batch, device, tol=1e-6, nearest=8):
    """Float64 restatements of the network on the leaky-ReLU branch assignments a float32 forward can take.

    A pre-activation within rounding of zero can land on either side in float32 and in float64, and there the derivative jumps
    by 0.99: the float64 gradient is then the gradient of another branch than the one a float32 forward (the native kernel's,
    the reference's) evaluates.  Yields (flipped units, restatement): first float64's own branches, then each of the ``nearest``
    units whose |pre-activation| <= tol * max|pre-activation of its layer| flipped alone, then every pair of them."""
    import itertools
    pre = []
    Restatement(model, torch.float64, device, pre).bridge_matching_losses(state, batch)
    close = []   # (relative distance to the kink, tensor, flat index)
    for t, a in enumerate(pre):
        rel = (a.abs() / a.abs().max().clamp(min=1e-300)).reshape(-1)
        vals, idx = torch.topk(rel, min(nearest, rel.numel()), largest=False)
        close += [(float(v), t, int(i)) for v, i in zip(vals, idx) if float(v) <= tol]
    close = sorted(close)[:nearest]
    base = [a > 0 for a in pre]
    del pre
    for size in range(3):
        for flips in itertools.combinations(close, size):
            masks = list(base)
            for _, t, i in flips:
                m = masks[t].clone().reshape(-1)
                m[i] = ~m[i]
                masks[t] = m.reshape(base[t].shape)
            yield [(t, i) for _, t, i in flips], Restatement(model, torch.float64, device, masks)
