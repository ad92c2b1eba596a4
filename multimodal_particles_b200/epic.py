"""EPiC encoder: parameter containers with the reference's state-dict keys + the native forward.

The reference builds the network from ``torch.nn`` layers and evaluates ~725 eager ops per step
(mp/models/architectures/epic.py:10-241, utils.py:6-198).  Here the modules only *hold* the
parameters (so checkpoints load unchanged: ``…weight_g [out,1]``, ``…weight_v [out,in]``, ``…bias``,
SURVEY.md §A.6); evaluation folds the weight norm once, packs everything into the blob described in
include/mmbridge.h and calls the sm_100a kernels.  No autograd on this generation path; ``packed_parameters`` gives the same
blob under autograd for the losses' backward pass (MultiModalBridgeMatching.bridge_matching_losses).
"""
from typing import Optional

import torch
from torch import nn

from . import _native
from .steptable import sinusoidal_time_embedding


class WeightNormLinear(nn.Module):
    """Parameters of ``weight_norm(nn.Linear(i, o))`` (old-style hook, dim=0): ``bias``,
    ``weight_g`` [o,1], ``weight_v`` [o,i].  Initialised through ``nn.Linear`` so that the RNG
    stream (and hence random-init weights under a fixed seed) equals the reference's."""

    def __init__(self, in_features: int, out_features: int):
        super().__init__()
        seed_layer = nn.Linear(in_features, out_features)
        self.bias = nn.Parameter(seed_layer.bias.detach().clone())
        v = seed_layer.weight.detach().clone()
        self.weight_g = nn.Parameter(torch.norm_except_dim(v, 2, 0))
        self.weight_v = nn.Parameter(v)

    def folded(self) -> torch.Tensor:
        # same ATen function the reference's forward pre-hook runs every step (epic.py:134)
        # (always on the host, so the packed weights do not depend on where the module lives)
        return torch._weight_norm(self.weight_v.detach().cpu().float(), self.weight_g.detach().cpu().float(), 0)


class SinusoidalPositionalEncoding(nn.Module):
    """Parameter-free; kept so the module tree matches (utils.py:175-198)."""

    def __init__(self, dim, max_period=10000):
        super().__init__()
        self.dim, self.max_period = dim, max_period

    def forward(self, timesteps):
        return sinusoidal_time_embedding(timesteps.reshape(-1), self.dim, self.max_period)


class InputEmbeddings(nn.Module):
    """utils.py:6-110.  Feature embeddings: the kinds every shipped config uses.  Context features (utils.py:84-110, 155-170):
    ``embedding_continuous_context`` (``nn.Linear`` for the reference's kind "Embedding", identity for None), same attribute
    name and construction order as the reference so checkpoints and seeded random-init weights match."""

    def __init__(self, config):
        super().__init__()
        d, e = config.data, config.encoder
        if e.embedding_time != "SinusoidalPositionalEncoding":
            raise NotImplementedError("native path supports embedding_time=SinusoidalPositionalEncoding only")
        if e.embedding_features_continuous != "Linear" or e.embedding_features_discrete != "Embedding":
            raise NotImplementedError("native path supports Linear continuous / Embedding discrete feature embeddings")
        if d.dim_features_discrete != 1:
            raise NotImplementedError("one discrete token per particle (dim_features_discrete=1)")
        self.embedding_time = SinusoidalPositionalEncoding(e.dim_emb_time, max_period=10000)
        dim_cont_emb = e.dim_emb_features_continuous or d.dim_features_continuous
        self.embedding_continuous = nn.Linear(d.dim_features_continuous, dim_cont_emb)
        self.embedding_discrete = nn.Embedding(d.vocab_size_features, e.dim_emb_features_discrete)
        self.dim_context = 0   # width of the embedded context behind the time embedding
        if d.dim_context_continuous:
            kind = e.embedding_context_continuous
            if kind == "Embedding":
                width = e.dim_emb_context_continuous or d.dim_context_continuous
                self.embedding_continuous_context = nn.Linear(d.dim_context_continuous, width)
            elif kind is None:
                width = d.dim_context_continuous
                self.embedding_continuous_context = nn.Identity()
            else:
                raise NotImplementedError("embedding_context_continuous: 'Embedding' (a Linear layer in the reference) or None")
            self.dim_context += width
        if d.dim_context_discrete and e.dim_emb_context_discrete:
            # The reference cannot run such a model: the constructor stores the module as `embedding_context_discrete`
            # (utils.py:100-106), forward looks for `embedding_discrete_context` (utils.py:161), the embedding is never appended
            # and global_0 fails with a shape error.  Nothing to be a drop-in for.
            raise NotImplementedError("discrete context features: the reference's forward never applies their embedding "
                                      "(utils.py:100 vs utils.py:161) and fails for dim_emb_context_discrete > 0")

    @torch.no_grad()
    def context(self, context_continuous, context_discrete, device) -> Optional[torch.Tensor]:
        """The part of the reference's per-jet ``context`` vector behind the time embedding (utils.py:155-170): [B, dim_context]
        fp32 on ``device`` — a Linear / table lookup on a few numbers per jet, once per call."""
        return self.embedded_context(context_continuous, context_discrete, device)

    def embedded_context(self, context_continuous, context_discrete, device) -> Optional[torch.Tensor]:
        """``context`` under the caller's grad mode: with gradients on, the result carries the graph of the context embedding."""
        if not self.dim_context:
            return None
        parts = []
        home = self.embedding_discrete.weight.device   # evaluated where the parameters live; only the result moves
        if hasattr(self, "embedding_continuous_context"):
            if context_continuous is None:
                raise ValueError("the model was built with dim_context_continuous > 0: batch.context_continuous is required")
            c = context_continuous.to(home, torch.float32)
            parts.append(self.embedding_continuous_context(c.reshape(c.shape[0], -1)))
        return torch.cat(parts, dim=-1).float().to(device).contiguous()


class EPiC_Projection(nn.Module):
    def __init__(self, dim_local, dim_global, dim_hidden_local, dim_hidden_global):
        super().__init__()
        self.local_0 = WeightNormLinear(dim_local, dim_hidden_local)
        self.global_0 = WeightNormLinear(2 * dim_hidden_local + dim_global, dim_hidden_local)
        self.global_1 = WeightNormLinear(dim_hidden_local, dim_hidden_local)
        self.global_2 = WeightNormLinear(dim_hidden_local, dim_hidden_global)


class EPiC_layer(nn.Module):
    def __init__(self, dim_local, dim_global, dim_hidden, dim_context):
        super().__init__()
        self.fc_global1 = WeightNormLinear(2 * dim_local + dim_global + dim_context, dim_hidden)
        self.fc_global2 = WeightNormLinear(dim_hidden, dim_global)
        self.fc_local1 = WeightNormLinear(dim_local + dim_global + dim_context, dim_hidden)
        self.fc_local2 = WeightNormLinear(dim_hidden, dim_local)


class EPiCNetwork(nn.Module):
    def __init__(self, dim_input, dim_output, dim_context, num_blocks, dim_hidden_local, dim_hidden_global,
                 use_skip_connection):
        super().__init__()
        self.num_blocks, self.use_skip_connection = num_blocks, use_skip_connection
        self.epic_proj = EPiC_Projection(dim_input, dim_context, dim_hidden_local, dim_hidden_global)
        self.epic_layers = nn.ModuleList(
            [EPiC_layer(dim_hidden_local, dim_hidden_global, dim_hidden_local, dim_context) for _ in range(num_blocks)])
        self.output_layer = WeightNormLinear(dim_hidden_local, dim_output)


def as_u8(t: torch.Tensor) -> torch.Tensor:
    """[B,N,1] int64 tokens / masks of the reference -> contiguous [B,N] uint8 for the kernels."""
    return t.reshape(t.shape[0], t.shape[1]).to(torch.uint8).contiguous()


class EPiCWrapper(nn.Module):
    """epic.py:10-91: ``forward(t, x, k, mask, context_continuous, context_discrete,
    output_hidden_local)`` -> ``h [B,N,Dc+S]`` (masked), optionally also the last local hidden."""

    def __init__(self, config):
        super().__init__()
        d, e = config.data, config.encoder
        self.dim_features_continuous = d.dim_features_continuous
        self.dim_features_discrete = d.dim_features_discrete
        self.vocab_size = d.vocab_size_features
        self.embedding = InputEmbeddings(config)
        dim_cont_emb = e.dim_emb_features_continuous or d.dim_features_continuous
        self.epic = EPiCNetwork(
            dim_input=e.dim_emb_time + dim_cont_emb + e.dim_emb_features_discrete,
            dim_output=d.dim_features_continuous + d.dim_features_discrete * d.vocab_size_features,
            dim_context=e.dim_emb_time + self.embedding.dim_context,
            num_blocks=e.num_blocks,
            dim_hidden_local=e.dim_hidden_local,
            dim_hidden_global=e.dim_hidden_glob,
            use_skip_connection=e.skip_connection,
        )
        self.precision = "fp32"
        self._dims = dict(dim_continuous=d.dim_features_continuous, vocab_size=d.vocab_size_features,
                          dim_time_emb=e.dim_emb_time, dim_cont_emb=dim_cont_emb,
                          dim_disc_emb=e.dim_emb_features_discrete, dim_hidden_local=e.dim_hidden_local,
                          dim_hidden_glob=e.dim_hidden_glob, num_blocks=e.num_blocks,
                          skip_connection=int(bool(e.skip_connection)), dim_context=self.embedding.dim_context)
        self._cache = {}

    # ---- packing -----------------------------------------------------------------------------
    def epic_dims(self, disc_head_hidden: int = 0) -> _native.EpicDims:
        return _native.EpicDims(**self._dims, disc_head_hidden=disc_head_hidden)

    def _blob_parts(self, head: Optional[nn.Sequential], fold) -> list:
        """The tensors of the blob in ``mmb_epic_layout`` order (include/mmbridge.h); ``fold`` gives a layer's folded weight."""
        emb, net = self.embedding, self.epic
        parts = [emb.embedding_continuous.weight, emb.embedding_continuous.bias, emb.embedding_discrete.weight]
        proj = net.epic_proj
        layers = [proj.local_0, proj.global_0, proj.global_1, proj.global_2]
        for block in net.epic_layers:
            layers += [block.fc_global1, block.fc_global2, block.fc_local1, block.fc_local2]
        for layer in layers + [net.output_layer]:
            parts.extend([fold(layer), layer.bias])
        if head is not None:
            parts.extend([head[0].weight, head[0].bias, head[2].weight, head[2].bias])
        return parts

    def pack_weights(self, head: Optional[nn.Sequential] = None) -> torch.Tensor:
        """Flat fp32 blob in the order of ``mmb_epic_layout`` (include/mmbridge.h)."""
        parts = self._blob_parts(head, WeightNormLinear.folded)
        return torch.cat([p.detach().to("cpu", torch.float32).reshape(-1) for p in parts])

    def packed_parameters(self, head: Optional[nn.Sequential] = None) -> torch.Tensor:
        """The blob of ``pack_weights`` as a differentiable fp32 tensor on the parameters' device: the weight norm is folded by
        ``torch._weight_norm`` under autograd, so a gradient of the blob reaches ``weight_g`` and ``weight_v``."""
        fold = lambda layer: torch._weight_norm(layer.weight_v.float(), layer.weight_g.float(), 0)
        return torch.cat([p.float().reshape(-1) for p in self._blob_parts(head, fold)])

    def native_model(self, device, head: Optional[nn.Sequential] = None) -> _native.EpicModel:
        """Device-resident packed model; rebuilt when any parameter changed (optimizer step,
        ``load_state_dict``) or the device differs."""
        params = list(self.parameters()) + (list(head.parameters()) if head is not None else [])
        stamp = (str(device), head is not None, tuple(p._version for p in params), tuple(p.data_ptr() for p in params))
        key = "head" if head is not None else "trunk"
        hit = self._cache.get(key)
        if hit is None or hit[0] != stamp:
            hidden = head[0].out_features if head is not None else 0
            model = _native.EpicModel(self.epic_dims(hidden), self.pack_weights(head), device)
            self._cache[key] = (stamp, model)
        return self._cache[key][1]

    # ---- evaluation --------------------------------------------------------------------------
    def time_embedding(self, t: torch.Tensor) -> torch.Tensor:
        """t [B,1] (generation) or [B,1,1] (training) -> [B,T] on t's device.  Evaluated on the host
        (B floats) so the sin/cos are the same libm values whichever device the caller uses; the
        generation loop does not come through here (it uses the precomputed step table)."""
        emb = self.embedding.embedding_time(t.detach().reshape(t.shape[0]).float().cpu())
        return emb.contiguous().to(t.device)

    def context_rows(self, t, context_continuous=None, context_discrete=None, device=None) -> torch.Tensor:
        """The reference's per-jet context vector [time embedding | embedded context] (utils.py:133-170), [B, T + X]."""
        device = device or t.device
        rows = self.time_embedding(t).to(device)
        ctx = self.embedding.context(context_continuous, context_discrete, device)
        return rows if ctx is None else torch.cat([rows, ctx], dim=-1).contiguous()

    def forward(self, t, x, k=None, mask=None, context_continuous=None, context_discrete=None,
                output_hidden_local=False):
        model = self.native_model(x.device)
        v, z, hidden = model.forward(x.contiguous().float(), as_u8(k), as_u8(mask),
                                     self.context_rows(t, context_continuous, context_discrete, x.device),
                                     want_hidden=True, precision=self.precision)
        h = torch.cat([v, z], dim=-1)
        return (h, hidden) if output_hidden_local else h
