"""MultiModalBridgeMatching — drop-in for the generation side of
mp/models/generative/multimodal_bridge_matching.py (:77-146, 199-216, 252-257).

Same constructor argument (``MultimodalBridgeMatchingConfig``), same ``forward(state, batch)``,
``simulate_dynamics(state, batch)`` and ``predict_step(batch, batch_idx)`` signatures, same output
containers and tensor layouts, same state-dict keys.  The compute is libmmbridge.so: the loop in
``simulate_dynamics`` is ONE call of ``mmb_generate`` with the state resident on the GPU, instead
of ~725 eager ops and 4 host syncs per step (SURVEY.md §3.1).  Training: ``sample_bridges`` and
``bridge_matching_losses`` (differentiable, native backward pass) make a training step in a user's loop; ``training_step`` and
``configure_optimizers`` are not wired and raise (SURVEY.md §8f N2).
"""
from types import SimpleNamespace

import torch
from torch import nn

from . import _native
from .bridges import LinearUniformBridge, TelegraphBridge
from .epic import EPiCWrapper, as_u8
from .sharding import next_jet_offset
from .states import HybridState, MultiHeadOutput
from .steptable import build_step_table

try:  # Lightning is optional: with it the class plugs into Trainer.predict as the reference does
    import lightning as L
    _ModuleBase = L.LightningModule
except Exception:  # pragma: no cover - lightning is not in this image
    class _ModuleBase(nn.Module):
        def save_hyperparameters(self, *args, **kwargs):
            pass

        def log(self, *args, **kwargs):
            pass

        @property
        def device(self):
            try:
                return next(self.parameters()).device
            except StopIteration:
                return torch.device("cpu")


class MultiHeadLoss(nn.Module):
    """Holds ``loss_multihead.weights`` so reference checkpoints load (mp/utils/losses.py:9-20)."""

    def __init__(self, number_of_losses=2):
        super().__init__()
        self.weights = nn.Parameter(torch.zeros(number_of_losses))

    def forward(self, losses):
        """'learnable' mode of the reference: sum_i exp(-w_i) L_i + w_i  (mp/utils/losses.py:21-29)"""
        w = self.weights.to(losses[0].device)
        return sum(torch.exp(-w[i]) * losses[i] + w[i] for i in range(len(losses))), losses


class MultiModalEPiC(nn.Module):
    """EPiC trunk + discrete head ``Linear -> SELU -> Linear`` on the logit slice (mbm.py:77-113)."""

    def __init__(self, config):
        super().__init__()
        d = config.data
        self.dim_features_continuous = d.dim_features_continuous
        self.dim_features_discrete = d.dim_features_discrete
        self.vocab_size = d.vocab_size_features
        self.output_dim = d.dim_features_continuous + d.dim_features_discrete * d.vocab_size_features
        self.epic = EPiCWrapper(config)
        self.add_discrete_head = config.encoder.add_discrete_head
        if self.add_discrete_head:
            width = d.dim_features_discrete * d.vocab_size_features
            self.fc_layer = nn.Sequential(nn.Linear(width, width), nn.SELU(), nn.Linear(width, width))
        self.precision = "fp32"

    def native_model(self, device) -> _native.EpicModel:
        return self.epic.native_model(device, self.fc_layer if self.add_discrete_head else None)

    def forward(self, t, x, k, mask=None, context_continuous=None, context_discrete=None):
        model = self.native_model(x.device)
        v, logits = model.forward(x.contiguous().float(), as_u8(k), as_u8(mask),
                                  self.epic.context_rows(t, context_continuous, context_discrete, x.device), precision=self.precision)
        return v, logits, mask


def to_host_async(t: torch.Tensor) -> torch.Tensor:
    """Device tensor -> pinned host tensor, asynchronous on the current stream (the caller synchronises once)."""
    out = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    out.copy_(t, non_blocking=True)
    return out


class _BridgeMatchingLosses(torch.autograd.Function):
    """(blob, embedded context) -> (loss_continuous, loss_discrete): one call of the native loss / gradient kernels; backward
    combines the two Jacobian rows with the incoming scalar gradients."""

    @staticmethod
    def forward(ctx, W, context, dims, x, k, mask, rows, x0, x1, k1):
        losses, jac, d_context = _native.epic_loss_grad(dims, W.detach().contiguous(), x, k, mask, rows, x0, x1, k1)
        ctx.save_for_backward(jac, d_context if d_context is not None else jac.new_empty(0))
        return losses[0].clone(), losses[1].clone()

    @staticmethod
    def backward(ctx, g_mse, g_ce):
        jac, d_context = ctx.saved_tensors
        d_w = g_mse * jac[0] + g_ce * jac[1]
        d_ctx = g_mse * d_context[0] + g_ce * d_context[1] if ctx.needs_input_grad[1] else None
        return (d_w, d_ctx) + (None,) * 8


class MultiModalBridgeMatching(_ModuleBase):
    """Model for hybrid data with varying size (mbm.py:115-269), generation side.

    ``precision`` of ``simulate_dynamics``: "fp32" = CUDA-core trunk, bit-identical to the CPU oracle; "bf16" = tcgen05
    engine; "f16" = warp-MMA engine (fp16 operands, fp32 accumulate: the fastest and the closest to fp32); "auto" (default)
    = the first of f16 / bf16 / fp32 that takes the model's shape.  ``forward`` always evaluates in fp32 unless asked.
    """

    def __init__(self, config, precision: str = "auto"):
        super().__init__()
        self.config = config
        self.vocab_size = config.data.vocab_size_features
        self.encoder = MultiModalEPiC(config)
        self.bridge_continuous = LinearUniformBridge(config)
        self.bridge_discrete = TelegraphBridge(config)
        self.bridge_absorbing = None
        self.loss_multihead = MultiHeadLoss(number_of_losses=2)
        self.precision = precision
        self.seed = 0           # Philox key of simulate_dynamics when no uniforms are injected
        # host -> host calls: 0 = direct mode (the generation kernel reads / writes the caller's page-locked buffers itself;
        # f16 engine, pinned tensors — anything else falls back to two slices); n > 0 = n slices of jets on their own streams,
        # when each slice has at least pipeline_min_jets jets
        self.pipeline_chunks = 0
        self.pipeline_min_jets = 1024
        self._jets_generated = 0
        self.save_hyperparameters()

    # ---- network ----------------------------------------------------------------------------
    def forward(self, state: HybridState, batch=None) -> MultiHeadOutput:
        continuous, discrete, absorbing = self.encoder(
            t=state.time, x=state.continuous, k=state.discrete, mask=state.absorbing,
            context_continuous=getattr(batch, "context_continuous", None),      # mbm.py:143-144
            context_discrete=getattr(batch, "context_discrete", None))
        return MultiHeadOutput(continuous, discrete, absorbing)

    # ---- generation -------------------------------------------------------------------------
    def step_table(self):
        """Per-step host scalars; cached (they depend on the bridge/encoder config only)."""
        b, e = self.config.bridge, self.config.encoder
        key = (b.num_timesteps, b.time_eps, self.vocab_size, b.gamma, e.dim_emb_time)
        if getattr(self, "_table_cache", None) is None or self._table_cache[0] != key:
            self._table_cache = (key, build_step_table(*key))
        return self._table_cache[1]

    @torch.no_grad()
    def simulate_dynamics(self, state: HybridState, batch=None, uniforms=None, precision=None,
                          jet_offset=None, return_device=False) -> HybridState:
        """Generate target data from the source state; returns the final state on the CPU,
        detached, like the reference (mbm.py:199-216).

        ``uniforms`` [T-1,B,N]: injected jump draws (parity); default: in-kernel Philox keyed by
        ``(self.seed, global jet index, step, particle)``.  The input state is consumed (the
        reference mutates it too); ``return_device=True`` skips the final D2H copy.
        """
        device = self._compute_device(state)
        table = self.step_table()
        k64 = state.discrete
        B, N = state.continuous.shape[0], state.continuous.shape[1]
        model = self.encoder.native_model(device)
        # embedded context features of the jets, constant over the steps (mbm.py:143-144 -> utils.py:155-170); None without
        on_host = (state.continuous.device.type == "cpu" and k64.device.type == "cpu" and state.absorbing.device.type == "cpu")
        embed_context = lambda where: self.encoder.epic.embedding.context(getattr(batch, "context_continuous", None),
                                                                          getattr(batch, "context_discrete", None), where)
        if on_host and uniforms is None and not return_device:
            # Host state in, host state out (what Trainer.predict does): ONE library call.  Direct mode: the kernel reads each
            # jet from the page-locked input and writes it to the page-locked output itself.  Sliced mode: H2D of slice c+1
            # and D2H of slice c-1 under the solver steps of slice c, tokens / masks narrowed and widened on the device.
            # Either way the reference's token-range assertion (bridges.py:111-115) is evaluated on the device, and Philox is
            # keyed by the global jet index, so the jets are bit-identical whatever the mode.
            if jet_offset is None:
                jet_offset = next_jet_offset(self, B)
            chunks = self.pipeline_chunks if B >= self.pipeline_chunks * self.pipeline_min_jets else 1   # 0 stays 0: direct mode
            x_host, k_host, flag, keep = model.generate_host(state.continuous, k64.reshape(B, N, 1), state.absorbing.reshape(B, N, 1), table,
                                                             seed=self.seed, jet_offset=jet_offset, chunks=chunks,
                                                             precision=precision or self.precision,
                                                             context=embed_context("cpu"))
            torch.cuda.current_stream(device).synchronize()
            del keep
            assert int(flag) == 0, "Values in `k` outside of bound! (0 <= k < {})".format(self.vocab_size)
            return HybridState(time=torch.full((B, 1), float(table.t[-1])), continuous=x_host, discrete=k_host,
                               absorbing=state.absorbing.detach())
        k_min, k_max = torch.aminmax(k64)   # the reference's assertion (bridges.py:111-115), one pass
        assert int(k_min) >= 0 and int(k_max) < self.vocab_size, \
            "Values in `k` outside of bound! k_min={}, k_max={}".format(int(k_min), int(k_max))
        x = state.continuous.to(device, torch.float32, non_blocking=True, copy=True).contiguous()
        k = as_u8(k64.to(device, non_blocking=True))
        mask = as_u8(state.absorbing.to(device, non_blocking=True))
        u = None if uniforms is None else uniforms.to(device, torch.float32).reshape(table.n_steps, B, N).contiguous()
        if jet_offset is None:
            jet_offset = next_jet_offset(self, B)
        model.generate(x, k, mask, table, u_jump=u, seed=self.seed, jet_offset=jet_offset,
                       precision=precision or self.precision, context=embed_context(device))
        t_last = float(table.t[-1])
        if return_device:
            return HybridState(time=torch.full((B, 1), t_last, device=device), continuous=x,
                               discrete=k.to(k64.dtype).unsqueeze(-1), absorbing=state.absorbing.to(device))
        # host result in the reference's layout: fp32 features and tokens widened to int64 on the device, into page-locked memory
        x_host, k_host = to_host_async(x), to_host_async(k.to(k64.dtype).unsqueeze(-1))
        torch.cuda.current_stream(device).synchronize()
        return HybridState(time=torch.full((B, 1), t_last), continuous=x_host, discrete=k_host,
                           absorbing=state.absorbing.detach().cpu())

    def predict_step(self, batch, batch_idx) -> HybridState:
        initial_state = HybridState(None, batch.source_continuous, batch.source_discrete, batch.source_mask)
        return self.simulate_dynamics(initial_state, batch)

    def _compute_device(self, state) -> torch.device:
        dev = self.device
        if dev.type != "cuda":
            dev = state.continuous.device
        if dev.type != "cuda":
            if not torch.cuda.is_available():
                raise _native.MmbError("generation needs a CUDA device: libmmbridge has no CPU path")
            dev = torch.device("cuda", torch.cuda.current_device())
        return dev

    # ---- forward half of a training / validation step (SURVEY.md §8f N2) ---------------------------------
    def reshape_time(self, t, x):
        return t if isinstance(t, (float, int)) else t.reshape(-1, *([1] * (x.dim() - 1)))

    @torch.no_grad()
    def sample_bridges(self, batch, t=None, z=None, u=None) -> HybridState:
        """Sample stochastic bridges (mbm.py:148-165): ``t ~ U(0,1)`` per jet, ``x_t = t x1 + (1-t) x0 + sigma z`` and
        ``k_t ~ telegraph posterior`` in one kernel.  ``t`` [B], ``z`` [B,N,3], ``u`` [B,N] inject the draws (parity);
        default: torch.rand for the times, in-kernel Philox for the rest."""
        device = self._compute_device(SimpleNamespace(continuous=batch.target_continuous))
        x1 = batch.target_continuous.to(device, torch.float32).contiguous()
        x0 = batch.source_continuous.to(device, torch.float32).contiguous()
        B = x1.shape[0]
        t = torch.rand(B, device=device) if t is None else t.to(device, torch.float32).contiguous()
        prep = lambda a: None if a is None else a.to(device, torch.float32).contiguous()
        jet_offset = next_jet_offset(self, B, "_bridges_sampled")
        xt, kt = _native.sample_bridges(x0, x1, as_u8(batch.source_discrete.to(device)), as_u8(batch.target_discrete.to(device)), t,
                                        self.bridge_continuous.sigma, self.bridge_discrete.gamma, self.vocab_size, prep(z), prep(u),
                                        seed=self.seed, jet_offset=jet_offset)
        return HybridState(self.reshape_time(t, x1), xt, kt.long().unsqueeze(-1), batch.target_mask.to(device))

    @torch.no_grad()
    def _losses(self, heads: MultiHeadOutput, state: HybridState, batch) -> torch.Tensor:
        dev = heads.continuous.device
        f = lambda a: a.to(dev, torch.float32).contiguous()
        return _native.bridge_losses(f(heads.continuous), f(heads.discrete), f(batch.source_continuous), f(batch.target_continuous),
                                     as_u8(batch.target_discrete.to(dev)), as_u8(state.absorbing.to(dev)))

    def loss_continuous(self, heads: MultiHeadOutput, state: HybridState, batch) -> torch.Tensor:
        """masked mean square error of the drift (mbm.py:167-183); forward value only (no autograd)"""
        return self._losses(heads, state, batch)[0]

    def loss_discrete(self, heads: MultiHeadOutput, state: HybridState, batch) -> torch.Tensor:
        """masked cross entropy of the token classifier (mbm.py:185-197); forward value only (no autograd)"""
        return self._losses(heads, state, batch)[1]

    def bridge_matching_losses(self, state: HybridState, batch):
        """``(loss_continuous, loss_discrete)`` of the network on the bridge state (mbm.py:167-197), differentiable with respect
        to every parameter of the encoder: ``backward()`` fills ``.grad`` under the reference's state-dict keys (``…weight_g``,
        ``…weight_v``, ``…bias``, the embeddings, ``encoder.fc_layer.*``, ``embedding_continuous_context.*``).  The network,
        both losses and both gradients are one pass of the native fp32 kernels (``mmb_epic_loss_grad``); torch adds the weight-norm
        chain rule and the context embedding.  A user's loop does what the reference's ``training_step`` does (mbm.py:232-240)::

            state = model.sample_bridges(batch)
            l0, l1 = model.bridge_matching_losses(state, batch)
            loss, _ = model.loss_multihead([l0, l1])
            loss.backward()
            opt.step()

        ``training_step`` and ``configure_optimizers`` still raise: wiring the Lightning step, the optimiser and its gradient
        clipping is separate work.  Under ``torch.no_grad()`` the same values come without building the Jacobian."""
        epic = self.encoder.epic
        head = self.encoder.fc_layer if self.encoder.add_discrete_head else None
        dev = self._compute_device(SimpleNamespace(continuous=state.continuous))
        dims = epic.epic_dims(head[0].out_features if head is not None else 0)
        f32 = lambda a: a.to(dev, torch.float32).contiguous()
        u8 = lambda a: as_u8(a.to(dev))
        x, k, mask = f32(state.continuous), u8(state.discrete), u8(state.absorbing)
        x0, x1, k1 = f32(batch.source_continuous), f32(batch.target_continuous), u8(batch.target_discrete)
        cc, cd = getattr(batch, "context_continuous", None), getattr(batch, "context_discrete", None)
        if not torch.is_grad_enabled():
            rows = epic.context_rows(state.time, cc, cd, dev)
            W = epic.packed_parameters(head).to(dev).contiguous()
            losses, _, _ = _native.epic_loss_grad(dims, W, x, k, mask, rows, x0, x1, k1, jacobian=False)
            return losses[0], losses[1]
        context = epic.embedding.embedded_context(cc, cd, dev)   # under autograd: the context Linear gets its gradient
        rows = epic.time_embedding(state.time).to(dev)
        if context is not None:
            rows = torch.cat([rows, context.detach()], dim=-1).contiguous()
        W = epic.packed_parameters(head).to(dev)
        return _BridgeMatchingLosses.apply(W, context, dims, x, k, mask, rows, x0, x1, k1)

    @torch.no_grad()
    def validation_step(self, batch, batch_idx=0) -> torch.Tensor:
        """mbm.py:241-250: bridges -> heads -> the two losses -> learnable multi-head weighting (forward only)."""
        state = self.sample_bridges(batch)
        heads = self.forward(state, batch)
        both = self._losses(heads, state, batch)
        loss, _ = self.loss_multihead([both[0], both[1]])
        return loss

    # ---- not wired yet: a user's loop over bridge_matching_losses does what training_step does ----------------
    def _training_not_in_scope(self, *args, **kwargs):
        raise NotImplementedError("the Lightning training step / optimiser are not wired: call bridge_matching_losses, "
                                  "loss_multihead and backward() in your own loop (SURVEY.md §8f N2)")

    training_step = configure_optimizers = _training_not_in_scope
