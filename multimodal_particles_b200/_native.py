"""ctypes binding of libmmbridge.so (include/mmbridge.h).

There is no CPU fallback: if the library is missing or a call fails, this raises.  PyTorch is used
only for device memory and streams; every pointer handed over is a ``data_ptr()`` of a contiguous
CUDA tensor and every launch goes to ``torch.cuda.current_stream()``.
"""
import ctypes
import os
from typing import Optional

import torch

from .steptable import CStepTable

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MMB_LIB_PATH") or os.path.join(_HERE, "csrc", "libmmbridge.so")   # MMB_LIB_PATH: a differently built copy (kernel experiments)

FLAG_MULTIMODAL = 0
FLAG_ABSORBING = 1
PREC_FP32 = 0
PREC_BF16 = 1
PREC_F16 = 2
# "bf16" = tcgen05 engine; "f16" = warp-MMA engine (generation only; fp16 operands, fp32 accumulate)
PRECISIONS = {"fp32": PREC_FP32, "bf16": PREC_BF16, "f16": PREC_F16}


class MmbError(RuntimeError):
    pass


class EpicDims(ctypes.Structure):
    """ctypes image of ``MmbEpicDims``."""

    _fields_ = [(n, ctypes.c_int32) for n in (
        "dim_continuous", "vocab_size", "dim_time_emb", "dim_cont_emb", "dim_disc_emb",
        "dim_hidden_local", "dim_hidden_glob", "num_blocks", "skip_connection", "disc_head_hidden", "dim_context")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class TransDims(ctypes.Structure):
    """ctypes image of ``MmbTransDims``."""

    _fields_ = [(n, ctypes.c_int32) for n in ("hidden", "vocab_size", "transformer_dim", "n_heads", "n_blocks", "max_particles", "rate_direct")]


class ForwardRate(ctypes.Structure):
    """ctypes image of ``MmbForwardRate`` (kind 0 = step, 1 = const)."""

    _fields_ = [("kind", ctypes.c_int32), ("scalar", ctypes.c_float), ("offset", ctypes.c_float), ("rate_cut_t", ctypes.c_float)]


_fptr = ctypes.POINTER(ctypes.c_float)


class JumpSchedule(ctypes.Structure):
    """ctypes image of ``MmbJumpSchedule``; keeps the numpy arrays it points into alive."""

    _fields_ = [("n_steps", ctypes.c_int32), ("ts", _fptr), ("c_decay", _fptr), ("c_score", _fptr), ("c_noise", _fptr),
                ("inv_std", _fptr), ("jump_dt", ctypes.c_float), ("kind", ctypes.POINTER(ctypes.c_uint8)), ("death_prob", _fptr),
                ("corrector_snr", ctypes.c_float), ("jump_corrector", ctypes.c_int32)]

    @classmethod
    def from_schedule(cls, sched):
        import numpy as np
        keep = [np.ascontiguousarray(getattr(sched, n), dtype=np.float32) for n in ("ts", "c_decay", "c_score", "c_noise", "inv_std")]
        kind = getattr(sched, "kind", None)
        kind_p, death_p = None, None
        if kind is not None and np.any(kind):
            kind = np.ascontiguousarray(kind, dtype=np.uint8)
            death = np.ascontiguousarray(sched.death_prob, dtype=np.float32)
            keep += [kind, death]
            kind_p, death_p = kind.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), death.ctypes.data_as(_fptr)
        out = cls(int(sched.n_steps), *[a.ctypes.data_as(_fptr) for a in keep[:5]], float(sched.jump_dt), kind_p, death_p,
                  float(getattr(sched, "corrector_snr", 0.0)), int(bool(getattr(sched, "jump_corrector", False))))
        out._keep = keep
        return out


_lib = None

# name -> (restype, argtypes); lists every symbol include/mmbridge.h declares
_vp, _i, _f, _sz, _u64, _i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t, ctypes.c_uint64, ctypes.c_int64
SIGNATURES = {
    "mmb_abi_version": (_i, []),
    "mmb_last_error": (ctypes.c_char_p, []),
    "mmb_epic_packed_floats": (_sz, [ctypes.POINTER(EpicDims)]),
    "mmb_epic_create": (_i, [ctypes.POINTER(EpicDims), _vp, _sz, _i, ctypes.POINTER(_vp)]),
    "mmb_epic_destroy": (None, [_vp]),
    "mmb_epic_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "mmb_bridge_update": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _i, _i, _i, _i, _i, _vp]),
    "mmb_generate_workspace_bytes": (_sz, [_vp, _i, _i, _i]),
    "mmb_generate_supported": (_i, [_vp, _i, _i]),
    "mmb_generate": (_i, [_vp, _vp, _vp, _vp, _vp, ctypes.POINTER(CStepTable), _vp, _u64, _u64, _i, _i, _vp, _sz, _i, _vp]),
    "mmb_generate_host_workspace_bytes": (_sz, [_vp, _i, _i, _i, _i, _i]),
    "mmb_generate_host": (_i, [_vp, _vp, _vp, _vp, _vp, ctypes.POINTER(CStepTable), _u64, _u64, _i, _i, _vp, _vp, _vp, _vp, _sz, _i, _i, _vp]),
    "mmb_jump_variants": (_i, [_vp, _vp, _vp, _f, _f, _f, _sz, _i, _vp, _vp, _vp, _vp]),
    "mmb_philox_uniforms": (_i, [_vp, _u64, _u64, _i, _i, _i, _vp]),
    "mmb_absorb_head_create": (_i, [_i, _i, _i, _i, _vp, _sz, _i, ctypes.POINTER(_vp)]),
    "mmb_absorb_head_destroy": (None, [_vp]),
    "mmb_absorb_head_workspace_bytes": (_sz, [_i]),
    "mmb_absorb_head_forward": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "mmb_generate_absorbing_workspace_bytes": (_sz, [_vp, _vp, _i, _i, _i]),
    "mmb_generate_absorbing": (_i, [_vp, _vp, _vp, _vp, _vp, ctypes.POINTER(CStepTable), _vp, _vp, _vp, _u64, _u64, _i, _i,
                                    _vp, _sz, _i, _vp]),
    "mmb_validation_histograms": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _f, _i, _vp, _vp]),
    "mmb_jet_observables": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "mmb_jet_substructure": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _f, _vp, _vp, _vp]),
    "mmb_wasserstein1d_workspace_bytes": (_sz, [_i, _i, _i]),
    "mmb_wasserstein1d": (_i, [_vp, _i64, _i, _vp, _i64, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "mmb_wasserstein1d_drawn_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "mmb_wasserstein1d_drawn": (_i, [_vp, _i64, _i64, _vp, _i64, _i, _vp, _i64, _i64, _vp, _i64, _i, _i, _i, _vp, _vp, _i, _i,
                                     _vp, _vp, _vp, _sz, _vp]),
    "mmb_energy_flow_polynomials": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _vp, _vp]),
    "mmb_energy_flow_polynomials_d4": (_i, [_vp, _vp, _vp, _vp, _i, _i, _f, _vp, _vp]),
    "mmb_sampled_moments": (_i, [_vp, _i64, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "mmb_kpd_mmd_workspace_bytes": (_sz, [_i, _i, _i]),
    "mmb_kpd_mmd": (_i, [_vp, _i64, _i, _vp, _i64, _i, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "mmb_sample_source": (_i, [_vp, _vp, _vp, _i, _i, _f, _vp, _vp, _u64, _u64, _vp]),
    "mmb_sample_bridges": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _f, _i, _vp, _vp, _u64, _u64, _i, _i, _vp, _vp, _vp]),
    "mmb_absorbing_sample": (_i, [_vp, _vp, _vp, _u64, _u64, _i, _i, _vp, _vp]),
    "mmb_bridge_losses_workspace_bytes": (_sz, [_i, _i]),
    "mmb_bridge_losses": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "mmb_epic_loss_grad_workspace_bytes": (_sz, [ctypes.POINTER(EpicDims), _i, _i]),
    "mmb_epic_loss_grad": (_i, [ctypes.POINTER(EpicDims), _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _sz,
                                _vp]),
    "mmb_trans_packed_floats": (_sz, [ctypes.POINTER(TransDims)]),
    "mmb_trans_create": (_i, [ctypes.POINTER(TransDims), _vp, _sz, _i, ctypes.POINTER(_vp)]),
    "mmb_trans_destroy": (None, [_vp]),
    "mmb_trans_forward_workspace_bytes": (_sz, [_vp, _vp, _i, _i]),
    "mmb_trans_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.POINTER(ForwardRate), _i, _i,
                               _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "mmb_trans_sample_workspace_bytes": (_sz, [_vp, _vp, _i, _i]),
    "mmb_trans_sample": (_i, [_vp, _vp, _vp, _vp, _vp, ctypes.POINTER(JumpSchedule), ctypes.POINTER(ForwardRate),
                              _vp, _vp, _vp, _vp, _vp, _u64, _u64, _i, _i, _vp, _sz, _i, _vp]),
    "mmb_trans_sampler_update": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _f, _vp, _vp, _vp,
                                      _u64, _u64, _i, _i, _i, _i, _vp]),
    "mmb_trans_corrector_update": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _f, _f, _f, _i, _f, _vp, _vp, _vp, _vp,
                                        _u64, _u64, _i, _i, _i, _i, _vp, _vp]),
}


def load():
    """Load the library once; raise loudly when it has not been built
    (``python -c 'import __graft_entry__ as g; g.build()'``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MmbError(f"{LIB_PATH} not built: the generation path has no CPU fallback")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc: int):
    if rc != 0:
        raise MmbError(f"libmmbridge error {rc}: {load().mmb_last_error().decode()}")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and (not t.is_cuda or not t.is_contiguous()):
            raise MmbError("libmmbridge takes contiguous CUDA tensors; there is no CPU path")


class EpicModel:
    """Owner of one ``MmbEpicModel*`` (device-resident weights)."""

    def __init__(self, dims: EpicDims, packed: torch.Tensor, device: torch.device):
        lib = load()
        packed = packed.detach().to("cpu", torch.float32).contiguous()
        expect = lib.mmb_epic_packed_floats(ctypes.byref(dims))
        if packed.numel() != expect:
            raise MmbError(f"packed weight blob has {packed.numel()} floats, layout wants {expect}")
        self.dims, self.device = dims, torch.device(device)
        self._handle = ctypes.c_void_p()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        check(lib.mmb_epic_create(ctypes.byref(dims), _ptr(packed), packed.numel(), index, ctypes.byref(self._handle)))

    def __del__(self):
        if getattr(self, "_handle", None) and _lib is not None:
            _lib.mmb_epic_destroy(self._handle)
            self._handle = None

    def forward(self, x, k_u8, mask_u8, temb, want_hidden=False, precision="fp32"):
        """x [B,N,Dc] f32, k/mask [B,N] u8, temb [B,T+X] or [1,T+X] (time embedding, then the jet's embedded context if the
        model has context features) -> (v, logits[, hidden])."""
        _require_cuda(x, k_u8, mask_u8, temb)
        B, N, _ = x.shape
        d = self.dims
        v = torch.empty(B, N, d.dim_continuous, device=x.device, dtype=torch.float32)
        logits = torch.empty(B, N, d.vocab_size, device=x.device, dtype=torch.float32)
        hidden = torch.empty(B, N, d.dim_hidden_local, device=x.device, dtype=torch.float32) if want_hidden else None
        width = d.dim_time_emb + d.dim_context
        if temb.shape[-1] != width:
            raise MmbError(f"context rows must hold {d.dim_time_emb} time + {d.dim_context} context entries, got {temb.shape[-1]}")
        stride = 0 if temb.shape[0] == 1 and B != 1 else width
        with torch.cuda.device(x.device):
            check(load().mmb_epic_forward(self._handle, _ptr(x), _ptr(k_u8), _ptr(mask_u8), _ptr(temb), stride, B, N,
                                          _ptr(v), _ptr(logits), _ptr(hidden), PRECISIONS[precision], _stream()))
        return (v, logits, hidden) if want_hidden else (v, logits)

    def generate_precision(self, N, precision="auto"):
        """Resolve "auto" to the fastest engine that takes this model at N particles per jet: warp-MMA fp16, tcgen05 bf16,
        CUDA-core fp32 (any shape)."""
        if precision != "auto":
            return precision
        lib = load()
        for name in ("f16", "bf16", "fp32"):
            if lib.mmb_generate_supported(self._handle, N, PRECISIONS[name]):
                return name
        return "fp32"

    def _context(self, context, B):
        X = self.dims.dim_context
        if (context is None) != (X == 0):
            raise MmbError(f"the model has {X} context features, context {'missing' if context is None else 'given'}")
        if context is None:
            return None
        if tuple(context.shape) != (B, X) or context.dtype != torch.float32 or not context.is_contiguous():
            raise MmbError(f"context must be a contiguous float32 [{B}, {X}] tensor")
        return context

    def generate(self, x, k_u8, mask_u8, table, u_jump=None, seed=0, jet_offset=0, precision="auto", context=None):
        """In-place generation of x/k over all steps of ``table`` (StepTable); ``context`` [B,X] f32: embedded context
        features of the jets (models built with ``dim_context`` > 0)."""
        _require_cuda(x, k_u8, mask_u8, u_jump, context)
        B, N, _ = x.shape
        context = self._context(context, B)
        lib = load()
        prec = PRECISIONS[self.generate_precision(N, precision)]
        need = lib.mmb_generate_workspace_bytes(self._handle, B, N, prec)
        ws = torch.empty(max(need, 16), device=x.device, dtype=torch.uint8)
        ctable = CStepTable.from_table(table)
        with torch.cuda.device(x.device):
            check(lib.mmb_generate(self._handle, _ptr(x), _ptr(k_u8), _ptr(mask_u8), _ptr(context), ctypes.byref(ctable), _ptr(u_jump),
                                   seed, jet_offset, B, N, _ptr(ws), ws.numel(), prec, _stream()))
        return x, k_u8


    def generate_host(self, x_host, k64_host, m64_host, table, seed=0, jet_offset=0, chunks=0, precision="auto", context=None):
        """Host state in the reference's layout (fp32 [B,N,Dc], int64 [B,N,1] tokens and masks) -> pinned host result
        (x [B,N,Dc] f32, k [B,N,1] int64, flag [1] int32: 1 = a token was out of range), asynchronous on the current stream of
        this model's device: ONE library call (direct mode for ``chunks=0``, else the sliced H2D / generate / D2H pipeline).
        The host-side work of a call is kept to one page-locked allocation and the call itself (it is on the critical path
        of a 1 ms generation)."""
        B, N, Dc = x_host.shape
        lib = load()
        dev = self.device
        prec = PRECISIONS[self.generate_precision(N, precision)]
        fix = lambda t, dt: t if (t.dtype == dt and t.is_contiguous()) else t.to(dt).contiguous()
        x_in, k_in, m_in = fix(x_host, torch.float32), fix(k64_host, torch.int64), fix(m64_host, torch.int64)
        c_in = None if context is None else self._context(fix(context.reshape(B, -1), torch.float32), B)   # host [B,X]
        if context is None:
            self._context(None, B)
        # one page-locked block: [x f32 | k int64 | flag], 16-byte aligned parts
        nx, nk = B * N * Dc * 4, B * N * 8
        block = torch.empty(nx + nk + 16, dtype=torch.uint8, pin_memory=True)
        x_out = block[:nx].view(torch.float32).view(B, N, Dc)
        k_out = block[nx:nx + nk].view(torch.int64).view(B, N, 1)
        flag = block[nx + nk:nx + nk + 4].view(torch.int32)
        key = (B, N, table.n_steps, chunks, prec)
        cache = self.__dict__.setdefault("_host_cache", {})
        need = cache.get(key)
        if need is None:
            need = cache[key] = lib.mmb_generate_host_workspace_bytes(self._handle, B, N, table.n_steps, chunks, prec)
        ws = getattr(self, "_host_ws", None)
        if ws is None or ws.numel() < need or ws.device != dev:
            ws = self._host_ws = torch.empty(max(need, 256), device=dev, dtype=torch.uint8)   # torch allocations are 512-byte aligned
        ctable = getattr(table, "_ctable", None)
        if ctable is None:
            ctable = table._ctable = CStepTable.from_table(table)
        stream = torch.cuda.current_stream(dev)
        rc = lib.mmb_generate_host(self._handle, x_in.data_ptr(), k_in.data_ptr(), m_in.data_ptr(), c_in.data_ptr() if c_in is not None else None,
                                   ctypes.byref(ctable), seed, jet_offset, B, N,
                                   x_out.data_ptr(), k_out.data_ptr(), flag.data_ptr(), ws.data_ptr(), ws.numel(), chunks, prec,
                                   stream.cuda_stream)
        check(rc)
        return x_out, k_out, flag, (x_in, k_in, m_in, c_in)   # the inputs must outlive the asynchronous copies


def bridge_update(x, k_u8, mask_u8, v, logits, u_jump, dt, bc, cc, absorb_logit=None, u_absorb=None, sp=0.0,
                  flags=FLAG_MULTIMODAL):
    """In-place fused Euler + telegraph jump (+ absorbing birth) on device tensors."""
    _require_cuda(x, k_u8, mask_u8, v, logits, u_jump, absorb_logit, u_absorb)
    B, N, Dc = x.shape
    S = logits.shape[-1] if logits is not None else 1
    with torch.cuda.device(x.device):
        check(load().mmb_bridge_update(_ptr(x), _ptr(k_u8), _ptr(mask_u8), _ptr(v), _ptr(logits), _ptr(absorb_logit),
                                       _ptr(u_jump), _ptr(u_absorb), dt, bc, cc, sp, B, N, Dc, S, flags, _stream()))


def jump_variants(logits, k_u8, u, dt, bc, cc):
    """Tokens chosen by the exact jump rule and by the fast variants of the tcgen05 / warp-MMA engines on identical inputs:
    logits [P,S] f32, k [P] u8, u [P] f32 (device) -> (exact, tc, mma) [P] u8."""
    _require_cuda(logits, k_u8, u)
    P, S = logits.shape
    outs = [torch.empty(P, dtype=torch.uint8, device=logits.device) for _ in range(3)]
    with torch.cuda.device(logits.device):
        check(load().mmb_jump_variants(_ptr(logits), _ptr(k_u8), _ptr(u), dt, bc, cc, P, S, *[_ptr(o) for o in outs], _stream()))
    return outs


def philox_uniforms(seed, jet_offset, n_steps, B, N, device):
    u = torch.empty(n_steps, B, N, device=device, dtype=torch.float32)
    with torch.cuda.device(device):
        check(load().mmb_philox_uniforms(_ptr(u), seed, jet_offset, n_steps, B, N, _stream()))
    return u


def validation_histograms(x, k_u8, mask_u8, counts, vocab_size, bins, lo, hi, max_mult):
    """Accumulate the validation histograms of (x, k, mask) into ``counts`` (int64, on device)."""
    _require_cuda(x, k_u8, mask_u8, counts)
    B, N, Dc = x.shape
    with torch.cuda.device(x.device):
        check(load().mmb_validation_histograms(_ptr(x), _ptr(k_u8), _ptr(mask_u8), B, N, Dc, vocab_size, bins, lo, hi,
                                               max_mult, _ptr(counts), _stream()))
    return counts


class AbsorbHead:
    """Owner of one ``MmbAbsorbHead*`` (device-resident transformer rate head)."""

    def __init__(self, hidden, transformer_dim, n_heads, n_blocks, packed: torch.Tensor, device):
        lib = load()
        packed = packed.detach().to("cpu", torch.float32).contiguous()
        self.device, self.n_blocks, self.dim = torch.device(device), n_blocks, transformer_dim
        self._handle = ctypes.c_void_p()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        check(lib.mmb_absorb_head_create(hidden, transformer_dim, n_heads, n_blocks, _ptr(packed), packed.numel(), index,
                                         ctypes.byref(self._handle)))

    def __del__(self):
        if getattr(self, "_handle", None) and _lib is not None:
            _lib.mmb_absorb_head_destroy(self._handle)
            self._handle = None

    def forward(self, hidden, mask_u8, tbias, pack=True):
        """hidden [B,N,H] f32, mask [B,N] u8, tbias [B or 1, n_blocks, C] -> rate logits [B,N].  ``pack``: padded slots once,
        several jets per tile (exact); False = one jet per tile, one row per slot."""
        hidden, tbias = hidden.contiguous(), tbias.contiguous()
        _require_cuda(hidden, mask_u8, tbias)
        B, N, _ = hidden.shape
        out = torch.empty(B, N, device=hidden.device, dtype=torch.float32)
        stride = 0 if tbias.shape[0] == 1 and B != 1 else self.n_blocks * self.dim
        lib = load()
        ws = torch.empty(max(lib.mmb_absorb_head_workspace_bytes(B), 16), device=hidden.device, dtype=torch.uint8) if pack else None
        with torch.cuda.device(hidden.device):
            check(lib.mmb_absorb_head_forward(self._handle, _ptr(hidden), _ptr(mask_u8), _ptr(tbias), stride, B, N, _ptr(out),
                                              _ptr(ws), ws.numel() if pack else 0, _stream()))
        return out


def generate_absorbing(trunk: EpicModel, head: AbsorbHead, x, k_u8, mask_u8, table, tbias_host, u_jump=None, u_absorb=None,
                       seed=0, jet_offset=0, precision="bf16"):
    """In-place absorbing-flow generation of x / k / mask over all steps of ``table``."""
    _require_cuda(x, k_u8, mask_u8, u_jump, u_absorb)
    B, N, _ = x.shape
    lib = load()
    tb = tbias_host.detach().to("cpu", torch.float32).contiguous()
    need = lib.mmb_generate_absorbing_workspace_bytes(trunk._handle, head._handle, B, N, table.n_steps)
    ws = torch.empty(max(need, 16), device=x.device, dtype=torch.uint8)
    ctable = CStepTable.from_table(table)
    with torch.cuda.device(x.device):
        check(lib.mmb_generate_absorbing(trunk._handle, head._handle, _ptr(x), _ptr(k_u8), _ptr(mask_u8), ctypes.byref(ctable),
                                         _ptr(tb), _ptr(u_jump), _ptr(u_absorb), seed, jet_offset, B, N, _ptr(ws), ws.numel(),
                                         PRECISIONS[precision], _stream()))
    return x, k_u8, mask_u8


# ---- trans-dimensional jump diffusion -----------------------------------------------------------------
class TransHeads:
    """Owner of one ``MmbTransHeads*`` (device-resident transformer stacks of TransdimensionalEPiC)."""

    def __init__(self, dims: TransDims, packed: torch.Tensor, device):
        lib = load()
        packed = packed.detach().to("cpu", torch.float32).contiguous()
        expect = lib.mmb_trans_packed_floats(ctypes.byref(dims))
        if packed.numel() != expect:
            raise MmbError(f"packed trans-heads blob has {packed.numel()} floats, layout wants {expect}")
        self.dims, self.device = dims, torch.device(device)
        self._handle = ctypes.c_void_p()
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        check(lib.mmb_trans_create(ctypes.byref(dims), _ptr(packed), packed.numel(), index, ctypes.byref(self._handle)))

    def __del__(self):
        if getattr(self, "_handle", None) and _lib is not None:
            _lib.mmb_trans_destroy(self._handle)
            self._handle = None


def _i32(t, device):
    return None if t is None else t.to(device=device, dtype=torch.int32).contiguous()


def _f32(t, device):
    return None if t is None else t.to(device=device, dtype=torch.float32).contiguous()


def trans_forward(trunk: EpicModel, heads: TransHeads, x, onehot, dims, ts, nearest_in, u_nearest, forward_rate: ForwardRate,
                  precision="bf16", want_auto=True):
    """One TransdimensionalEPiC evaluation on device tensors -> namespace(d_xt, rate, auto_mean, auto_std, x0_dim_logits,
    near_atom_logits, nearest)."""
    from types import SimpleNamespace
    dev = x.device
    x, onehot = _f32(x, dev), _f32(onehot, dev)
    _require_cuda(x, onehot)
    B, N, _ = x.shape
    S, R = heads.dims.vocab_size, heads.dims.max_particles
    F = 3 + S
    dims, ts, nearest_in, u_nearest = _i32(dims, dev), _f32(ts, dev), _i32(nearest_in, dev), _f32(u_nearest, dev)
    new = lambda *shape, dtype=torch.float32: torch.empty(*shape, device=dev, dtype=dtype)
    out = SimpleNamespace(d_xt=new(B, N * F), rate=new(B), auto_mean=new(B, N * F) if want_auto else None,
                          auto_std=new(B, N * F) if want_auto else None, x0_dim_logits=new(B, R), near_atom_logits=new(B, N),
                          nearest=new(B, dtype=torch.int32))
    lib = load()
    need = lib.mmb_trans_forward_workspace_bytes(trunk._handle, heads._handle, B, N)
    ws = torch.empty(max(need, 16), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        check(lib.mmb_trans_forward(trunk._handle, heads._handle, _ptr(x), _ptr(onehot), _ptr(dims), _ptr(ts), _ptr(nearest_in),
                                    _ptr(u_nearest), ctypes.byref(forward_rate), B, N, _ptr(out.d_xt), _ptr(out.rate),
                                    _ptr(out.auto_mean), _ptr(out.auto_std), _ptr(out.x0_dim_logits), _ptr(out.near_atom_logits),
                                    _ptr(out.nearest), _ptr(ws), ws.numel(), PRECISIONS[precision], _stream()))
    return out


def trans_sample(trunk: EpicModel, heads: TransHeads, x, onehot, dims, sched, forward_rate: ForwardRate, noise=None, seed=0,
                 jet_offset=0, precision="bf16"):
    """In-place JumpSampler loop on x [B,N,3], onehot [B,N,S], dims [B] int32 (device)."""
    _require_cuda(x, onehot, dims)
    assert dims.dtype == torch.int32
    B, N, _ = x.shape
    dev = x.device
    get = lambda name: _f32(getattr(noise, name), dev) if noise is not None and getattr(noise, name, None) is not None else None
    z_diff, u_near, u_jump, z_new, u_death = get("z_diff"), get("u_near"), get("u_jump"), get("z_new"), get("u_death")
    lib = load()
    need = lib.mmb_trans_sample_workspace_bytes(trunk._handle, heads._handle, B, N)
    ws = torch.empty(max(need, 16), device=dev, dtype=torch.uint8)
    csched = JumpSchedule.from_schedule(sched)
    with torch.cuda.device(dev):
        check(lib.mmb_trans_sample(trunk._handle, heads._handle, _ptr(x), _ptr(onehot), _ptr(dims), ctypes.byref(csched),
                                   ctypes.byref(forward_rate), _ptr(z_diff), _ptr(u_near), _ptr(u_jump), _ptr(z_new), _ptr(u_death),
                                   seed, jet_offset, B, N, _ptr(ws), ws.numel(), PRECISIONS[precision], _stream()))
    return x, onehot, dims


def trans_sampler_update(x, onehot, dims, v, logits, rate, new_mean, new_std, c_decay, c_score, c_noise, inv_std, jump_dt,
                         z_diff=None, u_jump=None, z_new=None, seed=0, jet_offset=0, step=0):
    """One fused sampler update in place (the HBM-bound kernel of the loop)."""
    _require_cuda(x, onehot, dims, v, logits, rate, new_mean, new_std, z_diff, u_jump, z_new)
    B, N, _ = x.shape
    S = onehot.shape[-1]
    with torch.cuda.device(x.device):
        check(load().mmb_trans_sampler_update(_ptr(x), _ptr(onehot), _ptr(dims), _ptr(v), _ptr(logits), _ptr(rate), _ptr(new_mean),
                                              _ptr(new_std), c_decay, c_score, c_noise, inv_std, jump_dt, _ptr(z_diff), _ptr(u_jump),
                                              _ptr(z_new), seed, jet_offset, step, B, N, S, _stream()))


def trans_corrector_update(x, onehot, dims, v, logits, rate, new_mean, new_std, alpha, noise_on, inv_std, corrector_snr, jump_dt,
                           jump_corrector=False, death_prob=0.0, mask_dims=None, z_diff=None, u_jump=None, u_death=None, z_new=None,
                           seed=0, jet_offset=0, step=0):
    """One Langevin corrector update in place; returns the step size the batch norms gave (a device scalar)."""
    _require_cuda(x, onehot, dims, v, logits, rate, new_mean, new_std, mask_dims, z_diff, u_jump, u_death, z_new)
    B, N, _ = x.shape
    S = onehot.shape[-1]
    scratch = torch.empty(2 * B + 4, device=x.device, dtype=torch.float32)
    with torch.cuda.device(x.device):
        check(load().mmb_trans_corrector_update(_ptr(x), _ptr(onehot), _ptr(dims), _ptr(mask_dims), _ptr(v), _ptr(logits), _ptr(rate),
                                                _ptr(new_mean), _ptr(new_std), alpha, int(noise_on), inv_std, corrector_snr, jump_dt,
                                                int(jump_corrector), death_prob, _ptr(z_diff), _ptr(u_jump), _ptr(u_death), _ptr(z_new),
                                                seed, jet_offset, step, B, N, S, _ptr(scratch), _stream()))
    return scratch[2 * B + 3]


# ---- forward half of a training / validation step ---------------------------------------------------------
def sample_bridges(x0, x1, k0_u8, k1_u8, t, sigma, gamma, S, z=None, u=None, seed=0, jet_offset=0):
    """-> (xt [B,N,3] f32, kt [B,N] u8) on the device of x0."""
    _require_cuda(x0, x1, k0_u8, k1_u8, t, z, u)
    B, N, _ = x0.shape
    xt = torch.empty_like(x0)
    kt = torch.empty(B, N, dtype=torch.uint8, device=x0.device)
    with torch.cuda.device(x0.device):
        check(load().mmb_sample_bridges(_ptr(x0), _ptr(x1), _ptr(k0_u8), _ptr(k1_u8), _ptr(t), float(sigma), float(gamma), S, _ptr(z), _ptr(u),
                                        seed, jet_offset, B, N, _ptr(xt), _ptr(kt), _stream()))
    return xt, kt


def absorbing_sample(sp, target_mask_u8, u=None, seed=0, jet_offset=0):
    _require_cuda(sp, target_mask_u8, u)
    B, N = target_mask_u8.shape
    out = torch.empty_like(target_mask_u8)
    with torch.cuda.device(sp.device):
        check(load().mmb_absorbing_sample(_ptr(sp), _ptr(target_mask_u8), _ptr(u), seed, jet_offset, B, N, _ptr(out), _stream()))
    return out


def bridge_losses(v, logits, x0, x1, k1_u8, mask_u8):
    """-> device tensor [3] = (masked MSE, masked cross entropy, live particles)."""
    _require_cuda(v, logits, x0, x1, k1_u8, mask_u8)
    B, N, S = logits.shape
    lib = load()
    out = torch.empty(3, device=v.device, dtype=torch.float32)
    ws = torch.empty(max(lib.mmb_bridge_losses_workspace_bytes(B, N), 16), device=v.device, dtype=torch.uint8)
    with torch.cuda.device(v.device):
        check(lib.mmb_bridge_losses(_ptr(v), _ptr(logits), _ptr(x0), _ptr(x1), _ptr(k1_u8), _ptr(mask_u8), B, N, S, _ptr(out), _ptr(ws),
                                    ws.numel(), _stream()))
    return out


def epic_loss_grad(dims: EpicDims, W, x, k_u8, mask_u8, rows, x0, x1, k1_u8, jacobian=True):
    """Bridge-matching losses of the fp32 network with weights ``W`` (device blob in ``mmb_epic_layout`` order) and, with
    ``jacobian``, their gradients: -> (losses [3] = (mse, ce, live), jac [2, total] or None, d_context [2, B, X] or None)."""
    _require_cuda(W, x, k_u8, mask_u8, rows, x0, x1, k1_u8)
    B, N, _ = x.shape
    lib = load()
    total = lib.mmb_epic_packed_floats(ctypes.byref(dims))
    if W.dtype != torch.float32 or W.numel() != total:
        raise MmbError(f"weight blob must hold {total} float32 values, got {W.numel()} {W.dtype}")
    width = dims.dim_time_emb + dims.dim_context
    if rows.shape[-1] != width:
        raise MmbError(f"context rows must hold {dims.dim_time_emb} time + {dims.dim_context} context entries, got {rows.shape[-1]}")
    stride = 0 if rows.shape[0] == 1 and B != 1 else width
    dev = x.device
    losses = torch.empty(3, device=dev, dtype=torch.float32)
    jac = torch.empty(2, total, device=dev, dtype=torch.float32) if jacobian else None
    d_context = torch.empty(2, B, dims.dim_context, device=dev, dtype=torch.float32) if jacobian and dims.dim_context else None
    need = lib.mmb_epic_loss_grad_workspace_bytes(ctypes.byref(dims), B, N)
    ws = torch.empty(max(need, 16), device=dev, dtype=torch.uint8)
    with torch.cuda.device(dev):
        check(lib.mmb_epic_loss_grad(ctypes.byref(dims), _ptr(W), _ptr(x), _ptr(k_u8), _ptr(mask_u8), _ptr(rows), stride, _ptr(x0), _ptr(x1),
                                     _ptr(k1_u8), B, N, _ptr(losses), _ptr(jac), _ptr(d_context), _ptr(ws), ws.numel(), _stream()))
    return losses, jac, d_context
