"""Post-processing and jet-level observables of generated jets — drop-in for the generation-side use of
``ParticleClouds`` (mp/data/particle_clouds/particles.py:22-156: construction from a ``HybridState``, ``postprocess``,
``compute_4mom``) and ``JetClassHighLevelFeatures`` (mp/data/particle_clouds/jets.py:85-141, 329-332: jet kinematics,
multiplicity, jet charges, 1-D Wasserstein distance), SURVEY.md §8f N1.  One fused kernel (``mmb_jet_observables``) does the
de-standardisation, ``tokens_to_physics``, the 4-momenta and the per-jet sums.  The clustering-based substructure (fastjet
N-subjettiness on exclusive kt / WTA axes and D2, jets.py:204-240) is a second kernel (``mmb_jet_substructure``,
``jet_substructure``); ``JetClassHighLevelFeatures.compute_substructure`` sets its columns.  The 1-D Wasserstein distance the
reference scores with (scipy.stats.wasserstein_distance, jets.py:329-332) is a third (``mmb_wasserstein1d``, ``wasserstein1d``,
``JetClassHighLevelFeatures.wasserstein1d``).  The energy flow polynomials of the JetNet metrics (arXiv:2211.10295) are a fourth
(``mmb_energy_flow_polynomials``, ``energy_flow_polynomials``, ``JetClassHighLevelFeatures.compute_efps``); ``fpd`` and ``kpd``
score them with the sample statistics of ``mmb_sampled_moments`` and ``mmb_kpd_mmd``; every EFP of degree <= 4, the feature set
JetNet scores FPD and KPD on, is a second instantiation of that kernel (``mmb_energy_flow_polynomials_d4``,
``energy_flow_polynomials_d4``, ``jetnet_fpd_features``).  JetNet's W1-M, W1-P and W1-EFP (``w1m``,
``w1p``, ``w1efp``) score seeded draws of jets with ``mmb_wasserstein1d_drawn`` (``wasserstein1d_drawn``).
"""
import ctypes

import numpy as np
import torch

from . import _native
from .epic import as_u8

JET_COLUMNS = ("px", "py", "pz", "e", "pt", "m", "eta", "phi", "multiplicity", "Q_total", "Q_jet")


def _stats_arrays(stats):
    """{"mean": [...], "std": [...]} (the first three entries: pt, eta, phi) -> (mean, std) as ctypes float[3], or (None, None)."""
    if stats is None:
        return None, None
    return tuple((ctypes.c_float * 3)(*[float(v) for v in stats[key][:3]]) for key in ("mean", "std"))


def _cuda_device(t):
    """The device of ``t`` when it is a CUDA device, else the current CUDA device."""
    if t.is_cuda:
        return t.device
    if not torch.cuda.is_available():
        raise _native.MmbError("libmmbridge has no CPU path: post-processing and the jet features need a CUDA device")
    return torch.device("cuda", torch.cuda.current_device())


def _rows(t, name):
    """[n, K] f32 CUDA tensor -> ([n, K] view with unit column stride, row stride)."""
    if t.dim() != 2 or t.dtype != torch.float32 or not t.is_cuda:
        raise _native.MmbError(f"{name} takes [n, K] float32 CUDA tensors; there is no CPU path")
    if t.stride(1) != 1 or (t.shape[0] > 1 and t.stride(0) < t.shape[1]):
        t = t.contiguous()
    return t, t.stride(0) if t.shape[0] > 1 else t.shape[1]


def jet_observables(x, k_u8, mask_u8, stats=None, want_particles=True):
    """x [B,N,3] f32, k/mask [B,N] u8 on the GPU -> (x_phys [B,N,3] | None, flavor_charge [B,N,2] int8 | None, jets [B,11])."""
    _native._require_cuda(x, k_u8, mask_u8)
    B, N, _ = x.shape
    dev = x.device
    x_phys = torch.empty_like(x) if want_particles else None
    fc = torch.empty(B, N, 2, dtype=torch.int8, device=dev) if want_particles else None
    jets = torch.empty(B, len(JET_COLUMNS), dtype=torch.float32, device=dev)
    mean, std = _stats_arrays(stats)
    with torch.cuda.device(dev):
        _native.check(_native.load().mmb_jet_observables(_native._ptr(x), _native._ptr(k_u8), _native._ptr(mask_u8), mean, std, B, N,
                                                         _native._ptr(x_phys), _native._ptr(fc), _native._ptr(jets), _native._stream()))
    return x_phys, fc, jets


SUBSTRUCTURE_COLUMNS = ("tau1", "tau2", "tau3", "tau21", "tau32", "e2", "e3", "d2")


def jet_substructure(x, mask_u8, stats=None, R=0.8, beta=1.0, want_axes=False):
    """x [B,N,3] f32 (pt, eta, phi; standardised when ``stats`` is given), mask [B,N] u8 on the GPU, N <= 256
    -> [B,8] f32 in the order of ``SUBSTRUCTURE_COLUMNS`` (, axes [B,6] int16: the particle slot of the tau1 axis, the two tau2
    axes and the three tau3 axes).  Jets with fewer than 3 used particles (mask and pt > 0) are NaN, axes -1.  R: radius of
    the exclusive kt clustering; beta: angular exponent of tau_N and of the energy correlation functions."""
    _native._require_cuda(x, mask_u8)
    B, N, _ = x.shape
    dev = x.device
    out = torch.empty(B, len(SUBSTRUCTURE_COLUMNS), dtype=torch.float32, device=dev)
    axes = torch.empty(B, 6, dtype=torch.int16, device=dev) if want_axes else None
    mean, std = _stats_arrays(stats)
    with torch.cuda.device(dev):
        _native.check(_native.load().mmb_jet_substructure(_native._ptr(x), _native._ptr(mask_u8), mean, std, B, N, float(R), float(beta),
                                                          _native._ptr(out), _native._ptr(axes), _native._stream()))
    return (out, axes) if want_axes else out


def wasserstein1d(x, y, return_counts=False):
    """x [n] or [n, K], y [m] or [m, K] f32 on the GPU -> W1 per column [K] f64 on the device (0-d for 1-D inputs): the
    scipy.stats.wasserstein_distance of the finite values of each column, NaN when a sample has none (DESIGN.md §4.6c).
    ``return_counts``: also the numbers of finite x and y values, [2, K] int64 ([2] for 1-D inputs)."""
    one = x.dim() == 1
    x2, ldx = _rows(x.reshape(-1, 1) if one else x, "wasserstein1d")
    y2, ldy = _rows(y.reshape(-1, 1) if y.dim() == 1 else y, "wasserstein1d")
    if x2.device != y2.device or x2.shape[1] != y2.shape[1]:
        raise _native.MmbError(f"wasserstein1d: x {tuple(x.shape)} on {x.device} and y {tuple(y.shape)} on {y.device} do not match")
    (n, K), m = x2.shape, y2.shape[0]
    dev = x2.device
    lib = _native.load()
    with torch.cuda.device(dev):
        need = lib.mmb_wasserstein1d_workspace_bytes(n, m, K)
        ws = torch.empty(max(need, 256), dtype=torch.uint8, device=dev)
        out = torch.empty(K, dtype=torch.float64, device=dev)
        used = torch.empty(2, K, dtype=torch.int64, device=dev)
        _native.check(lib.mmb_wasserstein1d(_native._ptr(x2) if n else None, ldx, n, _native._ptr(y2) if m else None, ldy, m, K,
                                            _native._ptr(out), _native._ptr(used), _native._ptr(ws), ws.numel(), _native._stream()))
    if one:
        out, used = out[0], used[:, 0]
    return (out, used) if return_counts else out


def _jets(t, mask, name):
    """[n, P, F] or [n, F] f32 CUDA tensor (+ [n, P] mask) -> (tensor, ld_jet, ld_slot, P, mask u8 or None, ldm)."""
    if t.dtype != torch.float32 or not t.is_cuda or t.dim() not in (2, 3):
        raise _native.MmbError(f"wasserstein1d_drawn: {name} must be a [n, P, F] or [n, F] float32 CUDA tensor; there is no CPU path")
    if t.stride(-1) != 1:
        t = t.contiguous()
    P = t.shape[1] if t.dim() == 3 else 1
    ld_jet, ld_slot = t.stride(0), (t.stride(1) if t.dim() == 3 else t.shape[1])
    if t.shape[0] == 1:
        ld_jet = max(ld_jet, P * t.shape[-1])
    if mask is not None:
        if not mask.is_cuda or mask.numel() != t.shape[0] * P:
            raise _native.MmbError(f"wasserstein1d_drawn: mask of {name} must be a [{t.shape[0]}, {P}] CUDA tensor")
        mask = as_u8(mask).contiguous()
    return t, ld_jet, ld_slot, P, mask, P


def wasserstein1d_drawn(x, idx_x, y, idx_y, mask_x=None, mask_y=None, return_counts=False):
    """Per draw t and feature c: the W1 (``wasserstein1d``) between the used slots of the jets x[idx_x[t]] and those of
    y[idx_y[t]], each taken in draw order and slot order (a jet drawn k times counts k times), without gathering them.
    x [n, P, F] or [n, F] (P = 1), y likewise, f32 on the GPU; masks [n, P] (None: every slot used); indices [draws, rows]
    -> [draws, F] f64 on the device, bit-identical to ``wasserstein1d`` on the gathered samples (DESIGN.md §4.6e).
    ``return_counts``: also the finite counts [2, draws, F] int64."""
    x, ldxj, ldxs, P, mx, ldmx = _jets(x, mask_x, "x")
    y, ldyj, ldys, Py, my, ldmy = _jets(y, mask_y, "y")
    if x.device != y.device or P != Py or x.shape[-1] != y.shape[-1] or idx_x.dim() != 2 or idx_x.shape != idx_y.shape:
        raise _native.MmbError(f"wasserstein1d_drawn: x {tuple(x.shape)}, y {tuple(y.shape)}, indices {tuple(idx_x.shape)} / "
                               f"{tuple(idx_y.shape)} do not match")
    if not idx_x.is_cuda or not idx_y.is_cuda:
        raise _native.MmbError("wasserstein1d_drawn: indices must be CUDA tensors; there is no CPU path")
    F = x.shape[-1]
    draws, rows = idx_x.shape
    ix, iy = _index(idx_x), _index(idx_y)
    dev = x.device
    lib = _native.load()
    with torch.cuda.device(dev):
        need = lib.mmb_wasserstein1d_drawn_workspace_bytes(draws, rows, P, F)
        ws = torch.empty(max(need, 256), dtype=torch.uint8, device=dev)
        out = torch.empty(draws, F, dtype=torch.float64, device=dev)
        used = torch.empty(2, draws, F, dtype=torch.int64, device=dev)
        _native.check(lib.mmb_wasserstein1d_drawn(_native._ptr(x), ldxj, ldxs, _native._ptr(mx), ldmx, x.shape[0],
                                                  _native._ptr(y), ldyj, ldys, _native._ptr(my), ldmy, y.shape[0], P, F,
                                                  _native._ptr(ix), _native._ptr(iy), draws, rows, _native._ptr(out), _native._ptr(used),
                                                  _native._ptr(ws), ws.numel(), _native._stream()))
    return (out, used) if return_counts else out


# energy flow polynomials (DESIGN.md §4.6d): the d = 1 EFP, then the five connected multigraphs with 4 vertices and 4 edges, the
# set JetNet's efps / w1efp use by default (("n==", 4), ("d==", 4), ("p==", 1)); W1-EFP, FPD and KPD score EFP_COLUMNS[1:]
EFP_COLUMNS = ("efp1", "efp4_square", "efp4_paw", "efp4_path_mid2", "efp4_path_end2", "efp4_star2")
# conventions of the JetNet metrics (arXiv:2211.10295), each in one place
EFP_BETA = 1.0                               # theta = dR^beta, hadronic measure, kappa = 1, normalised energies
KPD_DEGREE = 4                               # k(x, y) = (x . y / d + 1)^degree: gamma = 1 / d, c = 1
KPD_ERROR_RANGE = (16.275, 83.725)           # KPD error: half of this percentile range of the per-batch values


def energy_flow_polynomials(x, mask_u8, stats=None, beta=EFP_BETA):
    """x [B,N,3] f32 (pt, eta, phi; standardised when ``stats`` is given), mask [B,N] u8 on the GPU, N <= 256 -> [B,6] f32 in the
    order of ``EFP_COLUMNS``.  Jets with no used particle (mask and pt > 0) are NaN; jets with one are 0."""
    return _efp_call("mmb_energy_flow_polynomials", len(EFP_COLUMNS), x, mask_u8, stats, beta)


def _efp_call(name, columns, x, mask_u8, stats, beta):
    _native._require_cuda(x, mask_u8)
    B, N, _ = x.shape
    dev = x.device
    out = torch.empty(B, columns, dtype=torch.float32, device=dev)
    mean, std = _stats_arrays(stats)
    with torch.cuda.device(dev):
        _native.check(getattr(_native.load(), name)(_native._ptr(x), _native._ptr(mask_u8), mean, std, B, N, float(beta),
                                                    _native._ptr(out), _native._stream()))
    return out


# every EFP of degree d <= 4 (DESIGN.md §4.6f), the kernel's column order: by d, connected graphs before disconnected ones.  A
# disconnected graph is named by its components (its EFP is their product); "^k" is k copies of one component.  energyflow
# orders its graphs differently; FD and the polynomial-kernel MMD do not depend on the order of the features, and fpd / kpd
# normalise each column on its own, so the order does not change FPD or KPD.
EFP_D4_COLUMNS = ("efp0",
                  "efp1",
                  "efp2_double", "efp2_path", "efp1^2",
                  "efp3_triple", "efp3_path_double", "efp3_triangle", "efp3_path", "efp3_star",
                  "efp1*efp2_double", "efp1*efp2_path", "efp1^3",
                  "efp4_quadruple", "efp4_triple_single", "efp4_double_double", "efp4_triangle_double", "efp4_square", "efp4_paw",
                  "efp4_path_mid2", "efp4_path_end2", "efp4_star2", "efp4_path", "efp4_star", "efp4_fork",
                  "efp1*efp3_triple", "efp1*efp3_path_double", "efp1*efp3_triangle", "efp1*efp3_path", "efp1*efp3_star",
                  "efp2_double^2", "efp2_double*efp2_path", "efp2_path^2", "efp1^2*efp2_double", "efp1^2*efp2_path", "efp1^4")
# the features FPD / KPD score, as remembered of JetNet's get_fpd_kpd_jet_features (efps(jets, efpset_args=[("d<=", 4)]), "36
# EFPs"): every column, the empty graph and the disconnected graphs included.  The one place to change if the set turns out
# to be the prime (connected) graphs or to exclude efp0.
FPD_EFP_COLUMNS = EFP_D4_COLUMNS


def energy_flow_polynomials_d4(x, mask_u8, stats=None, beta=EFP_BETA):
    """Every EFP of degree <= 4 (``mmb_energy_flow_polynomials_d4``): x [B,N,3] f32 (pt, eta, phi; standardised when ``stats``
    is given), mask [B,N] u8 on the GPU, N <= 256 -> [B,36] f32 in the order of ``EFP_D4_COLUMNS``.  Jets with no used particle
    (mask and pt > 0) are NaN in every column; jets with one are 1 in efp0 and 0 elsewhere.  efp1 and the five efp4_* columns of
    ``EFP_COLUMNS`` are bit-identical to ``energy_flow_polynomials``'."""
    return _efp_call("mmb_energy_flow_polynomials_d4", len(EFP_D4_COLUMNS), x, mask_u8, stats, beta)


_FPD_PICK = [EFP_D4_COLUMNS.index(c) for c in FPD_EFP_COLUMNS]


def jetnet_fpd_features(x, mask_u8, stats=None):
    """The features ``fpd`` / ``kpd`` score as JetNet does (``FPD_EFP_COLUMNS`` of ``energy_flow_polynomials_d4`` at EFP_BETA):
    [B, len(FPD_EFP_COLUMNS)] f32 on the device."""
    out = energy_flow_polynomials_d4(x, mask_u8, stats)
    if _FPD_PICK == list(range(len(EFP_D4_COLUMNS))):
        return out
    return out[:, _FPD_PICK].contiguous()


def _index(idx):
    return idx.to(torch.int32).contiguous()


def sampled_moments(x, idx, scale=None):
    """x [n, d] f32, idx [draws, rows] (row indices) on the GPU -> (sum [draws, d], sum of x x^T [draws, d, d]) in f64 on the
    device, every value taken as x * scale (``scale`` [d] f32, None for 1; the product is exact in fp64)."""
    x2, ldx = _rows(x, "sampled_moments")
    (n, d), (draws, rows) = x2.shape, idx.shape
    idx = _index(idx)
    sums = torch.empty(draws, d, dtype=torch.float64, device=x2.device)
    sumsq = torch.empty(draws, d, d, dtype=torch.float64, device=x2.device)
    with torch.cuda.device(x2.device):
        _native.check(_native.load().mmb_sampled_moments(_native._ptr(x2), ldx, n, d, _native._ptr(scale), _native._ptr(idx), draws, rows,
                                                         _native._ptr(sums), _native._ptr(sumsq), _native._stream()))
    return sums, sumsq


def _mean_cov(sums, sumsq, rows):
    mu = sums / rows
    return mu, (sumsq - rows * mu[:, :, None] * mu[:, None, :]) / (rows - 1)


def frechet_distances(real, gen, idx_real, idx_gen, scale=None):
    """Per draw t: the Frechet distance between Gaussians fitted (mean, unbiased covariance) to real[idx_real[t]] and
    gen[idx_gen[t]], ||mu1 - mu2||^2 + Tr S1 + Tr S2 - 2 sum_i sqrt(max(l_i, 0)) with l the eigenvalues of S1^1/2 S2 S1^1/2
    (batched fp64 eigh on the device) -> [draws] f64 on the device."""
    m1, c1 = _mean_cov(*sampled_moments(real, idx_real, scale), idx_real.shape[1])
    m2, c2 = _mean_cov(*sampled_moments(gen, idx_gen, scale), idx_gen.shape[1])
    return _frechet(m1, c1, m2, c2)


def _frechet(m1, c1, m2, c2):
    w, v = torch.linalg.eigh(c1)
    root = (v * w.clamp(min=0).sqrt()[:, None, :]) @ v.transpose(1, 2)
    lam = torch.linalg.eigvalsh(root @ c2 @ root)
    diff = m1 - m2
    return (diff * diff).sum(1) + c1.diagonal(dim1=1, dim2=2).sum(1) + c2.diagonal(dim1=1, dim2=2).sum(1) - 2 * lam.clamp(min=0).sqrt().sum(1)


def kpd_mmd(real, gen, idx_real, idx_gen, scale=None, degree=KPD_DEGREE):
    """Per batch t: the unbiased MMD^2 between real[idx_real[t]] and gen[idx_gen[t]] (B rows each) with the polynomial kernel
    k(x, y) = (x . y / d + 1)^degree, in fp64 -> [batches] f64 on the device."""
    r2, ldr = _rows(real, "kpd_mmd")
    g2, ldg = _rows(gen, "kpd_mmd")
    if r2.shape[1] != g2.shape[1] or r2.device != g2.device or idx_real.shape != idx_gen.shape:
        raise _native.MmbError(f"kpd_mmd: real {tuple(real.shape)}, gen {tuple(gen.shape)}, indices {tuple(idx_real.shape)} / "
                               f"{tuple(idx_gen.shape)} do not match")
    (n, d), m = r2.shape, g2.shape[0]
    batches, B = idx_real.shape
    lib = _native.load()
    ir, ig = _index(idx_real), _index(idx_gen)
    with torch.cuda.device(r2.device):
        need = lib.mmb_kpd_mmd_workspace_bytes(batches, B, d)
        ws = torch.empty(max(need, 256), dtype=torch.uint8, device=r2.device)
        out = torch.empty(batches, dtype=torch.float64, device=r2.device)
        _native.check(lib.mmb_kpd_mmd(_native._ptr(r2), ldr, n, _native._ptr(g2), ldg, m, d, _native._ptr(scale), _native._ptr(ir),
                                      _native._ptr(ig), batches, B, int(degree), _native._ptr(out), _native._ptr(ws), ws.numel(),
                                      _native._stream()))
    return out


def _finite_rows_and_scale(real, gen, normalise):
    """Drops the rows with a non-finite value (one host synchronisation each) and returns the per-column scale 1 / max|real|
    (None without ``normalise``; 1 where a column of real is all zero)."""
    real, gen = [t[torch.isfinite(t).all(1)].to(torch.float32).contiguous() for t in (real, gen)]
    if len(real) == 0 or len(gen) == 0:
        raise ValueError("fpd / kpd: a sample has no row without a non-finite value")
    scale = None
    if normalise:
        top = real.abs().amax(0)
        scale = torch.where(top > 0, 1.0 / top, torch.ones_like(top)).contiguous()
    return real, gen, scale


def _generator(device, seed):
    return torch.Generator(device=device).manual_seed(seed)


def fpd(real, gen, min_samples=20_000, max_samples=50_000, num_batches=20, num_points=10, normalise=True, seed=42):
    """Frechet physics distance (arXiv:2211.10295, JetNet's ``fpd``) of two [n, d] f32 CUDA feature samples -> (value, error).
    For each of ``num_points`` sample sizes N = int(1 / linspace(1 / min_samples, 1 / max_samples)), ``num_batches`` draws with
    replacement of N rows of each sample (seeded device generator); the Frechet distances are averaged per size and
    ``a + b / N`` (a, b >= 0) is fitted; the value is ``a`` and the error the fit's standard error of ``a``.  The host waits only
    to drop non-finite rows and for the 10 averages (the eigendecompositions of all draws run in one batch)."""
    from scipy.optimize import curve_fit
    real, gen, scale = _finite_rows_and_scale(real, gen, normalise)
    sizes = (1 / np.linspace(1.0 / min_samples, 1.0 / max_samples, num_points)).astype("int32")
    g = _generator(real.device, seed)
    mom = []
    for N in sizes:
        N = int(N)
        ir = torch.randint(len(real), (num_batches, N), generator=g, device=real.device, dtype=torch.int32)
        ig = torch.randint(len(gen), (num_batches, N), generator=g, device=real.device, dtype=torch.int32)
        mom.append(_mean_cov(*sampled_moments(real, ir, scale), N) + _mean_cov(*sampled_moments(gen, ig, scale), N))
    m1, c1, m2, c2 = [torch.cat([p[i] for p in mom]) for i in range(4)]
    vals = _frechet(m1, c1, m2, c2).reshape(num_points, num_batches).mean(1).cpu().numpy()
    params, covs = curve_fit(lambda x, a, b: a + b * x, 1 / sizes, vals, bounds=([0, 0], [np.inf, np.inf]))
    return float(params[0]), float(np.sqrt(np.diag(covs)[0]))


def kpd(real, gen, num_batches=10, batch_size=5000, degree=KPD_DEGREE, normalise=True, seed=42):
    """Kernel physics distance (arXiv:2211.10295, JetNet's ``kpd``) of two [n, d] f32 CUDA feature samples -> (median, error):
    the unbiased MMD^2 with the polynomial kernel over ``num_batches`` draws with replacement of ``batch_size`` rows of each
    sample (seeded device generator), its median and half of its KPD_ERROR_RANGE percentile range."""
    real, gen, scale = _finite_rows_and_scale(real, gen, normalise)
    g = _generator(real.device, seed)
    ir = torch.randint(len(real), (num_batches, batch_size), generator=g, device=real.device, dtype=torch.int32)
    ig = torch.randint(len(gen), (num_batches, batch_size), generator=g, device=real.device, dtype=torch.int32)
    vals = kpd_mmd(real, gen, ir, ig, scale, degree).cpu().numpy()
    lo, hi = np.percentile(vals, KPD_ERROR_RANGE)
    return float(np.median(vals)), float((hi - lo) / 2)


# JetNet's W1-M, W1-P and W1-EFP (arXiv:2211.10295): each W1 is the mean +- std over W1_NUM_BATCHES draws of
# W1_NUM_EVAL_SAMPLES jets from each sample.  Conventions as remembered, not checked against JetNet (DESIGN.md §4.6e):
W1_NUM_EVAL_SAMPLES = 50_000
W1_NUM_BATCHES = 5
W1_STD_DDOF = 0                              # np.std over the batches
PARTICLE_COLUMNS = ("pt", "eta_rel", "phi_rel")   # W1-P features: ParticleClouds.continuous after postprocess (JetNet: pt_rel)


def jetnet_draws(n_real, n_gen, num_eval_samples=W1_NUM_EVAL_SAMPLES, num_batches=W1_NUM_BATCHES, seed=42, device=None):
    """The draws of w1m / w1p / w1efp, with replacement, from one seeded device generator: [num_batches, num_eval_samples]
    int32 indices into the real sample, then into the generated one."""
    g = _generator(device, seed)
    ir = torch.randint(n_real, (num_batches, num_eval_samples), generator=g, device=device, dtype=torch.int32)
    ig = torch.randint(n_gen, (num_batches, num_eval_samples), generator=g, device=device, dtype=torch.int32)
    return ir, ig


def w1_summary(values, average=True):
    """[batches, F] per-draw W1 values (host array) -> (mean, std): with ``average`` the mean over features of the per-feature
    means and sqrt(sum_c std_c^2) (np.linalg.norm), else the per-feature arrays.  A draw where a sample has no used particle
    is NaN (JetNet: inf) and makes its feature's mean and std NaN."""
    values = np.asarray(values, dtype=np.float64)
    means, stds = values.mean(0), values.std(0, ddof=W1_STD_DDOF)
    if average:
        return float(means.mean()), float(np.linalg.norm(stds))
    return means, stds


def _jet_level(t, name):
    if t.dim() not in (1, 2):
        raise _native.MmbError(f"{name} takes [n] or [n, d] float32 CUDA tensors")
    return t.reshape(t.shape[0], -1)


def w1m(real, gen, num_eval_samples=W1_NUM_EVAL_SAMPLES, num_batches=W1_NUM_BATCHES, seed=42):
    """JetNet's W1-M of two [n] f32 CUDA jet-mass samples -> (mean, std) over the draws (``jetnet_draws``); one host wait."""
    real, gen = _jet_level(real, "w1m"), _jet_level(gen, "w1m")
    ir, ig = jetnet_draws(len(real), len(gen), num_eval_samples, num_batches, seed, real.device)
    return w1_summary(wasserstein1d_drawn(real, ir, gen, ig).cpu().numpy())


def w1efp(real, gen, num_eval_samples=W1_NUM_EVAL_SAMPLES, num_batches=W1_NUM_BATCHES, average_over_efps=True, seed=42):
    """JetNet's W1-EFP of two [n, d] f32 CUDA EFP samples -> (mean, std) averaged over the EFPs (``w1_summary``), or per-EFP
    arrays with ``average_over_efps=False``; one host wait."""
    real, gen = _jet_level(real, "w1efp"), _jet_level(gen, "w1efp")
    ir, ig = jetnet_draws(len(real), len(gen), num_eval_samples, num_batches, seed, real.device)
    return w1_summary(wasserstein1d_drawn(real, ir, gen, ig).cpu().numpy(), average_over_efps)


def w1p(real, gen, mask_real=None, mask_gen=None, num_eval_samples=W1_NUM_EVAL_SAMPLES, num_batches=W1_NUM_BATCHES,
        average_over_features=True, seed=42):
    """JetNet's W1-P of two [n, N, F] f32 CUDA samples of post-processed particle features (PARTICLE_COLUMNS), masks [n, N]
    (None: every slot used) -> (mean, std) averaged over the features (``w1_summary``), or per-feature arrays with
    ``average_over_features=False``.  Per draw, the sample is the used particles of the drawn jets; one host wait."""
    ir, ig = jetnet_draws(len(real), len(gen), num_eval_samples, num_batches, seed, real.device)
    vals = wasserstein1d_drawn(real, ir, gen, ig, mask_real, mask_gen)
    return w1_summary(vals.cpu().numpy(), average_over_features)


class ParticleClouds:
    """Generated jets as the reference's container: ``ParticleClouds(dataset=HybridState)`` (particles.py:33-38)."""

    def __init__(self, dataset, data_paths=None, **data_params):
        if not hasattr(dataset, "continuous"):
            raise NotImplementedError("only construction from a generated HybridState is part of the generation path")
        mask = getattr(dataset, "absorbing", None)
        if mask is None:
            mask = getattr(dataset, "mask_t")
        self.continuous, self.discrete, self.mask = dataset.continuous, dataset.discrete, mask
        self._set_views()
        self.multiplicity = torch.sum(self.mask, dim=1)
        self._jets = None

    def _set_views(self):
        self.pt, self.eta_rel, self.phi_rel = self.continuous[..., 0], self.continuous[..., 1], self.continuous[..., 2]

    def __len__(self):
        return self.continuous.shape[0]

    def _run(self, stats):
        dev = _cuda_device(self.continuous)
        x = self.continuous.to(dev, torch.float32).contiguous()
        return jet_observables(x, as_u8(self.discrete.to(dev)), as_u8(self.mask.to(dev)), stats)

    def postprocess(self, input_continuous="standardize", input_discrete="tokens", stats=None):
        """In place, like the reference: continuous de-standardised and masked; ``flavor`` one-hot [B,N,5], ``charge`` [B,N,1]
        and ``discrete`` = cat(flavor, charge), all masked.  The jet sums computed in the same pass are kept for
        ``JetClassHighLevelFeatures``."""
        if input_discrete != "tokens":
            raise NotImplementedError("native post-processing covers input_discrete='tokens' (every shipped config)")
        stats = getattr(self, "stats", stats)
        out_dev = self.continuous.device
        x_phys, fc, jets = self._run(stats if input_continuous == "standardize" else None)
        live = as_u8(self.mask.to(fc.device)).bool()
        flavor = torch.nn.functional.one_hot(fc[..., 0].long(), num_classes=5) * live[..., None]
        self.continuous = x_phys.to(out_dev)
        self.flavor, self.charge = flavor.to(out_dev), fc[..., 1:2].long().to(out_dev)
        self.discrete = torch.cat([self.flavor, self.charge], dim=-1)
        self._set_views()
        self._jets = jets.to(out_dev)

    def compute_4mom(self):
        self.px = self.pt * torch.cos(self.phi_rel)
        self.py = self.pt * torch.sin(self.phi_rel)
        self.pz = self.pt * torch.sinh(self.eta_rel)
        self.e = self.pt * torch.cosh(self.eta_rel)


class JetClassHighLevelFeatures:
    """Jet kinematics, multiplicity and charges of post-processed constituents (jets.py:85-107, 138-141)."""

    def __init__(self, constituents: ParticleClouds):
        self.constituents = constituents
        jets = constituents._jets
        if jets is None:   # constituents already in physical units (no postprocess call): one pass without de-standardisation
            c = constituents
            dev = _cuda_device(c.continuous)
            tokens = c.discrete if c.discrete.shape[-1] == 1 else None
            if tokens is None:
                raise NotImplementedError("construct from token-valued clouds or call postprocess() first")
            _, _, jets = jet_observables(c.continuous.to(dev, torch.float32).contiguous(), as_u8(tokens.to(dev)), as_u8(c.mask.to(dev)),
                                         None, want_particles=False)
            jets = jets.to(c.continuous.device)
        for i, name in enumerate(JET_COLUMNS):
            setattr(self, name, jets[:, i])
        self.multiplicity = jets[:, JET_COLUMNS.index("multiplicity")].long().unsqueeze(-1)

    def substructure(self):
        raise NotImplementedError("fastjet substructure (jets.py:204-240) stays on the CPU side of the reference")

    def compute_substructure(self, R=0.8, beta=1.0):
        """N-subjettiness and D2 on the device (``jet_substructure``) from the physical constituents: sets ``tau1``, ``tau2``,
        ``tau3``, ``tau21``, ``tau32`` and ``d2`` over the jets with at least 3 used particles (the others are dropped, as
        the reference drops them), so that ``Wassertein1D("tau21", other)`` compares them."""
        c = self.constituents
        dev = _cuda_device(c.continuous)
        out, axes = jet_substructure(c.continuous.to(dev, torch.float32).contiguous(), as_u8(c.mask.to(dev)), None, R, beta,
                                     want_axes=True)
        keep = axes[:, 0] >= 0
        out = out[keep].to(c.continuous.device)
        for name in ("tau1", "tau2", "tau3", "tau21", "tau32", "d2"):
            setattr(self, name, out[:, SUBSTRUCTURE_COLUMNS.index(name)])

    def compute_efps(self, beta=EFP_BETA):
        """Energy flow polynomials on the device (``energy_flow_polynomials``) from the physical constituents: sets the six
        attributes of ``EFP_COLUMNS`` over the jets with at least one used particle, so that
        ``wasserstein1d(reference, EFP_COLUMNS[1:])`` is W1-EFP and ``Wassertein1D("efp4_square", other)`` compares one."""
        c = self.constituents
        dev = _cuda_device(c.continuous)
        out = energy_flow_polynomials(c.continuous.to(dev, torch.float32).contiguous(), as_u8(c.mask.to(dev)), None, beta)
        out = out[~torch.isnan(out[:, 0])].to(c.continuous.device)
        for i, name in enumerate(EFP_COLUMNS):
            setattr(self, name, out[:, i])

    def wasserstein1d(self, reference, features=("pt", "m", "eta", "phi", "multiplicity", "Q_total", "Q_jet")):
        """{feature: W1 between this sample and ``reference``} on the device (``wasserstein1d``), one host synchronisation;
        the same values as ``Wassertein1D(feature, reference)``.  tau1, tau2, tau3, tau21, tau32 and d2 need
        ``compute_substructure`` on both objects; they cover fewer jets, so features are grouped by length (one call each)."""
        dev = _cuda_device(self.pt)
        col = lambda obj, f: getattr(obj, f).reshape(-1).to(dev, torch.float32)
        groups = {}
        for f in features:
            groups.setdefault((getattr(self, f).numel(), getattr(reference, f).numel()), []).append(f)
        names, values = [], []
        for group in groups.values():
            values.append(wasserstein1d(torch.stack([col(self, f) for f in group], 1), torch.stack([col(reference, f) for f in group], 1)))
            names += group
        return dict(zip(names, torch.cat(values).tolist()))

    def Wassertein1D(self, feature, reference):
        import scipy.stats
        x, y = getattr(self, feature), getattr(reference, feature)
        return scipy.stats.wasserstein_distance(np.asarray(x.detach().cpu()).reshape(-1), np.asarray(y.detach().cpu()).reshape(-1))
