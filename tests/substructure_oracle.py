"""ctypes access to oracle_substructure/libmmbo_substructure.so (the CPU restatement of mmb_jet_substructure; test
infrastructure only) and a numpy fp64 brute-force statement of the same definitions."""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle_substructure")
ORACLE_SO = os.path.join(ORACLE_DIR, "libmmbo_substructure.so")
COLUMNS = ("tau1", "tau2", "tau3", "tau21", "tau32", "e2", "e3", "d2")

_lib = None
_fp = ctypes.POINTER(ctypes.c_float)


def lib():
    global _lib
    if _lib is None:
        src_mtime = max(os.path.getmtime(os.path.join(ORACLE_DIR, f)) for f in ("mmbo_substructure.c", "mmbo_substructure.h"))
        if not os.path.exists(ORACLE_SO) or (os.path.getmtime(ORACLE_SO) < src_mtime and os.access(ORACLE_DIR, os.W_OK)):
            subprocess.run(["make", "-C", ORACLE_DIR], check=True, capture_output=True)
        L = ctypes.CDLL(ORACLE_SO)
        L.mmbo_jet_substructure.restype = None
        L.mmbo_jet_substructure.argtypes = [_fp, ctypes.POINTER(ctypes.c_uint8), _fp, _fp, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                            ctypes.c_float, _fp, ctypes.POINTER(ctypes.c_int16)]
        L.mmbo_substructure_threads.restype = ctypes.c_int
        _lib = L
    return _lib


def jet_substructure(x, mask, stats=None, R=0.8, beta=1.0):
    """x [B,N,3], mask [B,N] -> (out [B,8] f32, axes [B,6] int16)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    B, N, _ = x.shape
    mask = np.ascontiguousarray(mask, dtype=np.uint8).reshape(B, N)
    mean = None if stats is None else np.ascontiguousarray(stats["mean"][:3], dtype=np.float32)
    sd = None if stats is None else np.ascontiguousarray(stats["std"][:3], dtype=np.float32)
    out, axes = np.empty((B, 8), np.float32), np.empty((B, 6), np.int16)
    p = lambda a: None if a is None else a.ctypes.data_as(_fp)
    lib().mmbo_jet_substructure(p(x), mask.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), p(mean), p(sd), B, N, R, beta, p(out),
                                axes.ctypes.data_as(ctypes.POINTER(ctypes.c_int16)))
    return out, axes


# ---- numpy restatement: every step scans all candidates at once ------------------------------------------------------
def _dr2(eta_a, phi_a, eta_b, phi_b):
    deta = eta_a - eta_b
    dphi = phi_a - phi_b
    dphi = np.where(dphi > np.pi, dphi - 2 * np.pi, np.where(dphi < -np.pi, dphi + 2 * np.pi, dphi))
    return deta * deta + dphi * dphi


def numpy_jet(pt, eta, phi, slots, R=0.8, beta=1.0, fp32_params=True):
    """One jet's used particles (fp64 arrays in slot order) -> (row [8] f64, axes [6]).  ``fp32_params``: R and beta as the
    C ABI receives them (fp32); False keeps them exact."""
    n = len(pt)
    if n < 3:
        return np.full(8, np.nan), np.full(6, -1)
    if fp32_params:
        R, beta = np.float64(np.float32(R)), np.float64(np.float32(beta))
    inv_r2 = 1.0 / (R * R)
    opt, dirs, alive = pt.copy(), np.arange(n), np.ones(n, bool)
    ax = {}
    left = n
    while True:
        if left <= 3:
            ax[left] = dirs[alive].copy()
        if left == 1:
            break
        idx = np.flatnonzero(alive)
        p2 = opt[idx] * opt[idx]
        lo, hi = np.triu_indices(len(idx), 1)
        a, b = dirs[idx[lo]], dirs[idx[hi]]
        d_pair = np.minimum(p2[lo], p2[hi]) * _dr2(eta[a], phi[a], eta[b], phi[b]) * inv_r2
        d = np.concatenate([p2, d_pair])
        cl = np.concatenate([idx, idx[lo]])
        ch = np.concatenate([idx, idx[hi]])
        pick = np.lexsort((ch, cl, d))[0]
        i, j = cl[pick], ch[pick]
        if i == j:
            alive[i] = False
        else:
            if opt[j] > opt[i]:
                dirs[i] = dirs[j]
            opt[i] = opt[i] + opt[j]
            alive[j] = False
        left -= 1
    apow = (lambda r2: np.sqrt(r2)) if beta == 1.0 else (lambda r2: r2 ** (0.5 * beta))
    tau = []
    for k in (1, 2, 3):
        m = np.min([_dr2(eta, phi, eta[q], phi[q]) for q in ax[k]], axis=0)
        tau.append(np.sum(pt * apow(m)) / (pt.sum() * apow(R * R)))
    z = pt / pt.sum()
    A = apow(_dr2(eta[:, None], phi[:, None], eta[None], phi[None]))
    i, j = np.triu_indices(n, 1)
    e2 = np.sum(z[i] * z[j] * A[i, j])
    # sum over i<j<k = 1/6 of the sum over all (i, j, k): A vanishes on the diagonal, so repeated indices add nothing
    P = z[:, None] * z[None] * A
    e3 = np.sum(P * (A @ (z[:, None] * A))) / 6.0
    with np.errstate(invalid="ignore", divide="ignore"):
        row = np.array([tau[0], tau[1], tau[2], tau[1] / tau[0], tau[2] / tau[1], e2, e3, e3 / e2 ** 3])
    return row, slots[np.concatenate([ax[1], ax[2], ax[3]])]


def numpy_batch(x, mask, stats=None, R=0.8, beta=1.0):
    """The inputs de-standardised like the kernel ((x * std + mean) in fp32), one numpy_jet per jet."""
    x = np.asarray(x, np.float32)
    if stats is not None:
        x = x * np.asarray(stats["std"][:3], np.float32) + np.asarray(stats["mean"][:3], np.float32)
    rows, axes = [], []
    for b in range(x.shape[0]):
        used = (np.asarray(mask[b]) != 0) & (x[b, :, 0] > 0)
        slots = np.flatnonzero(used)
        c = x[b, slots].astype(np.float64)
        r, a = numpy_jet(c[:, 0], c[:, 1], c[:, 2], slots, R, beta)
        rows.append(r)
        axes.append(a)
    return np.array(rows), np.array(axes)
