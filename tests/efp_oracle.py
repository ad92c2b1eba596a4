"""numpy fp64 statements of the energy flow polynomials of mmb_energy_flow_polynomials (closed forms and a brute-force sum over
every index tuple) and of the per-draw Frechet distance and unbiased MMD^2 behind FPD and KPD (DESIGN.md §4.6d)."""
import numpy as np

COLUMNS = ("efp1", "efp4_square", "efp4_paw", "efp4_path_mid2", "efp4_path_end2", "efp4_star2")
# edge lists of the graphs of COLUMNS (vertices 0..V-1); the d = 4 ones are every connected multigraph with 4 vertices, 4 edges
GRAPHS = (((0, 1),),
          ((0, 1), (1, 2), (2, 3), (3, 0)),      # 4-cycle
          ((0, 1), (1, 2), (2, 0), (0, 3)),      # triangle plus pendant
          ((0, 1), (1, 2), (1, 2), (2, 3)),      # 3-edge path, middle edge doubled
          ((0, 1), (0, 1), (1, 2), (2, 3)),      # 3-edge path, end edge doubled
          ((0, 1), (0, 1), (0, 2), (0, 3)))      # 3-star, one edge doubled


def theta(eta, phi, beta=1.0):
    deta = eta[:, None] - eta[None]
    dphi = phi[:, None] - phi[None]
    dphi = np.where(dphi > np.pi, dphi - 2 * np.pi, np.where(dphi < -np.pi, dphi + 2 * np.pi, dphi))
    return np.sqrt(deta * deta + dphi * dphi) ** beta


def closed_forms(pt, eta, phi, beta=1.0):
    """One jet's used particles (fp64) -> [6] in the order of COLUMNS; NaN for an empty jet."""
    if len(pt) == 0:
        return np.full(6, np.nan)
    z = pt / pt.sum()
    T = theta(eta, phi, beta)
    s, q = T @ z, (T * T) @ z
    M = T @ (z[:, None] * T)
    return np.array([z @ s,
                     z @ (M * M) @ z,
                     np.sum(z * s * ((T * M) @ z)),
                     (z * s) @ (T * T) @ (z * s),
                     (z * q) @ T @ (z * s),
                     np.sum(z * q * s * s)])


def brute_force(pt, eta, phi, beta=1.0):
    """Every EFP of COLUMNS as the literal sum over all index tuples (coincident indices included); small n only."""
    z = pt / pt.sum()
    T = theta(eta, phi, beta)
    letters = "abcd"
    out = []
    for edges in GRAPHS:
        V = 1 + max(max(e) for e in edges)
        spec = ",".join(letters[:V]) + "," + ",".join(letters[a] + letters[b] for a, b in edges) + "->"
        out.append(np.einsum(spec, *([z] * V), *([T] * len(edges))))
    return np.array(out)


def used_particles(x, mask, stats=None):
    """Per jet, (pt, eta, phi) fp64 of the used particles (mask and pt > 0), de-standardised like the kernel, in fp32."""
    x = np.asarray(x, np.float32)
    if stats is not None:
        x = x * np.asarray(stats["std"][:3], np.float32) + np.asarray(stats["mean"][:3], np.float32)
    jets = []
    for b in range(x.shape[0]):
        c = x[b, (np.asarray(mask[b]) != 0) & (x[b, :, 0] > 0)].astype(np.float64)
        jets.append((c[:, 0], c[:, 1], c[:, 2]))
    return jets


def numpy_batch(x, mask, stats=None, beta=1.0):
    return np.array([closed_forms(*j, beta) for j in used_particles(x, mask, stats)])


# ---- FPD / KPD -----------------------------------------------------------------------------------------------------------------
def frechet_distance(mu1, s1, mu2, s2):
    """||mu1 - mu2||^2 + Tr S1 + Tr S2 - 2 sum sqrt(max(l, 0)), l the eigenvalues of S1^1/2 S2 S1^1/2."""
    w, v = np.linalg.eigh(s1)
    root = (v * np.sqrt(np.clip(w, 0, None))) @ v.T
    lam = np.linalg.eigvalsh(root @ s2 @ root)
    d = mu1 - mu2
    return float(d @ d + np.trace(s1) + np.trace(s2) - 2 * np.sqrt(np.clip(lam, 0, None)).sum())


def gaussian(rows):
    return rows.mean(0), np.atleast_2d(np.cov(rows, rowvar=False, ddof=1))


def draw_rows(x, idx, scale=None):
    """x[idx] in fp64, times scale (f32 -> fp64, as the kernels take it)."""
    r = np.asarray(x, np.float32)[idx].astype(np.float64)
    return r if scale is None else r * np.asarray(scale, np.float32).astype(np.float64)


def mmd_unbiased(X, Y, degree=4):
    """(sum_{i != j} k(x_i, x_j) + sum_{i != j} k(y_i, y_j)) / (B (B - 1)) - 2 sum_{i,j} k(x_i, y_j) / B^2, k = (x.y / d + 1)^degree."""
    B, d = X.shape
    kxx, kyy, kxy = [(a @ b.T / d + 1.0) ** degree for a, b in ((X, X), (Y, Y), (X, Y))]
    return float((kxx.sum() - np.trace(kxx) + kyy.sum() - np.trace(kyy)) / (B * (B - 1)) - 2 * kxy.sum() / (B * B))
