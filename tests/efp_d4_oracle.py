"""numpy fp64 statements of every energy flow polynomial of degree d <= 4 (mmb_energy_flow_polynomials_d4, DESIGN.md §4.6f): the
closed forms, the literal sum over every index tuple of each graph's edge list, and the edge lists themselves in the kernel's
column order."""
import numpy as np

import efp_oracle as eo

# the 20 connected loopless multigraphs with 1 <= d <= 4 edges (vertices 0..V-1)
CONNECTED = {
    "efp1": ((0, 1),),
    "efp2_double": ((0, 1), (0, 1)),
    "efp2_path": ((0, 1), (1, 2)),
    "efp3_triple": ((0, 1), (0, 1), (0, 1)),
    "efp3_path_double": ((0, 1), (0, 1), (1, 2)),
    "efp3_triangle": ((0, 1), (1, 2), (2, 0)),
    "efp3_path": ((0, 1), (1, 2), (2, 3)),
    "efp3_star": ((0, 1), (0, 2), (0, 3)),
    "efp4_quadruple": ((0, 1), (0, 1), (0, 1), (0, 1)),
    "efp4_triple_single": ((0, 1), (0, 1), (0, 1), (1, 2)),
    "efp4_double_double": ((0, 1), (0, 1), (1, 2), (1, 2)),
    "efp4_triangle_double": ((0, 1), (0, 1), (1, 2), (2, 0)),
    **dict(zip(eo.COLUMNS[1:], eo.GRAPHS[1:])),        # the five 4-vertex, 4-edge graphs of mmb_energy_flow_polynomials
    "efp4_path": ((0, 1), (1, 2), (2, 3), (3, 4)),
    "efp4_star": ((0, 1), (0, 2), (0, 3), (0, 4)),
    "efp4_fork": ((0, 1), (0, 2), (0, 3), (3, 4)),   # 3-star, the leg to 3 extended to 4
}

# the kernel's columns: by d, connected before disconnected; "a*b" is the disjoint union of a and b, "a^k" k copies of a
COLUMNS = ("efp0",
           "efp1",
           "efp2_double", "efp2_path", "efp1^2",
           "efp3_triple", "efp3_path_double", "efp3_triangle", "efp3_path", "efp3_star",
           "efp1*efp2_double", "efp1*efp2_path", "efp1^3",
           "efp4_quadruple", "efp4_triple_single", "efp4_double_double", "efp4_triangle_double", "efp4_square", "efp4_paw",
           "efp4_path_mid2", "efp4_path_end2", "efp4_star2", "efp4_path", "efp4_star", "efp4_fork",
           "efp1*efp3_triple", "efp1*efp3_path_double", "efp1*efp3_triangle", "efp1*efp3_path", "efp1*efp3_star",
           "efp2_double^2", "efp2_double*efp2_path", "efp2_path^2", "efp1^2*efp2_double", "efp1^2*efp2_path", "efp1^4")


def components(name):
    """Column name -> the names of its connected components ([] for efp0)."""
    if name == "efp0":
        return []
    out = []
    for part in name.split("*"):
        base, _, k = part.partition("^")
        out += [base] * int(k or 1)
    return out


def disjoint_union(graphs):
    edges, offset = [], 0
    for g in graphs:
        edges += [(a + offset, b + offset) for a, b in g]
        offset += 1 + max(max(e) for e in g)
    return tuple(edges)


GRAPHS = tuple(disjoint_union([CONNECTED[c] for c in components(name)]) for name in COLUMNS)


def connected_closed_forms(pt, eta, phi, beta=1.0):
    """One jet's used particles (fp64) -> {name: EFP} of the 20 connected graphs, from the row sums s, q, c, r, u and M."""
    z = pt / pt.sum()
    T = eo.theta(eta, phi, beta)
    s, q, c, r = T @ z, (T ** 2) @ z, (T ** 3) @ z, (T ** 4) @ z
    u = T @ (z * s)
    M = T @ (z[:, None] * T)
    old = dict(zip(eo.COLUMNS, eo.closed_forms(pt, eta, phi, beta)))
    return {"efp1": z @ s,
            "efp2_double": z @ q, "efp2_path": z @ (s * s),
            "efp3_triple": z @ c, "efp3_path_double": z @ (q * s), "efp3_triangle": z @ (T * M) @ z, "efp3_path": z @ (s * u),
            "efp3_star": z @ s ** 3,
            "efp4_quadruple": z @ r, "efp4_triple_single": z @ (c * s), "efp4_double_double": z @ q ** 2,
            "efp4_triangle_double": z @ (T * T * M) @ z, **{k: old[k] for k in eo.COLUMNS[1:]},
            "efp4_path": z @ u ** 2, "efp4_star": z @ s ** 4, "efp4_fork": z @ (s * s * u)}


def closed_forms(pt, eta, phi, beta=1.0):
    """One jet's used particles (fp64) -> [36] in the order of COLUMNS (a disconnected graph: the product of its components');
    NaN for an empty jet."""
    if len(pt) == 0:
        return np.full(len(COLUMNS), np.nan)
    conn = connected_closed_forms(pt, eta, phi, beta)
    return np.array([np.prod([conn[c] for c in components(name)]) for name in COLUMNS])


def literal(edges, z, T):
    """sum over every index tuple (coincident indices included) of prod_v z_iv prod_{(a,b) in edges} T_{ia ib}."""
    if not edges:
        return 1.0
    V = 1 + max(max(e) for e in edges)
    letters = "abcdefghij"
    spec = ",".join(letters[:V]) + "," + ",".join(letters[a] + letters[b] for a, b in edges) + "->"
    return float(np.einsum(spec, *([z] * V), *([T] * len(edges)), optimize=V > 5))


def brute_force(pt, eta, phi, beta=1.0):
    """Every column as the literal sum over the index tuples of its edge list in GRAPHS; small n only."""
    z = pt / pt.sum()
    T = eo.theta(eta, phi, beta)
    return np.array([literal(g, z, T) for g in GRAPHS])


def numpy_batch(x, mask, stats=None, beta=1.0):
    return np.array([closed_forms(*j, beta) for j in eo.used_particles(x, mask, stats)])
