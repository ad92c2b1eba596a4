"""CPU: the numpy statements of tests/efp_d4_oracle.py — every EFP of degree <= 4 against the literal sum over index tuples, the
completeness of the graph set (brute-force enumeration up to isomorphism), the two-particle jet, symmetries and special jets,
and the agreement of the oracle's names with observables.EFP_D4_COLUMNS and the C header's enum."""
import itertools
import os
import re

import numpy as np
import pytest

import efp_d4_oracle as do
import efp_oracle as eo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def random_jet(g, n):
    return g.uniform(0.1, 5.0, n), g.normal(0, 0.4, n), g.normal(0, 0.4, n)


# ---- graphs up to isomorphism ----------------------------------------------------------------------------------------------
def split_components(edges):
    """Edge list -> list of connected components, each relabelled onto 0..V-1 (an edgeless graph has none)."""
    verts = sorted({v for e in edges for v in e})
    parent = {v: v for v in verts}

    def find(v):
        while parent[v] != v:
            v = parent[v]
        return v

    for a, b in edges:
        parent[find(a)] = find(b)
    groups = {}
    for e in edges:
        groups.setdefault(find(e[0]), []).append(e)
    out = []
    for comp in groups.values():
        label = {v: i for i, v in enumerate(sorted({v for e in comp for v in e}))}
        out.append(tuple((label[a], label[b]) for a, b in comp))
    return out


def canonical_connected(edges):
    """The lexicographically smallest sorted edge multiset over all relabellings of a connected graph's vertices."""
    V = 1 + max(max(e) for e in edges)
    best = None
    for perm in itertools.permutations(range(V)):
        form = tuple(sorted(tuple(sorted((perm[a], perm[b]))) for a, b in edges))
        if best is None or form < best:
            best = form
    return best


def canonical(edges):
    """An isomorphism-complete key of any multigraph without isolated vertices: the sorted multiset of its components' forms."""
    return tuple(sorted(canonical_connected(c) for c in split_components(edges)))


def is_connected(edges, V):
    seen, todo = {0}, [0]
    while todo:
        v = todo.pop()
        for a, b in edges:
            for x, y in ((a, b), (b, a)):
                if x == v and y not in seen:
                    seen.add(y)
                    todo.append(y)
    return len(seen) == V


def enumerate_connected(d_max=4):
    """{d: set of canonical forms} of the connected loopless multigraphs with d edges, by brute force: every multiset of d edges
    on V <= d + 1 vertices that uses every vertex and is connected."""
    out = {}
    for d in range(1, d_max + 1):
        found = set()
        for V in range(2, d + 2):
            pairs = list(itertools.combinations(range(V), 2))
            for edges in itertools.combinations_with_replacement(pairs, d):
                if len({v for e in edges for v in e}) == V and is_connected(edges, V):
                    found.add(canonical_connected(edges))
        out[d] = found
    return out


def test_connected_graph_counts():
    conn = enumerate_connected()
    assert [len(conn[d]) for d in (1, 2, 3, 4)] == [1, 2, 5, 12]


def test_oracle_graphs_are_exactly_every_graph_of_degree_at_most_4():
    conn = enumerate_connected()
    every = {(): 0}                                             # the empty graph
    pool = [(f, d) for d in conn for f in conn[d]]
    for k in range(1, 5):                                       # multisets of k connected components, total d <= 4
        for combo in itertools.combinations_with_replacement(sorted(pool), k):
            d = sum(c[1] for c in combo)
            if d <= 4:
                every[tuple(sorted(c[0] for c in combo))] = d
    by_degree = [sum(1 for d in every.values() if d == k) for k in range(5)]
    assert by_degree == [1, 1, 3, 8, 23]
    keys = [canonical(g) for g in do.GRAPHS]
    assert len(keys) == 36 and len(set(keys)) == 36            # pairwise non-isomorphic
    assert set(keys) == set(every)                              # and every graph of degree <= 4
    degrees = [len(g) for g in do.GRAPHS]
    assert degrees == sorted(degrees)                           # ordered by d ...
    for k in range(5):                                          # ... connected before disconnected
        conn_flags = [len(split_components(g)) == 1 for g, d in zip(do.GRAPHS, degrees) if d == k and g]
        assert conn_flags == sorted(conn_flags, reverse=True)
    assert {name for name in do.COLUMNS if len(do.components(name)) == 1} == set(do.CONNECTED)


def test_names_agree_with_python_and_header():
    from multimodal_particles_b200.observables import EFP_COLUMNS, EFP_D4_COLUMNS, FPD_EFP_COLUMNS
    assert EFP_D4_COLUMNS == do.COLUMNS and set(EFP_COLUMNS) <= set(EFP_D4_COLUMNS)
    assert set(FPD_EFP_COLUMNS) <= set(EFP_D4_COLUMNS) and len(FPD_EFP_COLUMNS) <= 64
    text = open(os.path.join(ROOT, "include", "mmbridge.h")).read()
    body = re.search(r"enum \{\s*(MMB_EFPD4_0 = 0,.*?MMB_EFPD4_OBS)\s*\};", text, re.S).group(1)
    names = [n.strip().split("=")[0].strip() for n in body.split(",")]
    assert names[-1] == "MMB_EFPD4_OBS" and len(names) == 37

    def c_name(col):   # efp1^2*efp2_double -> MMB_EFPD4_1_1_2_DOUBLE
        return "MMB_EFPD4_" + "_".join(c[3:].upper() for c in do.components(col)) if col != "efp0" else "MMB_EFPD4_0"
    assert names[:-1] == [c_name(c) for c in do.COLUMNS]


# ---- closed forms ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("beta", [0.5, 1.0, 2.0])
def test_closed_forms_equal_literal_sums(n, beta):
    g = np.random.default_rng(100 + n * 10 + int(beta * 2))
    jet = random_jet(g, n)
    np.testing.assert_allclose(do.closed_forms(*jet, beta), do.brute_force(*jet, beta), rtol=1e-12, atol=1e-15)


def test_shared_columns_equal_the_jetnet_set():
    g = np.random.default_rng(3)
    jet = random_jet(g, 30)
    got = dict(zip(do.COLUMNS, do.closed_forms(*jet)))
    np.testing.assert_allclose([got[c] for c in eo.COLUMNS], eo.closed_forms(*jet), rtol=1e-14)


def bipartition(edges):
    """Part sizes (p, r) of a connected graph's 2-colouring, or None if it has an odd cycle."""
    V = 1 + max(max(e) for e in edges)
    colour = {0: 0}
    todo = [0]
    while todo:
        v = todo.pop()
        for a, b in edges:
            for x, y in ((a, b), (b, a)):
                if x == v:
                    if y not in colour:
                        colour[y] = 1 - colour[v]
                        todo.append(y)
                    elif colour[y] == colour[v]:
                        return None
    p = sum(1 for v in range(V) if colour[v] == 0)
    return p, V - p


def test_two_particle_jet():
    # z = (a, b), theta = delta: a connected bipartite graph with parts (p, r) gives delta^d (a^p b^r + a^r b^p), any graph with
    # a triangle 0; a disconnected graph the product of its components
    pt, eta, phi = np.array([1.0, 3.0]), np.array([0.1, 0.6]), np.array([-0.2, 0.1])
    a, b = pt / pt.sum()
    for beta in (1.0, 2.0):
        delta = np.hypot(0.5, 0.3) ** beta
        want = {}
        for name, edges in do.CONNECTED.items():
            parts = bipartition(edges)
            want[name] = 0.0 if parts is None else delta ** len(edges) * (a ** parts[0] * b ** parts[1] + a ** parts[1] * b ** parts[0])
        assert want["efp3_triangle"] == want["efp4_triangle_double"] == want["efp4_paw"] == 0.0
        expect = [np.prod([want[c] for c in do.components(n)]) for n in do.COLUMNS]
        np.testing.assert_allclose(do.closed_forms(pt, eta, phi, beta), expect, rtol=1e-12, atol=1e-300)


def test_empty_and_single_particle():
    assert np.isnan(do.closed_forms(np.zeros(0), np.zeros(0), np.zeros(0))).all()
    assert do.closed_forms(np.array([2.0]), np.array([0.3]), np.array([1.0])).tolist() == [1.0] + [0.0] * 35


def test_permutation_eta_shift_and_phi_wrap():
    g = np.random.default_rng(7)
    pt, eta, phi = random_jet(g, 40)
    phi = np.clip(phi, -0.9, 0.9)
    base = do.closed_forms(pt, eta, phi)
    p = g.permutation(40)
    np.testing.assert_allclose(do.closed_forms(pt[p], eta[p], phi[p]), base, rtol=1e-12)
    np.testing.assert_allclose(do.closed_forms(pt, eta + 1.7, phi), base, rtol=1e-10)
    rot = phi + 2.8                                            # straddles +pi: wrapped differences are unchanged
    rot = np.where(rot > np.pi, rot - 2 * np.pi, rot)
    assert (rot > 0).any() and (rot < 0).any()
    np.testing.assert_allclose(do.closed_forms(pt, eta, rot), base, rtol=1e-10)


@pytest.mark.parametrize("beta", [0.5, 1.0, 2.0])
def test_double_edge_is_the_edge_at_twice_beta(beta):
    g = np.random.default_rng(11)
    jet = random_jet(g, 25)
    i2, i1 = do.COLUMNS.index("efp2_double"), do.COLUMNS.index("efp1")
    assert do.closed_forms(*jet, beta)[i2] == pytest.approx(do.closed_forms(*jet, 2 * beta)[i1], rel=1e-12)
