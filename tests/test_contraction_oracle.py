"""Pins the contraction oracle (oracle/contraction_oracle.py): golden vectors produced by the unmodified
reference (tests/golden/contract_*.npz, tests/golden/live_reference.npz), the reference's own known-answer
tests (tests/shm/coarsening/cluster_contraction_test.cc) and size-independent properties."""
import hashlib
import os

import numpy as np
import pytest

from kaminpar_b200 import graph as G
from oracle import contraction_oracle as CO
from tests import helpers as H

LIVE = os.path.join(H.GOLDEN, "live_reference.npz")
CASES = ["rgg2d_k4", "rgg16_w", "walshaw_k16", "walshaw_unsorted", "rmat13_w", "grid12", "road60", "star30000"]


def oracle_of(g, cl):
    return CO.contract(g.xadj, g.adjncy, g.vwgt, g.adjwgt, cl)


@pytest.mark.parametrize("name", CASES)
def test_oracle_reproduces_reference_golden(name):
    g, _ = H.load_case(name)
    d = np.load(os.path.join(H.GOLDEN, f"contract_{name}.npz"))
    ref = CO.canonicalize(int(d["c_n"][0]), d["c_xadj"], d["c_adjncy"], d["c_vwgt"], d["c_adjwgt"], d["mapping"],
                          clustering=d["clustering"])
    assert CO.equal(oracle_of(g, d["clustering"]), ref)


def grid2d(rows, cols):  # tests/shm/graph_factories.h make_grid_graph: row by row
    edges = []
    for r in range(rows):
        for c in range(cols):
            u = r * cols + c
            if c + 1 < cols:
                edges.append((u, u + 1))
            if r + 1 < rows:
                edges.append((u, u + cols))
    return H.from_edges(rows * cols, edges)


def weighted_endpoints(o):
    src = np.repeat(np.arange(o["c_n"]), np.diff(o["c_xadj"].astype(np.int64)))
    return {(int(o["c_vwgt"][a]), int(o["c_vwgt"][b])) for a, b in zip(src, o["c_adjncy"])}


def test_reference_kats():
    # ContractingToSingleNodeWorks (cluster_contraction_test.cc:19-43)
    g = grid2d(2, 2)
    for c in range(4):
        o = oracle_of(g, np.full(4, c, np.uint32))
        assert o["c_n"] == 1 and len(o["c_adjncy"]) == 0 and o["c_vwgt"][0] == 4
    # ContractingToSingletonsWorks (:45-77)
    g.vwgt = np.array([1, 2, 3, 4], np.int32)
    o = oracle_of(g, np.arange(4, dtype=np.uint32))
    assert o["c_n"] == 4 and len(o["c_adjncy"]) == g.m and o["c_vwgt"].sum() == 10 and o["c_adjwgt"].sum() == g.m
    assert {(1, 2), (1, 3), (2, 4), (3, 4)} <= weighted_endpoints(o)
    # ContractingAllNodesButOneWorks (:79-105)
    g = grid2d(2, 2)
    o = oracle_of(g, np.array([0, 1, 1, 1], np.uint32))
    assert o["c_n"] == 2 and len(o["c_adjncy"]) == 2 and o["c_adjwgt"].sum() == 4 and (1, 3) in weighted_endpoints(o)
    # ContractingGridHorizontallyWorks (:107-145)
    g = grid2d(2, 4)
    g.vwgt = np.array([1, 2, 3, 4, 10, 20, 30, 40], np.int32)
    o = oracle_of(g, np.array([0, 1, 2, 3, 0, 1, 2, 3], np.uint32))
    assert o["c_n"] == 4 and len(o["c_adjncy"]) == 6 and sorted(o["c_vwgt"]) == [11, 22, 33, 44]
    assert o["c_adjwgt"].sum() == 12 and {(11, 22), (22, 33), (33, 44)} <= weighted_endpoints(o)
    # ContractingGridVerticallyWorks (:147-185)
    g = grid2d(4, 2)
    g.vwgt = np.array([1, 10, 2, 20, 3, 30, 4, 40], np.int32)
    o = oracle_of(g, np.array([0, 0, 2, 2, 4, 4, 6, 6], np.uint32))
    assert o["c_n"] == 4 and len(o["c_adjncy"]) == 6 and sorted(o["c_vwgt"]) == [11, 22, 33, 44]
    assert o["c_adjwgt"].sum() == 12 and {(11, 22), (22, 33), (33, 44)} <= weighted_endpoints(o)


def live_graphs():
    return [G.rmat(12, 8, 3), G.grid3d(9), G.random_weights(G.rgg2d(3000, 1), 5, max_vwgt=3, max_adjwgt=5), H.big_star(5000)]


def live_clusterings(g, rng):
    return (rng.integers(0, g.n, g.n).astype(np.uint32), np.arange(g.n, dtype=np.uint32),
            (np.arange(g.n) // 7 * 7).astype(np.uint32), np.zeros(g.n, np.uint32))


def digest(o):
    """sha256 of a canonical contraction result (the fixture stores the reference's as this fingerprint)."""
    h = hashlib.sha256(np.int64(o["c_n"]).tobytes())
    for key, dtype in (("c_xadj", np.uint32), ("c_adjncy", np.uint32), ("c_vwgt", np.int32), ("c_adjwgt", np.int32),
                       ("mapping", np.uint32)):
        h.update(np.ascontiguousarray(o[key], dtype).tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("algorithm", [0, 1, 2])
def test_oracle_matches_live_reference(algorithm):
    """The oracle == the reference's BUFFERED (0), UNBUFFERED (1) and UNBUFFERED_NAIVE (2) contraction after
    canonicalisation; the reference's results are stored by tests/golden/make_live_reference_golden.py."""
    d = np.load(LIVE)
    want = zip(d[f"contract_a{algorithm}_c_n"], d[f"contract_a{algorithm}_c_m"], d[f"contract_a{algorithm}_sha256"])
    rng = np.random.default_rng(algorithm)
    got = [(o["c_n"], len(o["c_adjncy"]), digest(o)) for g in live_graphs() for o in
           (oracle_of(g, cl) for cl in live_clusterings(g, rng))]
    assert got == [(int(c_n), int(c_m), str(h)) for c_n, c_m, h in want]


def test_properties():
    rng = np.random.default_rng(7)
    g = G.random_weights(G.rmat(13, 8, 5), 3, max_vwgt=4, max_adjwgt=6)
    cl = rng.integers(0, g.n // 5, g.n).astype(np.uint32)
    o = oracle_of(g, cl)
    assert o["c_vwgt"].sum() == g.total_node_weight()
    src = np.repeat(np.arange(g.n), np.diff(g.xadj.astype(np.int64)))
    cut_w = g.adjwgt[o["mapping"][src] != o["mapping"][g.adjncy]].astype(np.int64).sum()
    assert o["c_adjwgt"].astype(np.int64).sum() == cut_w
    csrc = np.repeat(np.arange(o["c_n"]), np.diff(o["c_xadj"].astype(np.int64)))
    assert (csrc != o["c_adjncy"]).all()  # no self-loops
    fwd = dict(zip(zip(csrc.tolist(), o["c_adjncy"].tolist()), o["c_adjwgt"].tolist()))
    assert all(fwd[(b, a)] == w for (a, b), w in fwd.items())  # symmetric with equal weights
    # idempotence: contracting the coarse graph by the identity clustering changes nothing
    o2 = CO.contract(o["c_xadj"], o["c_adjncy"], o["c_vwgt"], o["c_adjwgt"], np.arange(o["c_n"]))
    assert all(np.array_equal(o[k], o2[k]) for k in ("c_xadj", "c_adjncy", "c_vwgt", "c_adjwgt"))
    # projections
    coarse = rng.integers(0, 8, o["c_n"]).astype(np.uint32)
    fine = CO.project_up(o["mapping"], coarse)
    assert np.array_equal(CO.project_down(o["mapping"], fine, o["c_n"]), coarse)


def test_empty_graph():
    o = CO.contract(np.zeros(1, np.uint32), np.zeros(0, np.uint32), None, None, np.zeros(0, np.uint32))
    assert o["c_n"] == 0 and len(o["c_xadj"]) == 1


def multigraph_cases():
    """Random small graphs with parallel edges, self-loops and weights, and random clusterings (seeded)."""
    draw = np.random.default_rng(2)
    params = [(1, 0, 0), (1, 3, 1), (40, 0, 2), (40, 120, 3)]
    params += [(int(draw.integers(1, 41)), int(draw.integers(0, 121)), int(draw.integers(0, 2**31 - 1))) for _ in range(36)]
    for n, m_und, seed in params:
        rng = np.random.default_rng(seed)
        edges = [(int(a), int(b)) for a, b in rng.integers(0, n, (m_und, 2))]
        g = H.from_edges(n, edges, vwgt=rng.integers(1, 5, n), ew=rng.integers(1, 6, m_und).tolist())
        yield g, rng.integers(0, n, n).astype(np.uint32)


def test_oracle_matches_live_reference_random_multigraphs():
    """The oracle == the unmodified reference (default algorithm, raw results stored by
    tests/golden/make_live_reference_golden.py) after canonicalisation."""
    d = np.load(LIVE)
    cases = list(multigraph_cases())
    assert len(cases) == len(d["multigraph_c_n"])
    for i, (g, cl) in enumerate(cases):
        r = {k: d[f"multigraph{i}_{k}"] for k in ("c_xadj", "c_adjncy", "c_vwgt", "c_adjwgt", "mapping")}
        assert CO.equal(oracle_of(g, cl), CO.canonicalize(int(d["multigraph_c_n"][i]), **r, clustering=cl))
