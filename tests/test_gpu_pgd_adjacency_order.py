"""The adjacency-ordered buffers of the one-GPU streamed PGD path: pass 1 stores its partner sums into P1 and both
copies of S_t into S_adj in adjacency order; pass 2 adds its sums to P1 and stores the finished (A, B) of every edge.

Every row position is written by the CTA of its vertex, so the row ends are where a wrong offset shows: vertices
with in-edges but no own edges and the reverse, vertex 0 (no in-edges) and vertex n-1 (no own edges), edges without
slots between edges with slots (they keep S = 1, and their S_adj copies must still hold it), a degree near the table
limit, and the Adam rule.  Each case must match the oracle, and a second solve on the same handle must repeat the
first bit for bit (a stale entry of an earlier solve would show there)."""
import numpy as np
import pytest

import desc_b200
from oracle import desc_oracle as O
from gpu_util import run_oracle, assert_solution_close
from test_gpu_pgd_tables import _holes_graph, _hub_graph

pytestmark = pytest.mark.gpu

RULES = {
    "constant": (lambda: desc_b200.ConstantStepSize(0.05), lambda: O.ConstantStepSize(0.05)),
    "adam": (lambda: desc_b200.HybridGradient(0.002, 0.9, 0.999, 25), lambda: O.HybridGradient(0.002, 0.9, 0.999, 25)),
}


@pytest.fixture(autouse=True)
def _streamed_path(monkeypatch):
    monkeypatch.setenv("DESC_B200_PGD_PATH", "stream")


def _random_rotations(k, rng):
    q = rng.standard_normal((k, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def _pendant_graph():
    """a dense 200-vertex graph whose vertices are spread over ids 0..219; the 20 ids left over (0, 219 and 18
    between) are pendant vertices, each with one edge to a dense vertex.  A pendant edge closes no triangle: no
    slots.  Pendant 0 has one own edge and no in-edges, pendant 219 one in-edge and no own edges, and the others
    put slot-less edges between edges with slots, in the middle of their dense neighbour's row."""
    rng = np.random.default_rng(71)
    mo = O.uniform_topology(200, 0.6, 0.2, 0.1, "uniform", rng=71)
    n = 220
    pend = np.concatenate([[0], np.sort(rng.choice(np.arange(1, n - 1), 18, replace=False)), [n - 1]])
    dense = np.setdiff1d(np.arange(n), pend)            # increasing: (i, j)-order and i < j are kept
    ij = dense[mo["Ind"].astype(np.int64) - 1]
    Rij = mo["RijMat"]
    anchor = rng.choice(dense, pend.size)
    pe = np.stack([np.minimum(pend, anchor), np.maximum(pend, anchor)], axis=1)
    ij = np.concatenate([ij, pe])
    Rij = np.concatenate([Rij, _random_rotations(pend.size, rng)], axis=2)
    order = np.lexsort((ij[:, 1], ij[:, 0]))
    return (ij[order] + 1).astype(np.float64), np.ascontiguousarray(Rij[:, :, order])


def _two_solves(Ind, RijMat, rule_c, iters, ns, seed=3):
    """the first solve as run_cuda returns it, and the (S_vec, hist, w) of a second solve on the same handle"""
    out = {}
    with desc_b200.Solver(Ind, RijMat) as s:
        out["info"] = s.build_incidence(n_sample=ns, seed=seed)
        out["rowptr"], _ = s.incidence()
        s.cycle_inconsistency()
        out["S0"] = s.S0()
        S, hist, it = s.pgd(iters, rule_c())
        out["S_vec"], out["hist"], out["iters_run"] = np.array(S, copy=True), np.array(hist, copy=True), it
        out["w"] = np.array(s.w(), copy=True)
        out["timings"] = s.timings()
        S2, hist2, it2 = s.pgd(iters, rule_c())
        second = (np.array(S2, copy=True), np.array(hist2, copy=True), it2, np.array(s.w(), copy=True))
    return out, second


def _check(Ind, RijMat, rule, iters, ns):
    rule_c, rule_o = RULES[rule]
    c, second = _two_solves(Ind, RijMat, rule_c, iters, ns)
    assert c["timings"]["pgd_pass2_ms"] > 0.0                 # the two-pass streamed path ran
    o = run_oracle(Ind, RijMat, rule_o(), iters, n_sample=ns or None, seed=3, gcw=False)
    assert_solution_close(c, o)
    S2, hist2, it2, w2 = second
    assert it2 == c["iters_run"]
    np.testing.assert_array_equal(S2, c["S_vec"])
    np.testing.assert_array_equal(hist2, c["hist"])
    np.testing.assert_array_equal(w2, c["w"])
    return c


@pytest.mark.parametrize("rule", sorted(RULES))
@pytest.mark.parametrize("ns", [0, 12, 33])
def test_slotless_edges_and_row_ends(rule, ns):
    Ind, RijMat = _pendant_graph()
    i, j = Ind[:, 0] - 1, Ind[:, 1] - 1
    assert np.any(i == 0) and not np.any(j == 0) and np.any(j == 219) and not np.any(i == 219)
    c = _check(Ind, RijMat, rule, 20, ns)
    nslots = np.diff(c["rowptr"])
    empty = nslots == 0
    assert 20 <= empty.sum() < empty.size                     # the pendant edges, next to edges with slots
    assert np.any(empty[:-1] & ~empty[1:]) and np.any(~empty[:-1] & empty[1:]) and np.any(empty[1:-1] & ~empty[:-2] & ~empty[2:])
    np.testing.assert_array_equal(c["S_vec"].ravel()[empty], 1.0)   # S_vec = ones(1, m) where no cycle moves it


@pytest.mark.parametrize("rule", sorted(RULES))
@pytest.mark.parametrize("ns", [0, 40])
def test_rows_without_in_edges_or_own_edges(rule, ns):
    Ind, RijMat = _holes_graph()
    i, j = Ind[:, 0] - 1, Ind[:, 1] - 1
    assert not np.any(i == 40) and np.any(j == 40) and not np.any(j == 90) and np.any(i == 90)
    assert not np.any(j == 0) and not np.any(i == 199)       # vertex 0: own edges only; vertex n-1: in-edges only
    _check(Ind, RijMat, rule, 25, ns)


@pytest.mark.parametrize("rule", sorted(RULES))
def test_degree_near_the_table_limit(rule):
    Ind, RijMat = _hub_graph()
    _check(Ind, RijMat, rule, 12, 0)
