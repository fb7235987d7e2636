"""The per-vertex tables of the streamed PGD path: S in adjacency order (S_adj, refilled after every pass 1) and
the partner sums of the pass over larger endpoints (acc2, plain stores, ping-ponged with acc).

Stale entries of either buffer would leak values of an earlier iteration, solve or incidence into a later one, so
repeated solves on one handle must equal a fresh handle bit for bit; table edge cases (odd row offsets, vertices
without lower neighbours or without own edges, a degree near the table limit, slot lists across 32 / 64, Adam)
must match the oracle at the usual bars."""
import numpy as np
import pytest

import desc_b200
from oracle import desc_oracle as O
from gpu_util import run_cuda, run_oracle, assert_solution_close

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _streamed_path(monkeypatch):
    monkeypatch.setenv("DESC_B200_PGD_PATH", "stream")


def _subgraph(mo, keep):
    """the model restricted to the edges `keep` (a boolean mask): Ind stays (i,j)-sorted, vertices keep their ids"""
    return mo["Ind"][keep], mo["RijMat"][:, :, keep]


def _holes_graph():
    """vertex 40 without own edges (no neighbour above it), vertex 90 without lower neighbours"""
    mo = O.uniform_topology(200, 0.7, 0.2, 0.1, "uniform", rng=61)
    i, j = mo["Ind"][:, 0] - 1, mo["Ind"][:, 1] - 1
    return _subgraph(mo, ~((i == 40) | (j == 90)))


def _hub_graph():
    """one vertex adjacent to 2860 of 2900 others: a table of ~2860 entries (the second pass's shared-memory
    table holds about 2890), among sparse random edges that close triangles through the hub"""
    rng = np.random.default_rng(62)
    n, hub = 2900, 1500
    others = np.setdiff1d(np.arange(n), [hub])
    nb = np.sort(rng.choice(others, 2860, replace=False))
    pairs = {(min(hub, int(k)), max(hub, int(k))) for k in nb}
    while len(pairs) < 2860 + 9000:
        a, b = (int(x) for x in rng.choice(others, 2, replace=False))
        pairs.add((min(a, b), max(a, b)))
    ij = np.array(sorted(pairs), dtype=np.int64)
    Ind = (ij + 1).astype(np.float64)
    q = rng.standard_normal((len(ij), 4))                     # random rotations from unit quaternions
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    w, x, y, z = q.T
    Rij = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                    [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                    [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
    return Ind, Rij


def _degrees(Ind, n):
    return np.bincount((Ind.astype(np.int64) - 1).ravel(), minlength=n)


def _check(Ind, RijMat, rule_c, rule_o, iters, ns, seed=3):
    c = run_cuda(Ind, RijMat, rule_c, iters, n_sample=ns, seed=seed, gcw=False)
    assert c["timings"]["pgd_pass2_ms"] > 0.0                 # the two-pass streamed path ran
    o = run_oracle(Ind, RijMat, rule_o, iters, n_sample=ns or None, seed=seed, gcw=False)
    assert_solution_close(c, o)
    return c


@pytest.mark.parametrize("ns", [32, 33, 64, 65])
def test_rows_without_lower_or_upper_neighbours(ns):
    Ind, RijMat = _holes_graph()
    deg = _degrees(Ind, 200)
    assert np.any(np.cumsum(deg)[:-1] % 2 == 1)               # odd row offsets: the widened S-table copy
    i, j = Ind[:, 0] - 1, Ind[:, 1] - 1
    assert not np.any(i == 40) and np.any(j == 40) and not np.any(j == 90) and np.any(i == 90)
    c = _check(Ind, RijMat, desc_b200.ConstantStepSize(0.05), O.ConstantStepSize(0.05), 20, ns)
    assert c["info"]["max_slots_per_edge"] == ns              # slot lists right at / just past 32 and 64


def test_degree_near_the_table_limit():
    Ind, RijMat = _hub_graph()
    assert 2850 <= _degrees(Ind, 2900).max() <= 2890
    _check(Ind, RijMat, desc_b200.ConstantStepSize(0.05), O.ConstantStepSize(0.05), 12, 0)


def test_adam_rule():
    Ind, RijMat = _holes_graph()
    _check(Ind, RijMat, desc_b200.HybridGradient(0.002, 0.9, 0.999, 25), O.HybridGradient(0.002, 0.9, 0.999, 25),
           30, 40)


def _solve(s, n_sample, iters=25):
    s.build_incidence(n_sample=n_sample, seed=5)
    s.cycle_inconsistency()
    S, hist, it = s.pgd(iters, desc_b200.ConstantStepSize(0.05))
    return np.array(S, copy=True), np.array(hist, copy=True), it, np.array(s.w(), copy=True)


def _fresh(Ind, RijMat, n_sample, iters=25):
    with desc_b200.Solver(Ind, RijMat) as s:
        return _solve(s, n_sample, iters)


def _same(a, b):
    for x, y in zip(a, b):
        if isinstance(x, np.ndarray):
            np.testing.assert_array_equal(x, y)
        else:
            assert x == y


def test_repeated_solves_and_rebuilt_incidence_equal_a_fresh_handle():
    """every S_adj / acc2 entry is rewritten by every solve: nothing of an earlier solve or incidence leaks in"""
    Ind, RijMat = _holes_graph()
    ref40, ref12 = _fresh(Ind, RijMat, 40), _fresh(Ind, RijMat, 12)
    ref40_odd = _fresh(Ind, RijMat, 40, iters=7)               # ends on the other ping-pong buffer
    with desc_b200.Solver(Ind, RijMat) as s:
        _same(_solve(s, 40), ref40)
        _same(_solve(s, 40), ref40)
        _same(_solve(s, 12), ref12)                            # fewer slots: rows that had in-edges may have none
        _same(_solve(s, 40, iters=7), ref40_odd)
        _same(_solve(s, 40), ref40)
