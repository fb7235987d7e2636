"""GPU parity tests: CUDA path (through the C ABI) vs the CPU oracle and the golden fixtures.

Run on a B200 with ``pytest -m gpu``.  Everything goes through ``libdesc_b200.so``; if the
library is missing or no device is visible these tests FAIL (there is no fallback to test).
"""
import numpy as np
import pytest

import desc_b200
from desc_b200 import _lib
from conftest import golden_names, load_golden, golden_rule, golden_csr
from oracle import desc_oracle as O
from gpu_util import (run_cuda, run_oracle, assert_incidence_equal, assert_solution_close, rel_err, RTOL,
                      ROT_TOL_DEG)

pytestmark = pytest.mark.gpu


def _ns_args(ns):
    """(cuda n_sample, oracle n_sample) for a fixture/override value: None/-1 -> reference rule"""
    if ns is None or ns < 0:
        return 0, None
    return int(ns), int(ns)


# ---------------------------------------------------------------------------------------------
# golden fixtures (literal restatement of DESC.m / GCW.m)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", golden_names())
def test_golden_fixture(name):
    g = load_golden(name)
    cns, _ = _ns_args(int(g["n_sample_arg"]))
    c = run_cuda(g["Ind"], g["RijMat"], golden_rule(g, desc_b200), int(g["iters"]), n_sample=cns,
                 seed=int(g["sampler_seed"]))
    assert c["info"]["n_sample"] == int(g["n_sample"])
    m = g["Ind"].shape[0]
    cnt = np.zeros(m, dtype=np.int64)
    cnt[g["CoDeg_pos_ind"] - 1] = np.diff(g["cum_ind"])
    np.testing.assert_array_equal(np.diff(c["rowptr"]), cnt)
    np.testing.assert_array_equal(c["apex"] + 1, g["IJK"])
    np.testing.assert_array_equal(c["e_jk"] + 1, g["Ind_jk"])
    np.testing.assert_array_equal(c["e_ki"] + 1, g["Ind_ki"])
    np.testing.assert_array_equal(c["ikj"], g["IKJ"] > 0)
    np.testing.assert_array_equal(c["jki"], g["JKI"] > 0)
    assert rel_err(c["S0"], g["S0_long"], floor=1e-30) <= RTOL
    assert c["iters_run"] == int(g["iters_run"])
    assert rel_err(c["S_vec"], g["S_vec"], floor=1e-12) <= RTOL
    assert rel_err(c["hist"][:, 1], g["hist"][:, 1], floor=1e-9) <= RTOL
    assert np.max(np.abs(c["w"] - g["wijk"])) <= 1e-11
    ang = O.aligned_angle_deg(c["R"], g["R_est"])
    assert ang.mean() <= ROT_TOL_DEG


@pytest.mark.parametrize("name", golden_names())
def test_golden_fixture_laa_refinement(name):
    """DESC.m:265-312 on the fixture's own (S_vec, R_est): same IRLS iterations, scores and rotations"""
    g = load_golden(name)
    with desc_b200.Solver(g["Ind"], g["RijMat"]) as s:
        R, scores = s.refine(S_vec=g["S_vec"], R_init=g["R_est"])
    assert len(scores) == len(g["laa_scores"])
    np.testing.assert_allclose(scores, g["laa_scores"], rtol=1e-7, atol=1e-11)
    assert O.aligned_angle_deg(R, g["R_laa"]).mean() <= ROT_TOL_DEG


@pytest.mark.parametrize("name", ["uniform_n60_sigma0", "nonuniform_n64_adv"])
def test_golden_fixture_explicit_cycle_lists(name):
    """the cycle lists of a reference run can be passed in (what a MATLAB datasample drew),
    here in a random per-edge order as datasample would return them"""
    g = load_golden(name)
    ptr, apex = golden_csr(g)
    rng = np.random.default_rng(5)
    apex = apex.copy()
    for e in range(ptr.size - 1):
        apex[ptr[e]:ptr[e + 1]] = rng.permutation(apex[ptr[e]:ptr[e + 1]])
    rule_c, rule_o = golden_rule(g, desc_b200), golden_rule(g, O)
    c = run_cuda(g["Ind"], g["RijMat"], rule_c, int(g["iters"]), cycles=(ptr, apex))
    o = run_oracle(g["Ind"], g["RijMat"], rule_o, int(g["iters"]), cycles=(ptr, apex))
    np.testing.assert_array_equal(c["apex"], apex)
    np.testing.assert_array_equal(c["e_jk"], o["inc"].e_jk)
    np.testing.assert_array_equal(c["ikj"], o["inc"].IKJ >= 0)
    np.testing.assert_array_equal(c["jki"], o["inc"].JKI >= 0)
    assert_solution_close(c, o)
    # permuting the lists only changes FP summation order: same S_vec as the fixture
    assert rel_err(c["S_vec"], g["S_vec"], floor=1e-12) <= RTOL


# ---------------------------------------------------------------------------------------------
# BASELINE.json configurations against the oracle on the same seeded inputs
# ---------------------------------------------------------------------------------------------
def test_config1_uniform_n200_sigma0():
    """configs[0]: Uniform_Topology n=200 p=0.5 q=0.2 sigma=0, iters=100, ConstantStepSize(0.01)"""
    mo = O.uniform_topology(200, 0.5, 0.2, 0.0, "uniform", rng=0)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.01), 100, seed=1)
    o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(0.01), 100, seed=1)
    assert_incidence_equal(c, o["inc"])
    assert_solution_close(c, o)
    assert np.mean(np.abs(c["S_vec"] - mo["ErrVec"])) < 2e-3       # exact-recovery regime
    _, _, mean_err, _ = O.rotation_alignment(c["R"], mo["R_orig"])
    assert mean_err < 0.05


def test_config2_shape_reduced_n400():
    """configs[1] shape (p=0.5 q=0.3 sigma=0.1) at n=400 so the oracle finishes in seconds"""
    mo = O.uniform_topology(400, 0.5, 0.3, 0.1, "uniform", rng=2)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.01), 60, seed=9)
    o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(0.01), 60, seed=9)
    assert_incidence_equal(c, o["inc"])
    assert_solution_close(c, o)


def test_config2_full_n1000_few_iterations():
    """configs[1] at full size: incidence, d_ijk and 3 PGD iterations against the oracle"""
    mo = O.uniform_topology(1000, 0.5, 0.3, 0.1, "uniform", rng=4)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.01), 3, seed=2, want_w=False)
    o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(0.01), 3, seed=2)
    assert c["info"]["n_sample"] == 63
    assert_incidence_equal(c, o["inc"])
    assert_solution_close(c, o)


def test_config3_nonuniform_adversarial_reduced():
    """configs[2] shape (Nonuniform_Topology, self-consistent adversarial corruption) at n=300"""
    for crpt in ("adv", "self-consistent"):
        mo = O.nonuniform_topology(300, 0.5, 0.3, 0.5, 0.1, 0.1, crpt, rng=6)
        c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.01), 50, seed=3)
        o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(0.01), 50, seed=3)
        assert_incidence_equal(c, o["inc"])
        assert_solution_close(c, o)


def test_large_scale_settings_lr1_iters30():
    """Demo/compare_algorithms.m:2-5: learning_rate=1, ConstantStepSize(1), iters=30"""
    mo = O.uniform_topology(250, 0.3, 0.2, 0.05, "self-consistent", rng=8)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(1.0), 30, seed=4)
    o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(1.0), 30, seed=4)
    assert_incidence_equal(c, o["inc"])
    assert_solution_close(c, o)


@pytest.mark.parametrize("ns", [-1, 5, 17, 40, 100])
def test_sampling_budgets(ns):
    """n_sample below / around / above the co-degrees, and 'keep every triangle'"""
    mo = O.uniform_topology(120, 0.5, 0.2, 0.1, "uniform", rng=10)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.02), 25, n_sample=ns, seed=77)
    o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(0.02), 25, n_sample=ns, seed=77)
    if ns > 0:
        assert_incidence_equal(c, o["inc"])
    else:
        np.testing.assert_array_equal(c["apex"], o["inc"].k)
        np.testing.assert_array_equal(c["ikj"], o["inc"].IKJ >= 0)
    assert_solution_close(c, o)


def test_step_rules_piecewise_and_adam():
    mo = O.uniform_topology(150, 0.4, 0.25, 0.05, "uniform", rng=12)
    for mk in (lambda M: M.PiecewiseStepSize(0.05, 7), lambda M: M.HybridGradient(0.003, 0.9, 0.999, 10),
               lambda M: M.HybridGradient(0.0005, 0.9, 0.999, 5).stopAdam()):
        rc, ro = mk(desc_b200), mk(O)
        c = run_cuda(mo["Ind"], mo["RijMat"], rc, 40, seed=5, gcw=False)
        o = run_oracle(mo["Ind"], mo["RijMat"], ro, 40, seed=5, gcw=False)
        assert_solution_close(c, o, check_R=False)
        assert rc.t == ro.t == 40                       # the rule object's call counter advances


def test_early_stop_patience_matches_reference():
    """DESC.m:243-256: stop after 30 consecutive iterations with objective decrease < 1e-5"""
    mo = O.uniform_topology(80, 0.5, 0.1, 0.0, "uniform", rng=14)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(1.0), 400, seed=6)
    o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(1.0), 400, seed=6)
    assert o["iters_run"] < 400, "test graph should trigger the early stop"
    assert_solution_close(c, o)


# ---------------------------------------------------------------------------------------------
# edge cases
# ---------------------------------------------------------------------------------------------
def _rot_edges(Ind, n, seed):
    rng = np.random.default_rng(seed)
    Rn = O.proj_so3(rng.standard_normal((n, 3, 3)))
    ei, ej = Ind[:, 0].astype(int) - 1, Ind[:, 1].astype(int) - 1
    R = Rn[ei] @ Rn[ej].transpose(0, 2, 1)
    R = O.proj_so3(R + 0.05 * rng.standard_normal(R.shape))
    return O.to_matlab(R)


def test_edges_without_cycles_keep_s_equal_one():
    Ind = [[i, j] for i in range(1, 7) for j in range(i + 1, 7)] + [[6, 7], [7, 8], [3, 8]]
    Ind = np.array(sorted(Ind), dtype=np.float64)
    R = _rot_edges(Ind, 8, 1)
    c = run_cuda(Ind, R, desc_b200.ConstantStepSize(0.05), 20)
    o = run_oracle(Ind, R, O.ConstantStepSize(0.05), 20)
    assert_incidence_equal(c, o["inc"])
    assert_solution_close(c, o)
    assert (c["S_vec"][c["codeg"] == 0] == 1.0).all() and (c["codeg"] == 0).sum() == 3


def test_triangle_free_graph():
    """no 3-cycle at all: m_cycle = 0, S_vec stays ones(1,m) (DESC.m:148), GCW still runs"""
    n = 12
    Ind = np.array([[i, i + 1] for i in range(1, n)] + [[1, n]], dtype=np.float64)
    Ind = Ind[np.lexsort((Ind[:, 1], Ind[:, 0]))]
    R = _rot_edges(Ind, n, 2)
    c = run_cuda(Ind, R, desc_b200.ConstantStepSize(0.05), 5)
    assert c["info"]["m_cycle"] == 0 and c["info"]["m_pos"] == 0
    np.testing.assert_array_equal(c["S_vec"], 1.0)
    o_R = O.gcw(Ind, R, np.ones(Ind.shape[0]))
    assert O.aligned_angle_deg(c["R"], o_R).mean() <= 1e-5      # ring graph: tiny spectral gap


def test_single_triangle():
    Ind = np.array([[1, 2], [1, 3], [2, 3]], dtype=np.float64)
    R = _rot_edges(Ind, 3, 3)
    c = run_cuda(Ind, R, desc_b200.ConstantStepSize(0.1), 10)
    o = run_oracle(Ind, R, O.ConstantStepSize(0.1), 10)
    assert_incidence_equal(c, o["inc"])
    assert_solution_close(c, o)


def test_zero_iterations_returns_initial_state():
    mo = O.uniform_topology(60, 0.5, 0.2, 0.1, rng=20)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.01), 0, gcw=False)
    o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(0.01), 0, gcw=False)
    assert c["iters_run"] == 0
    assert rel_err(c["S_vec"], o["S_vec"], floor=1e-12) <= RTOL


def test_clean_graph_known_answer():
    """q=0, sigma=0: every d_ijk is rounding noise, S_vec ~ 0, rotations exact (SURVEY section 4)"""
    mo = O.uniform_topology(90, 0.5, 0.0, 0.0, rng=21)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.01), 10)
    assert c["S0"].max() < 1e-7 and c["S_vec"].max() < 1e-7
    assert O.aligned_angle_deg(c["R"], mo["R_orig"]).max() < 1e-5


@pytest.mark.parametrize("kind", ["errvec", "random_sq", "ones", "tiny"])
def test_gcw_standalone_matches_oracle_and_returns_rotations(kind):
    """GCW on its own (Utils/GCW.m:1) for S_vec inputs of very different conditioning: the true
    corruption levels (large spectral gap), random weights spanning 8 decades (tiny gap), all ones
    (unweighted, = Spectral.m up to row normalisation) and all ~0 (weights 1e8)"""
    mo = O.uniform_topology(150, 0.3, 0.2, 0.1, rng=22)
    rng = np.random.default_rng(0)
    m = mo["Ind"].shape[0]
    S = {"errvec": mo["ErrVec"], "random_sq": rng.random(m) ** 2, "ones": np.ones(m),
         "tiny": 1e-9 * rng.random(m)}[kind]
    R = desc_b200.GCW(mo["Ind"], mo["AdjMat"], mo["RijMat"], S)
    Ro = O.gcw(mo["Ind"], mo["RijMat"], S)
    assert O.aligned_angle_deg(R, Ro).mean() <= ROT_TOL_DEG
    Ri = O.to_internal(R)
    np.testing.assert_allclose(Ri @ Ri.transpose(0, 2, 1), np.broadcast_to(np.eye(3), Ri.shape), atol=1e-12)
    np.testing.assert_allclose(np.linalg.det(Ri), 1.0, atol=1e-12)


def test_reference_style_entry_points():
    mo = O.uniform_topology(100, 0.5, 0.2, 0.1, rng=23)
    params = dict(iters=30, learning_rate=0.01, make_plots=False, Gradient=desc_b200.ConstantStepSize(0.01),
                  R_orig=mo["R_orig"], ErrVec=mo["ErrVec"], seed=3)
    S1 = desc_b200.DESC_PGD(mo["Ind"], mo["RijMat"], params)
    R2, S2 = desc_b200.DESC_init(mo["Ind"], mo["RijMat"], params)
    assert S1.shape == (1, mo["Ind"].shape[0]) and R2.shape == (3, 3, 100)
    np.testing.assert_array_equal(S1, S2)                        # atomic-free path: bit-reproducible
    oR, oS = O.DESC_init(mo["Ind"], mo["RijMat"], dict(iters=30, Gradient=O.ConstantStepSize(0.01)), seed=3)
    assert rel_err(S2.ravel(), oS, floor=1e-12) <= RTOL
    assert O.aligned_angle_deg(R2, oR).mean() <= ROT_TOL_DEG


# ---------------------------------------------------------------------------------------------
# error behaviour of the boundary
# ---------------------------------------------------------------------------------------------
def test_boundary_rejects_contract_violations():
    mo = O.uniform_topology(30, 0.5, 0.2, 0.1, rng=24)
    Ind, R = mo["Ind"], mo["RijMat"]
    bad = Ind.copy()
    bad[[0, 1]] = bad[[1, 0]]                                   # not sorted by (i,j)
    with pytest.raises(desc_b200.DescError) as e:
        desc_b200.Solver(bad, R)
    assert e.value.code == _lib.ERR_ARG
    bad = Ind.copy()
    bad[:, [0, 1]] = bad[:, [1, 0]]                             # i > j
    with pytest.raises(desc_b200.DescError):
        desc_b200.Solver(bad, R)
    bad = Ind.copy()
    bad[bad == bad.max()] += 1                                  # node n is isolated -> GCW.m:21 divides by 0
    with pytest.raises(desc_b200.DescError) as e:
        desc_b200.Solver(bad, R)
    assert e.value.code == _lib.ERR_ARG
    with desc_b200.Solver(Ind, R) as s:
        with pytest.raises(desc_b200.DescError) as e:
            s.cycle_inconsistency()                             # before build_incidence
        assert e.value.code == _lib.ERR_STATE
        s.build_incidence()
        with pytest.raises(desc_b200.DescError) as e:
            s.pgd(3, desc_b200.ConstantStepSize(0.1))           # before cycle_inconsistency
        assert e.value.code == _lib.ERR_STATE
        with pytest.raises(desc_b200.DescError) as e:
            s.gcw()                                             # no S_vec yet
        assert e.value.code == _lib.ERR_STATE
        ptr = np.arange(Ind.shape[0] + 1, dtype=np.int64)
        with pytest.raises(desc_b200.DescError) as e:
            s.build_incidence(cycles=(ptr, np.full(Ind.shape[0], int(Ind[0, 0]) - 1, dtype=np.int32)))
        assert e.value.code == _lib.ERR_ARG                     # apex is not a common neighbour
    with desc_b200.Solver(Ind, R) as s:
        with pytest.raises(desc_b200.DescError) as e:
            s.refine()                                          # no S_vec / R_init on the handle yet
        assert e.value.code == _lib.ERR_STATE
        with pytest.raises(desc_b200.DescError) as e:
            s.refine(S_vec=np.full(Ind.shape[0], 0.1))          # S_vec given, but no rotations to start from
        assert e.value.code == _lib.ERR_STATE
        with pytest.raises(ValueError):
            s.refine(S_vec=np.zeros(3), R_init=mo["R_orig"])
        Rr, sc = s.refine(S_vec=np.full(Ind.shape[0], 0.1), R_init=mo["R_orig"])   # explicit inputs suffice
        assert Rr.shape == mo["R_orig"].shape and len(sc) >= 1


def test_solve_entry_point_and_device_resident_inputs():
    import ctypes as C
    import torch
    mo = O.uniform_topology(120, 0.5, 0.2, 0.1, rng=25)
    m = mo["Ind"].shape[0]
    Ind_d = torch.from_numpy(np.asfortranarray(mo["Ind"]).ravel(order="K").copy()).cuda()
    R_d = torch.from_numpy(np.asfortranarray(mo["RijMat"]).ravel(order="K").copy()).cuda()
    lib = _lib.load()
    with desc_b200.Solver(Ind_d, R_d) as s:
        S = np.empty(m)
        R = np.empty((3, 3, 120), order="F")
        hist = np.zeros((20, 2))
        run = C.c_int32(0)
        rule = desc_b200.ConstantStepSize(0.01)._to_c()
        _lib.check(lib.desc_b200_solve(s._h, 0, 7, 20, C.byref(rule), S.ctypes.data, R.ctypes.data,
                                       hist.ctypes.data, C.byref(run)))
        t = s.timings()
    oR, oS = O.DESC_init(mo["Ind"], mo["RijMat"], dict(iters=20, Gradient=O.ConstantStepSize(0.01)), seed=7)
    assert run.value == 20 and t["h2d_ms"] == 0.0 and t["pgd_launches"] > 0
    assert rel_err(S, oS, floor=1e-12) <= RTOL
    assert O.aligned_angle_deg(R, oR).mean() <= ROT_TOL_DEG


def test_multi_gpu_parity_when_more_than_one_device():
    """N-rank (NCCL) solve == 1-rank solve; needs >= 2 visible GPUs, otherwise skipped (the N>1 host
    logic is covered on CPU by tests/test_dist_cpu.py)"""
    import os
    import subprocess
    import sys
    n = desc_b200.device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    n = 2 if n < 4 else (4 if n < 8 else 8)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n),
                        "--master-addr", "127.0.0.1", "--master-port", "29517",
                        os.path.join(root, "tests", "multi_gpu_check.py"), "--full"], capture_output=True, text=True,
                       timeout=1200)
    assert "MULTI_GPU_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_generic_atomic_path_still_matches_oracle(monkeypatch):
    """the edge-range FP64-atomic kernel is the fallback for graphs whose degrees exceed the
    shared-memory tables of the vertex-blocked kernel; force it and check parity"""
    monkeypatch.setenv("DESC_B200_PGD_PATH", "generic")
    mo = O.uniform_topology(160, 0.5, 0.25, 0.1, "uniform", rng=31)
    for ns in (0, 70):
        c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.02), 40, n_sample=ns, seed=8)
        o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(0.02), 40, n_sample=ns or None, seed=8)
        assert_incidence_equal(c, o["inc"])
        assert_solution_close(c, o)


@pytest.mark.parametrize("path", ["stream"])
def test_default_paths_are_bit_reproducible(monkeypatch, path):
    """streamed path: no atomics at all.  Two runs give bit-identical S_vec, w and history"""
    monkeypatch.setenv("DESC_B200_PGD_PATH", path)
    mo = O.uniform_topology(220, 0.4, 0.2, 0.1, "uniform", rng=32)
    a = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.01), 50, seed=1, gcw=False)
    b = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.01), 50, seed=1, gcw=False)
    np.testing.assert_array_equal(a["S_vec"], b["S_vec"])
    np.testing.assert_array_equal(a["w"], b["w"])
    np.testing.assert_array_equal(a["hist"], b["hist"])


def test_blocked_direct_load_path_still_matches_oracle(monkeypatch):
    """k_pgd_block + k_pgd_scatter (same shared-memory tables, direct loads, L2 gather) is the fallback for
    slot lists longer than the streamed kernel supports; force it and check parity"""
    monkeypatch.setenv("DESC_B200_PGD_PATH", "blocked")
    mo = O.uniform_topology(160, 0.5, 0.25, 0.1, "uniform", rng=33)
    for ns in (0, 70):
        c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.02), 40, n_sample=ns, seed=8)
        o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(0.02), 40, n_sample=ns or None, seed=8)
        assert_incidence_equal(c, o["inc"])
        assert_solution_close(c, o)


@pytest.mark.parametrize("ns", [0, 6, 12, 45, 100])
@pytest.mark.parametrize("rule", ["const", "adam"])
def test_streamed_path_slot_list_lengths_and_rules(monkeypatch, ns, rule):
    """the streamed kernels with slot lists of <= 32, <= 64 and <= 128 entries (4, 8 and 16 lanes per edge), constant
    step and Adam, against the oracle.  This graph has m < 100 n, so one GPU would take the blocked kernels unless
    the path is forced"""
    monkeypatch.setenv("DESC_B200_PGD_PATH", "stream")
    mo = O.uniform_topology(240, 0.65, 0.2, 0.1, "uniform", rng=34)
    if rule == "const":
        rc, ro = desc_b200.ConstantStepSize(0.05), O.ConstantStepSize(0.05)
    else:
        rc, ro = desc_b200.HybridGradient(0.002, 0.9, 0.999, 25), O.HybridGradient(0.002, 0.9, 0.999, 25)
    c = run_cuda(mo["Ind"], mo["RijMat"], rc, 20, n_sample=ns, seed=4, gcw=False)
    assert c["timings"]["pgd_pass2_ms"] > 0.0                 # the two-pass streamed path ran
    assert c["info"]["max_slots_per_edge"] > (32 if ns > 32 else 0)
    o = run_oracle(mo["Ind"], mo["RijMat"], ro, 20, n_sample=(None if ns == 0 else ns), seed=4, gcw=False)
    assert_incidence_equal(c, o["inc"])
    assert_solution_close(c, o)


def test_hybrid_gradient_rule_reuse_on_new_handle_is_rejected():
    """HybridGradient.m:24-27 zeroes the moments only at t == 0: a rule object that has already stepped cannot be
    continued on a handle that does not hold its moments (ADVICE r1); a fresh rule on the same handle works, and a
    second call with the advanced rule on the SAME handle continues the first"""
    mo = O.uniform_topology(120, 0.5, 0.2, 0.1, "uniform", rng=37)
    rule = desc_b200.HybridGradient(0.002, 0.9, 0.999, 25)
    orule = O.HybridGradient(0.002, 0.9, 0.999, 25)
    with desc_b200.Solver(mo["Ind"], mo["RijMat"]) as s:
        s.build_incidence(seed=2)
        s.cycle_inconsistency()
        s.pgd(6, rule)
        S_second, _, _ = s.pgd(4, rule)                  # same handle: the rule's t and moments continue, weights restart
        assert rule.t == 10
    inc = O.build_incidence(mo["Ind"], seed=2)
    S0 = O.cycle_inconsistency(inc, mo["RijMat"])
    two = O.HybridGradient(0.002, 0.9, 0.999, 25)
    O.pgd(inc, S0, 6, two)
    oS_second, _, _ = O.pgd(inc, S0, 4, two)
    assert rel_err(S_second, oS_second, floor=1e-12) <= RTOL
    with desc_b200.Solver(mo["Ind"], mo["RijMat"]) as s:
        s.build_incidence(seed=2)
        s.cycle_inconsistency()
        with pytest.raises(desc_b200.DescError) as e:
            s.pgd(10, rule)
        assert e.value.code == _lib.ERR_STATE
        fresh = desc_b200.HybridGradient(0.002, 0.9, 0.999, 25)
        S, _, _ = s.pgd(10, fresh)
    oS, _, _ = O.pgd(inc, S0, 10, orule)
    assert rel_err(S, oS, floor=1e-12) <= RTOL


def test_pgd_rejects_cycle_lists_with_repeated_apex():
    """explicit lists may repeat an apex (CEMP's with-replacement draw, CEMP.m:63); CEMP runs on them, DESC's PGD
    refuses (its kernels, like the reference's datasample without replacement, need distinct 3-cycles per edge)"""
    mo = O.uniform_topology(60, 0.5, 0.2, 0.1, "uniform", rng=38)
    inc = O.build_incidence(mo["Ind"], n_sample=8, seed=1)
    cnt = np.zeros(inc.m, dtype=np.int64)
    cnt[inc.pos_edges] = np.diff(inc.rowptr)
    ptr = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    apex = inc.k.astype(np.int32).copy()
    e = int(np.flatnonzero(cnt >= 2)[0])
    apex[ptr[e] + 1] = apex[ptr[e]]                                 # one repeated apex
    with desc_b200.Solver(mo["Ind"], mo["RijMat"]) as s:
        s.build_incidence(cycles=(ptr, apex))
        s.cycle_inconsistency()
        s.cemp(3, [1.0, 2.0, 4.0])                                  # legal for CEMP
        with pytest.raises(desc_b200.DescError) as err:
            s.pgd(3, desc_b200.ConstantStepSize(0.01))
        assert err.value.code == _lib.ERR_STATE
        s.build_incidence(cycles=(ptr, inc.k.astype(np.int32)))     # distinct again: accepted
        s.cycle_inconsistency()
        s.pgd(3, desc_b200.ConstantStepSize(0.01))


_ORACLE_CACHE = {}


def _cached_case(n, p, rng, lr, iters, ns, seed):
    key = (n, p, rng, lr, iters, ns, seed)
    if key not in _ORACLE_CACHE:
        mo = O.uniform_topology(n, p, 0.2, 0.1, "uniform", rng=rng)
        o = run_oracle(mo["Ind"], mo["RijMat"], O.ConstantStepSize(lr), iters, n_sample=(None if ns == 0 else ns),
                       seed=seed, gcw=False)
        _ORACLE_CACHE[key] = (mo, o)
    return _ORACLE_CACHE[key]


@pytest.mark.parametrize("path", ["stream"])
def test_slot_lists_up_to_256(monkeypatch, path):
    """all triangles of a dense graph (co-degrees above 128): the widest lanes-per-edge instantiations"""
    monkeypatch.setenv("DESC_B200_PGD_PATH", path)
    mo, o = _cached_case(380, 0.62, 36, 0.05, 6, -1, 4)
    c = run_cuda(mo["Ind"], mo["RijMat"], desc_b200.ConstantStepSize(0.05), 6, n_sample=-1, seed=4, gcw=False)
    assert 128 < c["info"]["max_slots_per_edge"] <= 256
    np.testing.assert_array_equal(c["apex"], o["inc"].k)          # (n_sample is reported differently for "all")
    np.testing.assert_array_equal(c["ikj"], o["inc"].IKJ >= 0)
    assert_solution_close(c, o)


@pytest.mark.parametrize("case", [(140, 0.5, 0.2, 0.1, 21), (120, 0.6, 0.3, 0.05, 22), (100, 0.5, 0.15, 0.0, 23)])
def test_laa_refinement_matches_oracle(case):
    """DESC step 5 (DESC.m:265-312): IRLS / weighted Lie-algebraic averaging on the device (CG on the
    grounded weighted Laplacian, radix-select quantile) against the oracle (sparse direct solve, sort)."""
    n, p, q, sigma, rng = case
    mo = O.uniform_topology(n, p, q, sigma, "uniform", rng=rng)
    oR_init, oS = O.DESC_init(mo["Ind"], mo["RijMat"], dict(iters=40, Gradient=O.ConstantStepSize(0.01)), seed=3)
    oR, info = O.laa_refine(mo["Ind"], mo["RijMat"], oS, oR_init, return_info=True)
    with desc_b200.Solver(mo["Ind"], mo["RijMat"]) as s:
        R, scores = s.refine(S_vec=oS, R_init=oR_init)      # same inputs as the oracle: isolates the stage
        t = s.timings()
    assert len(scores) == info["iterations"] and t["laa_iters"] == info["iterations"]
    np.testing.assert_allclose(scores, info["scores"], rtol=1e-8, atol=1e-12)
    assert O.aligned_angle_deg(R, oR).mean() <= ROT_TOL_DEG
    # the whole reference-style call
    params = dict(iters=40, Gradient=desc_b200.ConstantStepSize(0.01), seed=3)
    R_est, R_init, S_vec = desc_b200.DESC(mo["Ind"], mo["RijMat"], params)
    assert R_est.shape == (3, 3, n) and R_init.shape == (3, 3, n) and S_vec.shape == (1, mo["Ind"].shape[0])
    assert rel_err(S_vec.ravel(), oS, floor=1e-12) <= RTOL
    assert O.aligned_angle_deg(R_init, oR_init).mean() <= ROT_TOL_DEG
    assert O.aligned_angle_deg(R_est, oR).mean() <= 10 * ROT_TOL_DEG   # (R_init differs from the oracle's by its own 1e-6 deg)
