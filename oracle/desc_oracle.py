"""CPU oracle for the DESC solver hot path  --  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product package
(``desc_b200``) never imports anything from ``oracle/``.

PARITY UNPINNED: the reference (ColeWyeth/DESC, /root/reference) is 100 % MATLAB, ships
no tests / golden vectors / fixed seeds, and neither MATLAB nor Octave exists in this
image, so this restatement could not be checked against an execution of the reference.
It is pinned instead by (i) a second, literal loop-for-loop restatement
(``oracle/desc_literal.py``) that it must agree with, and (ii) analytic known-answer
properties of the algorithm (``tests/test_oracle.py``).

This file restates, with CSR data structures (same values as the reference's dense
n x n / n x m_pos arrays):

* ``Algorithms/DESC.m:14-263``  (== ``DESC_PGD.m:14-261``, ``DESC_init.m:14-253``)
* ``Utils/GCW.m:1-38``
* ``Utils/ConstantStepSize.m``, ``PiecewiseStepSize.m``, ``HybridGradient.m``
* ``Utils/Rotation_Alignment.m:13-38``
* ``Models/Uniform_Topology.m:24-111``, ``Models/Nonuniform_Topology.m:26-157``

Conventions: python arrays are 0-based; ``Ind`` at function boundaries is the
reference's m x 2, 1-based, i<j, sorted by (i, j) array; rotations are held as
``R[e, r, c]`` (shape (m,3,3)) inside the oracle and as MATLAB's 3x3xm at the boundary.

The one thing that cannot be restated is ``datasample(..., 'Replace', false)``
(``DESC.m:84``: Statistics Toolbox + MATLAB's global RNG stream).  It is replaced by a
counter-based sampler shared bit-for-bit with the CUDA build (``sampler_keys`` below):
an edge with codegree >= n_sample keeps the n_sample common neighbours with the smallest
64-bit key; kept apices are stored in ascending order (order only changes FP summation
order in the reference).  Explicit cycle lists can be supplied instead.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

# --------------------------------------------------------------------------------------
# MATLAB semantics helpers
# --------------------------------------------------------------------------------------


def matlab_median(x):
    """MATLAB ``median`` of a vector: mean of the two middle values when even (DESC.m:43)."""
    x = np.sort(np.asarray(x, dtype=np.float64).ravel())
    k = x.size
    if k == 0:
        return float("nan")
    if k % 2:
        return float(x[k // 2])
    return float((x[k // 2 - 1] + x[k // 2]) / 2.0)


def abs_acos(x):
    """``abs(acos(x))`` with MATLAB's complex branch for |x|>1 (DESC.m:147, SURVEY H2).

    x in [-1,1]: acos(x).  x>1: acos(x) = i*acosh(x), modulus acosh(x).
    x<-1: acos(x) = pi - i*acosh(-x), modulus sqrt(pi^2 + acosh(-x)^2).
    """
    x = np.asarray(x, dtype=np.float64)
    out = np.empty_like(x)
    mid = (x >= -1.0) & (x <= 1.0)
    out[mid] = np.arccos(x[mid])
    hi = x > 1.0
    if hi.any():
        t = x[hi] - 1.0  # exact (Sterbenz) for x close to 1
        out[hi] = np.log1p(t + np.sqrt(t * (t + 2.0)))
    lo = x < -1.0
    if lo.any():
        t = -x[lo] - 1.0
        a = np.log1p(t + np.sqrt(t * (t + 2.0)))
        out[lo] = np.sqrt(np.pi * np.pi + a * a)
    nan = np.isnan(x)
    out[nan] = np.nan
    return out


def proj_so3(Q):
    """``[U,~,V]=svd(Q); U*diag([1,1,det(U*V')])*V'`` batched (Uniform_Topology.m:41-44, GCW.m:32-34)."""
    Q = np.asarray(Q, dtype=np.float64)
    U, _, Vt = np.linalg.svd(Q)
    d = np.linalg.det(U @ Vt)
    U = U.copy()
    U[..., :, 2] *= d[..., None]
    return U @ Vt


def to_internal(RijMat):
    """MATLAB 3x3xm -> (m,3,3) with R[e,r,c]."""
    RijMat = np.asarray(RijMat, dtype=np.float64)
    assert RijMat.shape[:2] == (3, 3)
    return np.ascontiguousarray(RijMat.transpose(2, 0, 1))


def to_matlab(R):
    """(m,3,3) -> MATLAB 3x3xm (Fortran order, i.e. MATLAB's memory layout)."""
    return np.asfortranarray(np.asarray(R).transpose(1, 2, 0))


# --------------------------------------------------------------------------------------
# Synthetic models (input layout contract + fixture generator)
# --------------------------------------------------------------------------------------


def _er_graph(n, p, rng):
    """Uniform_Topology.m:29-35: G=tril(rand(n)<p,-1); [Ind_j,Ind_i]=find(G) (column-major)."""
    G = np.tril(rng.random((n, n)) < p, -1)
    cols, rows = np.nonzero(G.T)  # sorted by column then row == MATLAB find order
    Ind = np.stack([cols + 1, rows + 1], axis=1).astype(np.float64)  # [Ind_i, Ind_j], i<j
    AdjMat = (G | G.T).astype(np.float64)
    return AdjMat, Ind


def _rand_rot(k, rng):
    return proj_so3(rng.standard_normal((k, 3, 3)))


def _err_vec(Rij_orig, RijMat):
    """Uniform_Topology.m:94-101: trace(Rij_orig * RijMat') accumulated column by column."""
    acc = np.zeros((Rij_orig.shape[0], 3))
    for j in range(3):
        acc = acc + Rij_orig[:, :, j] * RijMat[:, :, j]
    tr = (acc[:, 0] + acc[:, 1]) + acc[:, 2]
    return abs_acos((tr - 1.0) / 2.0) / np.pi


def uniform_topology(n, p, q, sigma, model="uniform", rng=None):
    """Models/Uniform_Topology.m:24-111.  Returns a dict with the reference's field names."""
    rng = np.random.default_rng(rng)
    AdjMat, Ind = _er_graph(n, p, rng)
    ei = Ind[:, 0].astype(np.int64) - 1
    ej = Ind[:, 1].astype(np.int64) - 1
    m = ei.size
    R_orig = _rand_rot(n, rng)
    Rij_orig = R_orig[ei] @ R_orig[ej].transpose(0, 2, 1)
    RijMat = Rij_orig.copy()
    noise = rng.random(m) >= q
    corr = ~noise
    RijMat[noise] = RijMat[noise] + sigma * rng.standard_normal((int(noise.sum()), 3, 3))
    RijMat[noise] = proj_so3(RijMat[noise])
    R_corr = _rand_rot(n, rng)
    nc = int(corr.sum())
    if model == "uniform":
        RijMat[corr] = _rand_rot(nc, rng)
    else:
        Q = R_corr[ei[corr]] @ R_corr[ej[corr]].transpose(0, 2, 1) + sigma * rng.standard_normal((nc, 3, 3))
        RijMat[corr] = proj_so3(Q)
    ErrVec = _err_vec(Rij_orig, RijMat)
    return dict(AdjMat=AdjMat, Ind=Ind, RijMat=to_matlab(RijMat), Rij_orig=to_matlab(Rij_orig),
                R_orig=to_matlab(R_orig), ErrVec=ErrVec)


def nonuniform_topology(n, p, p_node_crpt, p_edge_crpt, sigma_in, sigma_out, crpt_type="uniform", rng=None):
    """Models/Nonuniform_Topology.m:26-157."""
    rng = np.random.default_rng(rng)
    AdjMat, Ind = _er_graph(n, p, rng)
    ei = Ind[:, 0].astype(np.int64) - 1
    ej = Ind[:, 1].astype(np.int64) - 1
    m = ei.size
    R_orig = _rand_rot(n, rng)
    Rij_orig = R_orig[ei] @ R_orig[ej].transpose(0, 2, 1)
    RijMat = Rij_orig.copy()
    # IndMat(i,j)=k, IndMat(j,i)=-k  (:57-58), 1-based k
    IndMat = {}
    for k in range(m):
        IndMat[(int(ei[k]), int(ej[k]))] = k + 1
        IndMat[(int(ej[k]), int(ei[k]))] = -(k + 1)
    node_crpt = rng.permutation(n)[: int(math.floor(n * p_node_crpt))]
    crpt = np.zeros(m, dtype=bool)
    R_crpt = _rand_rot(n, rng)
    # Ind_full = [Ind_j, Ind_i; Ind_i, Ind_j]  (:42)
    full_a = np.concatenate([ej, ei])
    full_b = np.concatenate([ei, ej])
    for i in node_crpt:
        cand = full_b[full_a == i]
        perm = rng.permutation(cand.size)
        nn = int(math.floor(p_edge_crpt * cand.size))
        for j in cand[perm[:nn]]:
            k = IndMat[(int(i), int(j))]
            crpt[abs(k) - 1] = True
            R0 = _rand_rot(1, rng)[0]
            if crpt_type == "uniform":
                M = R0
            elif crpt_type == "self-consistent":
                M = R_crpt[i] @ R_crpt[j].T
            elif crpt_type == "adv":
                M = R_crpt[i] @ R_orig[j].T
            else:
                raise ValueError(crpt_type)
            RijMat[abs(k) - 1] = M if k > 0 else M.T
    noise = ~crpt
    RijMat[noise] = RijMat[noise] + sigma_in * rng.standard_normal((int(noise.sum()), 3, 3))
    RijMat[crpt] = RijMat[crpt] + sigma_out * rng.standard_normal((int(crpt.sum()), 3, 3))
    RijMat = proj_so3(RijMat)
    ErrVec = _err_vec(Rij_orig, RijMat)
    return dict(AdjMat=AdjMat, Ind=Ind, RijMat=to_matlab(RijMat), Rij_orig=to_matlab(Rij_orig),
                R_orig=to_matlab(R_orig), ErrVec=ErrVec)


# --------------------------------------------------------------------------------------
# Step rules (Utils/ConstantStepSize.m, PiecewiseStepSize.m, HybridGradient.m)
# --------------------------------------------------------------------------------------


class ConstantStepSize:
    """Utils/ConstantStepSize.m:9-11."""

    def __init__(self, learning_rate):
        self.learning_rate = float(learning_rate)

    def GetStep(self, grad):
        return -self.learning_rate * grad


class PiecewiseStepSize:
    """Utils/PiecewiseStepSize.m:13-18 (``fix`` == truncation toward zero)."""

    def __init__(self, learning_rate, decay_interval):
        self.learning_rate = float(learning_rate)
        self.decay_interval = float(decay_interval)
        self.t = 0

    def GetStep(self, grad):
        self.t += 1
        step_size = self.learning_rate / (math.trunc(self.t / self.decay_interval) + 1)
        return -step_size * grad


class HybridGradient:
    """Utils/HybridGradient.m:23-52: Adam (strategy 0) or 100x decayed SGD (strategy 1)."""

    def __init__(self, lr, beta_1, beta_2, decay_interval):
        self.lr, self.beta_1, self.beta_2 = float(lr), float(beta_1), float(beta_2)
        self.decay_interval = float(decay_interval)
        self.t = 0
        self.strategy = 0
        self.m_t = None
        self.v_t = None

    def GetStep(self, grad):
        if self.t == 0:
            self.m_t = np.zeros_like(grad)
            self.v_t = np.zeros_like(grad)
        if self.strategy == 0:
            self.t += 1
            self.m_t = (self.beta_1 * self.m_t) + (1 - self.beta_1) * grad
            self.v_t = (self.beta_2 * self.v_t) + (1 - self.beta_2) * (grad ** 2)
            corr_m = self.m_t / (1 - self.beta_1 ** self.t)
            corr_v = self.v_t / (1 - self.beta_2 ** self.t)
            return -self.lr * corr_m / (np.sqrt(corr_v) + 1e-8)
        self.t += 1
        step_size = 100 * (self.lr / (math.trunc(self.t / self.decay_interval) + 1))
        return -step_size * grad

    def stopAdam(self):
        self.strategy = 1
        return self


# --------------------------------------------------------------------------------------
# Deterministic sampler shared with the CUDA build (replaces datasample, DESC.m:83-85)
# --------------------------------------------------------------------------------------

_M1 = np.uint64(0x9E3779B97F4A7C15)
_M2 = np.uint64(0xD1B54A32D192ED03)
_M3 = np.uint64(0xBF58476D1CE4E5B9)
_M4 = np.uint64(0x94D049BB133111EB)


def sampler_keys(seed, edge, k):
    """64-bit key of (edge id 0-based, apex 0-based).  Same arithmetic as csrc ``desc_key``."""
    with np.errstate(over="ignore"):
        edge = np.asarray(edge).astype(np.uint64)
        k = np.asarray(k).astype(np.uint64)
        z = np.uint64(seed) + _M1 * (edge + np.uint64(1))
        z = z ^ (_M2 * (k + np.uint64(1)))
        z = (z ^ (z >> np.uint64(30))) * _M3
        z = (z ^ (z >> np.uint64(27))) * _M4
        z = z ^ (z >> np.uint64(31))
    return z


# --------------------------------------------------------------------------------------
# A1-A4: graph, co-degree, sampling budget, incidence, reciprocal-slot maps
# --------------------------------------------------------------------------------------


@dataclass
class Incidence:
    n: int
    m: int
    ei: np.ndarray            # (m,) 0-based smaller endpoint
    ej: np.ndarray            # (m,) 0-based larger endpoint
    codeg: np.ndarray         # (m,) true co-degree of every edge (0 where the reference has -1)
    n_sample: int
    pos_edges: np.ndarray     # CoDeg_pos_ind (0-based edge ids), DESC.m:36
    rowptr: np.ndarray        # cum_ind, DESC.m:49 (length m_pos+1)
    e_ij: np.ndarray          # Ind_ij per slot (0-based edge id), DESC.m:86
    e_jk: np.ndarray          # Ind_jk, DESC.m:87
    e_ki: np.ndarray          # Ind_ki, DESC.m:88
    k: np.ndarray             # IJK (0-based apex), DESC.m:93
    IKJ: np.ndarray           # 0-based slot index of (ik; j), -1 where ~IKJ_appears, DESC.m:116
    JKI: np.ndarray           # 0-based slot index of (jk; i), -1 where ~JKI_appears, DESC.m:125
    extras: dict = field(default_factory=dict)

    @property
    def m_pos(self):
        return int(self.pos_edges.size)

    @property
    def m_cycle(self):
        return int(self.rowptr[-1])


def check_ind(Ind):
    """SURVEY H9: the reference silently needs i<j rows sorted by (i, j), no duplicates."""
    Ind = np.asarray(Ind)
    if Ind.ndim != 2 or Ind.shape[1] != 2:
        raise ValueError("Ind must be m x 2")
    ei = Ind[:, 0].astype(np.int64) - 1
    ej = Ind[:, 1].astype(np.int64) - 1
    if (ei < 0).any() or (ei >= ej).any():
        raise ValueError("Ind rows must satisfy 1 <= i < j")
    n = int(ej.max()) + 1 if ej.size else 0
    key = ei * n + ej
    if (np.diff(key) <= 0).any():
        raise ValueError("Ind rows must be strictly sorted by (i, j)")
    return n, ei, ej


def _candidates(n, ei, ej, chunk_cells=40_000_000):
    """All (edge, apex) pairs with apex a common neighbour: find(AdjMat(:,i).*AdjMat(:,j)), DESC.m:82."""
    m = ei.size
    A = np.zeros((n, n), dtype=bool)
    A[ei, ej] = True
    A[ej, ei] = True
    ce, ck = [], []
    step = max(1, chunk_cells // max(n, 1))
    for a in range(0, m, step):
        b = min(m, a + step)
        common = A[ei[a:b]] & A[ej[a:b]]
        r, c = np.nonzero(common)  # sorted by edge then apex (ascending k, like find)
        ce.append((r + a).astype(np.int64))
        ck.append(c.astype(np.int64))
    if ce:
        return np.concatenate(ce), np.concatenate(ck)
    return np.zeros(0, np.int64), np.zeros(0, np.int64)


def build_incidence(Ind, n_sample=None, seed=0, cycles=None):
    """DESC.m:19-127 with CSR storage.

    n_sample: None -> reference rule ``max(ceil(median(codeg_pos)/4),30)`` (DESC.m:43);
              an int -> that budget;  -1 -> keep every triangle.
    cycles:   optional explicit ``(ptr, apex)`` with ``ptr`` of length m+1 over ALL edges and
              0-based apices in the order to be used (what a MATLAB run's datasample produced).
    """
    n, ei, ej = check_ind(Ind)
    m = ei.size
    cand_e, cand_k = _candidates(n, ei, ej)
    codeg = np.bincount(cand_e, minlength=m).astype(np.int64)
    pos_mask = codeg > 0
    pos_edges = np.nonzero(pos_mask)[0]
    if n_sample is None:
        n_sample = max(int(math.ceil(matlab_median(codeg[pos_mask]) / 4.0)), 30) if pos_edges.size else 30
    elif n_sample < 0:
        n_sample = int(codeg.max()) + 1 if m else 1
    n_sample = int(n_sample)

    if cycles is None:
        keys = sampler_keys(seed, cand_e, cand_k)
        order = np.lexsort((cand_k, keys, cand_e))
        se = cand_e[order]
        start = np.concatenate([[0], np.cumsum(codeg)])[se]
        rank = np.arange(se.size) - start
        keep = order[rank < n_sample]
        keep.sort()  # back to (edge, ascending apex) order
        sl_e, sl_k = cand_e[keep], cand_k[keep]
    else:
        ptr, apex = cycles
        ptr = np.asarray(ptr, dtype=np.int64)
        apex = np.asarray(apex, dtype=np.int64)
        cnt = np.diff(ptr)
        sl_e = np.repeat(np.arange(m, dtype=np.int64), cnt)
        sl_k = apex
        # every listed apex must be a common neighbour, no duplicates
        ck = set(zip(cand_e.tolist(), cand_k.tolist()))
        lst = list(zip(sl_e.tolist(), sl_k.tolist()))
        if len(set(lst)) != len(lst) or not set(lst) <= ck:
            raise ValueError("explicit cycle list is not a duplicate-free subset of the triangles")
        if ((cnt > 0) != pos_mask).any():
            raise ValueError("explicit cycle list must be non-empty exactly for edges with triangles")

    ns_all = np.bincount(sl_e, minlength=m).astype(np.int64)
    rowptr = np.concatenate([[0], np.cumsum(ns_all[pos_edges])]).astype(np.int64)
    # IndMat (DESC.m:67-68) as a sorted-key lookup
    ekey = ei * n + ej

    def edge_id(a, b):
        lo, hi = np.minimum(a, b), np.maximum(a, b)
        idx = np.searchsorted(ekey, lo * n + hi)
        assert (ekey[idx] == lo * n + hi).all()
        return idx

    si, sj = ei[sl_e], ej[sl_e]
    e_jk = edge_id(sj, sl_k)
    e_ki = edge_id(sl_k, si)
    # reciprocal slots (DESC.m:98-127): slot of (edge, apex) by sorted key lookup
    skey = sl_e * n + sl_k
    sorder = np.argsort(skey, kind="stable")
    skey_sorted = skey[sorder]

    def slot_of(edge, apex):
        q = edge * n + apex
        pos = np.searchsorted(skey_sorted, q)
        pos = np.minimum(pos, max(skey_sorted.size - 1, 0))
        hit = skey_sorted[pos] == q if skey_sorted.size else np.zeros(q.shape, bool)
        return np.where(hit, sorder[pos], -1)

    IKJ = slot_of(e_ki, sj)
    JKI = slot_of(e_jk, si)
    return Incidence(n=n, m=m, ei=ei, ej=ej, codeg=codeg, n_sample=n_sample, pos_edges=pos_edges,
                     rowptr=rowptr, e_ij=sl_e, e_jk=e_jk, e_ki=e_ki, k=sl_k, IKJ=IKJ, JKI=JKI)


# --------------------------------------------------------------------------------------
# A5: cycle inconsistency d_ijk  (DESC.m:129-147), unfused, reference accumulation order
# --------------------------------------------------------------------------------------


def cycle_inconsistency(inc: Incidence, RijMat, chunk=2_000_000):
    R = to_internal(RijMat)
    S0 = np.empty(inc.m_cycle, dtype=np.float64)
    for a in range(0, inc.m_cycle, chunk):
        b = min(inc.m_cycle, a + chunk)
        i = inc.ei[inc.e_ij[a:b]]
        j = inc.ej[inc.e_ij[a:b]]
        k = inc.k[a:b]
        Rij = R[inc.e_ij[a:b]]
        Rjk = R[inc.e_jk[a:b]]
        Rjk = np.where((j < k)[:, None, None], Rjk, Rjk.transpose(0, 2, 1))  # RijMat4d(:,:,j,k), DESC.m:65-66
        Rki = R[inc.e_ki[a:b]]
        Rki = np.where((k < i)[:, None, None], Rki, Rki.transpose(0, 2, 1))  # RijMat4d(:,:,k,i)
        # R_cycle0 = sum_j Rij(:,j).*Rjk(j,:), accumulated j=1,2,3 from zero (DESC.m:137-139)
        C0 = np.zeros((b - a, 3, 3))
        for jj in range(3):
            C0 = C0 + Rij[:, :, jj, None] * Rjk[:, jj, None, :]
        # only the diagonal of R_cycle = sum_j R_cycle0(:,j).*Rki(j,:) is used (DESC.m:141-146)
        D = np.zeros((b - a, 3))
        for jj in range(3):
            D = D + C0[:, :, jj] * Rki[:, jj, :]
        tr = (D[:, 0] + D[:, 1]) + D[:, 2]
        S0[a:b] = abs_acos((tr - 1.0) / 2.0) / np.pi
    return S0


# --------------------------------------------------------------------------------------
# A6-A12: projected gradient descent  (DESC.m:148-261)
# --------------------------------------------------------------------------------------


def _project_simplex_rows(w, ptr, ns, seg):
    """DESC.m:213-224 for every edge at once: ascending sort, first Ti with
    sum(w(Ti:end)-w(Ti)) < 1, T = w(Ti) - (1 - that sum)/length(w(Ti:end)); max(w_new-T,0)."""
    m_pos = ns.size
    width = int(ns.max()) if m_pos else 0
    col = np.arange(w.size) - ptr[:-1][seg]
    pad = np.full((m_pos, width), np.inf)
    pad[seg, col] = w
    srt = np.sort(pad, axis=1)
    fin = np.isfinite(srt)
    vals = np.where(fin, srt, 0.0)
    suf = np.cumsum(vals[:, ::-1], axis=1)[:, ::-1]          # sum_{t>=i} w_t
    cnt = ns[:, None] - np.arange(width)[None, :]              # length(w(i:end))
    excess = suf - cnt * vals                                  # sum(w(i:end)-w(i))
    ok = fin & (excess < 1.0)
    Ti = np.argmax(ok, axis=1)
    r = np.arange(m_pos)
    T = vals[r, Ti] - (1.0 - excess[r, Ti]) / cnt[r, Ti]
    return np.maximum(w - T[seg], 0.0)


def pgd(inc: Incidence, S0, iters, rule, patience=30, tol=1e-5, verbose=False, return_w=False, S_hist=None):
    """DESC.m:148-261.  Returns (S_vec (m,), hist (iters_run,2)=[average_change, obj], iters_run).
    ``S_hist``: a list that receives a copy of S_vec after every iteration (make_plots diagnostics, :235-239)."""
    m = inc.m
    ptr = inc.rowptr
    ns = np.diff(ptr)
    m_pos = ns.size
    seg = np.repeat(np.arange(m_pos), ns)
    starts = ptr[:-1]
    S_vec = np.ones(m)
    hist = []
    if m_pos == 0:
        return (S_vec, np.zeros((0, 2)), 0) + ((np.zeros(0),) if return_w else ())

    def seg_sum(x):
        return np.add.reduceat(x, starts)

    wijk = 1.0 / ns[seg].astype(np.float64)                    # DESC.m:151-155
    S_vec[inc.pos_edges] = seg_sum(wijk * S0)                   # DESC.m:156
    appA = inc.IKJ >= 0
    appB = inc.JKI >= 0
    ikj = np.where(appA, inc.IKJ, 0)
    jki = np.where(appB, inc.JKI, 0)
    nv = 1.0 / np.sqrt(ns.astype(np.float64))
    S_last = S_vec.copy()
    misses = 0
    iters_run = 0
    for it in range(1, iters + 1):
        A = seg_sum(np.where(appA, wijk[ikj], 0.0))             # DESC.m:189
        B = seg_sum(np.where(appB, wijk[jki], 0.0))             # DESC.m:190
        sum_ikj = np.where(appA, A[seg], 0.0)
        sum_jki = np.where(appB, B[seg], 0.0)
        grad = S_vec[inc.e_jk] + S_vec[inc.e_ki] + (sum_ikj + sum_jki) * S0   # DESC.m:193
        dot = seg_sum(grad * nv[seg])                           # DESC.m:201
        grad = grad - dot[seg] * nv[seg]
        wijk = wijk + rule.GetStep(grad)                        # DESC.m:207
        wijk = _project_simplex_rows(wijk, ptr, ns, seg)        # DESC.m:208-224
        S_vec[inc.pos_edges] = seg_sum(wijk * S0)               # DESC.m:229
        average_change = float(np.mean(np.abs(S_vec - S_last)))  # DESC.m:232
        obj = float(np.dot(wijk, S_vec[inc.e_jk] + S_vec[inc.e_ki]))  # DESC.m:233
        hist.append((average_change, obj))
        if S_hist is not None:
            S_hist.append(S_vec.copy())
        iters_run = it
        if verbose:
            print("iter %d: average change in S_vec %f, objective value: %f" % (it, average_change, obj))
        if it > 1 and hist[-2][1] - hist[-1][1] < tol:          # DESC.m:243-256
            misses += 1
            if misses >= patience:
                break
        else:
            misses = 0
        S_last = S_vec.copy()
    out = (S_vec, np.array(hist).reshape(-1, 2), iters_run)
    if return_w:
        out = out + (wijk,)
    return out


# --------------------------------------------------------------------------------------
# A13: GCW  (Utils/GCW.m:1-38)
# --------------------------------------------------------------------------------------


def gcw(Ind, RijMat, S_vec, dense_limit=400, power=1.5, return_eigs=False):
    """Top-3 eigenvectors ('la') of D^-1 (W o R), computed through the similar symmetric matrix
    D^-1/2 (W o R) D^-1/2 (SURVEY H4), unit 2-norm columns, sign rule GCW.m:28, SVD projection :30-36.
    ``power=1.5``: GCW.m:20;  ``power=1``: the weights of CEMP_GCW.m:141, ``1./(S+1e-8)`` (the rest of
    CEMP_GCW.m:127-159 is GCW.m line for line).  ``return_eigs``: also return the largest eigenvalues of the
    symmetric matrix in descending order (four with the dense solve, three with the sparse one)."""
    n, ei, ej = check_ind(Ind)
    R = to_internal(RijMat)
    S_vec = np.asarray(S_vec, dtype=np.float64).ravel()
    if power is None:                                            # Spectral.m:36-40: unweighted, un-normalised
        om = np.ones(ei.size)
        isd = np.ones(n)
    else:
        om = 1.0 / ((S_vec ** 1.5 if power == 1.5 else S_vec) + 1e-8)   # GCW.m:20 / CEMP_GCW.m:141
        d = np.bincount(ei, om, n) + np.bincount(ej, om, n)      # sum(Weights,2), GCW.m:21
        isd = 1.0 / np.sqrt(d)
    c = (om * isd[ei] * isd[ej])[:, None, None]
    blk = c * R
    if n <= dense_limit:
        N = np.zeros((n, 3, n, 3))
        N[ei, :, ej, :] = blk
        N[ej, :, ei, :] = blk.transpose(0, 2, 1)
        N = N.reshape(3 * n, 3 * n)
        lam, U = np.linalg.eigh(N)
        lam = lam[::-1][:4]
        U = U[:, ::-1][:, :3]
    else:
        import scipy.sparse as sp
        from scipy.sparse.linalg import eigsh
        r = (3 * ei[:, None, None] + np.arange(3)[None, :, None]) + np.zeros((1, 1, 3), np.int64)
        cidx = (3 * ej[:, None, None] + np.arange(3)[None, None, :]) + np.zeros((1, 3, 1), np.int64)
        Msp = sp.coo_matrix((blk.ravel(), (r.ravel(), cidx.ravel())), shape=(3 * n, 3 * n)).tocsr()
        Msp = Msp + Msp.T
        lam, U = eigsh(Msp, k=3, which="LA", tol=1e-14)
        U = U[:, np.argsort(-lam)]
        lam = np.sort(lam)[::-1]
    V = U * np.repeat(isd, 3)[:, None]
    V = V / np.linalg.norm(V, axis=0, keepdims=True)
    if np.linalg.det(V[:3, :]) < 0:                              # GCW.m:28
        V[:, 0] = -V[:, 0]
    R_est = to_matlab(proj_so3(V.reshape(n, 3, 3)))              # GCW.m:30-36
    return (R_est, lam) if return_eigs else R_est


# --------------------------------------------------------------------------------------
# Metric: Utils/Rotation_Alignment.m:13-38
# --------------------------------------------------------------------------------------


def rotation_alignment(R_est, R_gt):
    Re, Rg = to_internal(R_est), to_internal(R_gt)
    A = np.einsum("kab,kac->bc", Re, Rg)                         # sum U'*V, :17-21
    U1, _, V1t = np.linalg.svd(A)
    R_align = U1 @ np.diag([1.0, 1.0, np.linalg.det(U1 @ V1t)]) @ V1t
    R_out = Re @ R_align
    tr = np.einsum("kab,kab->k", Rg, R_out)                      # trace(R_gt*R_out')
    MSEVec = abs_acos((tr - 1.0) / 2.0) / np.pi * 180.0
    return to_matlab(R_out), R_align, float(np.mean(MSEVec)), matlab_median(MSEVec)


def aligned_angle_deg(R_a, R_b):
    """Well-conditioned per-node angle (deg) between two rotation sets after gauge alignment
    (SURVEY H4): 2*asin(||Ra*Q - Rb||_F / (2*sqrt(2)))."""
    R_out, _, _, _ = rotation_alignment(R_a, R_b)
    D = to_internal(R_out) - to_internal(R_b)
    f = np.sqrt((D ** 2).sum(axis=(1, 2)))
    return np.degrees(2.0 * np.arcsin(np.minimum(f / (2.0 * math.sqrt(2.0)), 1.0)))


# --------------------------------------------------------------------------------------
# Entry points with the reference's signatures
# --------------------------------------------------------------------------------------


def DESC_PGD(Ind, RijMat, params, n_sample=None, seed=0, cycles=None, full=False):
    """Algorithms/DESC_PGD.m:14.  params: dict with 'iters', 'Gradient' (step-rule object)."""
    inc = build_incidence(Ind, n_sample=n_sample, seed=seed, cycles=cycles)
    S0 = cycle_inconsistency(inc, RijMat)
    S_vec, hist, iters_run, w = pgd(inc, S0, int(params["iters"]), params["Gradient"],
                                    verbose=bool(params.get("verbose", False)), return_w=True)
    if full:
        return dict(S_vec=S_vec, hist=hist, iters_run=iters_run, w=w, S0=S0, inc=inc)
    return S_vec


def DESC_init(Ind, RijMat, params, **kw):
    """Algorithms/DESC_init.m:14.  Returns (R_est, S_vec)."""
    S_vec = DESC_PGD(Ind, RijMat, params, **kw)
    return gcw(Ind, RijMat, S_vec), S_vec


# --------------------------------------------------------------------------------------------
# DESC step 5: weighted Lie-algebraic averaging refinement (Algorithms/DESC.m:265-312)
# --------------------------------------------------------------------------------------------
def matlab_quantile(x, p):
    """MATLAB ``quantile(x, p)`` for a vector: sample quantiles at (k-0.5)/n, linear interpolation,
    clamped to the extremes (used at DESC.m:276,301)."""
    xs = np.sort(np.asarray(x, dtype=np.float64).ravel())
    n = xs.size
    pos = n * p + 0.5                      # 1-based fractional position
    if pos <= 1.0:
        return float(xs[0])
    if pos >= n:
        return float(xs[-1])
    lo = int(math.floor(pos))
    frac = pos - lo
    return float(xs[lo - 1] + frac * (xs[lo] - xs[lo - 1]))


def R2Q(Rot):
    """Utils/R2Q.m:7-13.  Rot: (3,3,K) MATLAB layout -> (K,4) quaternions [cos(t/2), sin(t/2) axis]."""
    q0 = (Rot[0, 0, :] + Rot[1, 1, :] + Rot[2, 2, :] - 1.0) / 2.0
    qv = np.stack([Rot[2, 1, :] - Rot[1, 2, :], Rot[0, 2, :] - Rot[2, 0, :], Rot[1, 0, :] - Rot[0, 1, :]], axis=1) / 2.0
    q0 = np.sqrt((q0 + 1.0) / 2.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        qv = (qv / q0[:, None]) / 2.0
    return np.concatenate([q0[:, None], qv], axis=1)


def q2R(q):
    """Utils/q2R.m:1-24 for one quaternion -> 3x3 (identity when abs(abs(q0)-1) <= 1e-12)."""
    c2 = q[0]
    if abs(abs(c2) - 1.0) > 1e-12:
        s2 = math.sqrt(q[1] * q[1] + q[2] * q[2] + q[3] * q[3])
        s = 2.0 * s2 * c2
        c = 2.0 * c2 * c2 - 1.0
        n1, n2, n3 = q[1] / s2, q[2] / s2, q[3] / s2
        cc = 1.0 - c
        n12, n23, n31 = n1 * n2 * cc, n2 * n3 * cc, n3 * n1 * cc
        return np.array([[c + n1 * n1 * cc, n12 - n3 * s, n31 + n2 * s],
                         [n12 + n3 * s, c + n2 * n2 * cc, n23 - n1 * s],
                         [n31 - n2 * s, n23 + n1 * s, c + n3 * n3 * cc]])
    return np.eye(3)


def _qmul_lines(a0, av, b0, bv):
    """the quaternion product pattern of Weighted_LAA.m:12-14,48-50: (a0 b0 - av.bv, a0 bv + b0 av + av x bv)
    written as the reference writes it (``[a0.*b0 - sum(av.*bv), a0.*bv + b0.*av + cross]`` with
    cross = [av2 bv3 - av3 bv2, av3 bv1 - av1 bv3, av1 bv2 - av2 bv1])."""
    s = a0 * b0 - np.sum(av * bv, axis=1)
    cr = np.stack([av[:, 1] * bv[:, 2] - av[:, 2] * bv[:, 1], av[:, 2] * bv[:, 0] - av[:, 0] * bv[:, 2],
                   av[:, 0] * bv[:, 1] - av[:, 1] * bv[:, 0]], axis=1)
    return s, a0[:, None] * bv + b0[:, None] * av + cr


def build_amatrix(ei, ej, n):
    """Utils/Build_Amatrix.m:6-14: m x (n-1) signed incidence, node 1 grounded: -1 at i, +1 at j."""
    import scipy.sparse as sp
    m = ei.size
    rows = np.concatenate([np.arange(m), np.arange(m)])
    cols = np.concatenate([ei, ej]) - 1              # 0-based node -> column (node 0 dropped)
    vals = np.concatenate([-np.ones(m), np.ones(m)])
    keep = cols >= 0
    return sp.csr_matrix((vals[keep], (rows[keep], cols[keep])), shape=(m, n - 1))


def weighted_laa(ei, ej, Q, QQ, A, Weights):
    """Utils/Weighted_LAA.m:4-52.  One weighted Lie-algebraic averaging step.
    Returns (Q_new, W, B, score) exactly as the reference does (W is the QUATERNION of the update,
    which is what DESC.m:290 multiplies with the A matrix)."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    N = Q.shape[0]
    # w = Qij * Qi   (:12-14)
    s, v = _qmul_lines(QQ[:, 0], QQ[:, 1:4], Q[ei, 0], Q[ei, 1:4])
    # w = inv(Qj) * w  (:17-19): scalar -Qj0 w0 - Qjv.wv ; vector -Qj0 wv + w0 Qjv + Qjv x wv
    Qj0, Qjv = Q[ej, 0], Q[ej, 1:4]
    s2_ = -Qj0 * s - np.sum(Qjv * v, axis=1)
    cr = np.stack([Qjv[:, 1] * v[:, 2] - Qjv[:, 2] * v[:, 1], Qjv[:, 2] * v[:, 0] - Qjv[:, 0] * v[:, 2],
                   Qjv[:, 0] * v[:, 1] - Qjv[:, 1] * v[:, 0]], axis=1)
    v2 = (-Qj0)[:, None] * v + s[:, None] * Qjv + cr
    s2 = np.sqrt(np.sum(v2 * v2, axis=1))                      # (:22)
    th = 2.0 * np.arctan2(s2, s2_)                             # (:23)
    th = np.where(th < -math.pi, th + 2 * math.pi, th)         # (:24)
    th = np.where(th >= math.pi, th - 2 * math.pi, th)
    with np.errstate(divide="ignore", invalid="ignore"):
        B = v2 * (th / s2)[:, None]                            # (:25)
    B[np.isnan(B)] = 0.0                                       # (:36)
    # weighted least squares (diag(W) A) \ (W .* B)  (:40), via the normal equations (unique solution)
    WA = sp.diags(Weights) @ A
    lhs = (WA.T @ WA).tocsc()
    rhs = WA.T @ (Weights[:, None] * B)
    X = spla.splu(lhs).solve(rhs)
    W = np.zeros((N, 4))
    W[0, :] = [1.0, 0.0, 0.0, 0.0]                             # (:38)
    W[1:, 1:4] = X
    score = float(np.sum(np.sqrt(np.sum(W[1:, 1:4] ** 2, axis=1))) / N)   # (:42)
    theta = np.sqrt(np.sum(W[:, 1:4] ** 2, axis=1))            # (:44)
    W[:, 0] = np.cos(theta / 2.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        W[:, 1:4] = W[:, 1:4] * (np.sin(theta / 2.0) / theta)[:, None]
    W[np.isnan(W)] = 0.0                                       # (:48)
    s3, v3 = _qmul_lines(Q[:, 0], Q[:, 1:4], W[:, 0], W[:, 1:4])   # Q = Q * W (:50-52)
    return np.concatenate([s3[:, None], v3], axis=1), W, B, score


def laa_refine(Ind, RijMat, S_vec, R_init, stop_threshold=1e-3, max_iters=100, quant_ratio_min=0.8,
               weight_max=1e4, weight_min=1e-4, return_info=False):
    """Algorithms/DESC.m:265-312: IRLS with weighted Lie-algebraic averaging, starting from R_init."""
    n, ei, ej = check_ind(Ind)
    S = np.asarray(S_vec, dtype=np.float64).ravel()
    RR = np.transpose(np.asarray(RijMat, dtype=np.float64), (1, 0, 2))       # (:265)
    A = build_amatrix(ei, ej, n)                                              # (:269)
    Q = R2Q(np.asarray(R_init, dtype=np.float64))                             # (:270)
    QQ = R2Q(RR)                                                              # (:271)
    score, it = math.inf, 1
    quant_ratio = 1.0
    thresh = matlab_quantile(S, quant_ratio)                                  # (:276)
    with np.errstate(divide="ignore"):
        Weights = 1.0 / S ** 0.75                                             # (:278)
    Weights[Weights > weight_max] = weight_max
    Weights[S > thresh] = weight_min
    scores = []
    RSVec = S.copy()
    while score > stop_threshold and it < max_iters:                         # (:287)
        lam = 1.0 / (it + 1)
        Q, W, B, score = weighted_laa(ei, ej, Q, QQ, A, Weights)
        E = A @ W[1:, 1:4] - B                                                # (:290)
        ResVec = np.sqrt(np.sum(E * E, axis=1)) / math.pi
        RSVec = (1.0 - lam) * ResVec + lam * S
        with np.errstate(divide="ignore"):
            Weights = 1.0 / RSVec ** 0.75                                     # (:298)
        quant_ratio = max(quant_ratio_min, quant_ratio - 0.05)
        thresh = matlab_quantile(RSVec, quant_ratio)                          # (:301)
        Weights[Weights > weight_max] = weight_max
        Weights[RSVec > thresh] = weight_min
        scores.append(score)
        it += 1
    R_est = np.zeros((3, 3, n))
    for i in range(n):
        R_est[:, :, i] = q2R(Q[i])                                            # (:309-312)
    if return_info:
        return R_est, dict(scores=np.array(scores), iterations=it - 1, RSVec=RSVec, Weights=Weights, thresh=thresh)
    return R_est


def DESC(Ind, RijMat, params, **kw):
    """Algorithms/DESC.m:14.  Returns (R_est, R_init, S_vec)."""
    R_init, S_vec = DESC_init(Ind, RijMat, params, **kw)
    return laa_refine(Ind, RijMat, S_vec, R_init), R_init, S_vec


# --------------------------------------------------------------------------------------------
# SURVEY 8(f) #3: CEMP / CEMP+GCW on the same incidence (Algorithms/CEMP.m, CEMP_GCW.m)
# --------------------------------------------------------------------------------------------
def spectral(Ind, RijMat):
    """``R_est = Spectral(Ind, RijMat)`` (Algorithms/Spectral.m:15-47): GCW.m's pipeline on the plain block matrix."""
    return gcw(Ind, RijMat, np.ones(np.asarray(Ind).shape[0]), power=None)


def cemp_incidence(Ind, nsample=50, seed=0, cycles=None):
    """Cycle lists for CEMP as an ``Incidence`` (IKJ/JKI unused, left empty).

    CEMP.m:63 draws ``datasample(find(...), nsample)`` -- WITH replacement, so every edge with a
    triangle gets exactly ``nsample`` slots and an apex may repeat.  MATLAB's RNG stream cannot be
    restated; as for DESC (module header) the stand-in is the shared counter-based sampler
    (``nsample`` smallest keys, no repeats, at most co-degree slots), or explicit ``(ptr, apex)`` lists
    over ALL edges, which MAY contain repeated apices (e.g. the CoIndMat a MATLAB run drew)."""
    if cycles is None:
        return build_incidence(Ind, n_sample=int(nsample), seed=seed)
    n, ei, ej = check_ind(Ind)
    m = ei.size
    ptr = np.asarray(cycles[0], dtype=np.int64)
    apex = np.asarray(cycles[1], dtype=np.int64)
    cnt = np.diff(ptr)
    sl_e = np.repeat(np.arange(m, dtype=np.int64), cnt)
    ekey = ei * n + ej

    def edge_id(a, b):
        lo, hi = np.minimum(a, b), np.maximum(a, b)
        idx = np.searchsorted(ekey, lo * n + hi)
        if not (idx < m).all() or not (ekey[np.minimum(idx, m - 1)] == lo * n + hi).all():
            raise ValueError("explicit cycle list contains an apex that is not a common neighbour")
        return idx

    e_jk = edge_id(ej[sl_e], apex)
    e_ki = edge_id(apex, ei[sl_e])
    pos_edges = np.nonzero(cnt > 0)[0]
    rowptr = np.concatenate([[0], np.cumsum(cnt[pos_edges])]).astype(np.int64)
    none = np.zeros(0, np.int64)
    return Incidence(n=n, m=m, ei=ei, ej=ej, codeg=cnt.copy(), n_sample=int(cnt.max()) if m else 0,
                     pos_edges=pos_edges, rowptr=rowptr, e_ij=sl_e, e_jk=e_jk, e_ki=e_ki, k=apex, IKJ=none, JKI=none)


def cemp_betas(max_iter, reweighting):
    """CEMP.m:26-34: a short reweighting vector is padded with its last element."""
    beta = [float(b) for b in np.asarray(reweighting, dtype=np.float64).ravel()]
    T = int(max_iter)
    if len(beta) < T:
        beta = beta + [beta[-1]] * (T - len(beta))
    return beta[:T]


def cemp_reweight(inc: Incidence, S0, SVec, beta, empty_value=1.0):
    """One CEMP reweighting (CEMP.m:109-125): per edge, ``sum_s w_s/sum(w) * S0_s`` with
    ``w_s = exp(-beta*(SVec(e_ki)+SVec(e_jk)))``; edges without cycles get ``empty_value`` (:125)."""
    seg = inc.rowptr[:-1]
    Smax = SVec[inc.e_ki] + SVec[inc.e_jk]                                   # Ski+Sjk, :117
    W = np.exp(-beta * Smax)                                                  # :119
    out = np.full(inc.m, empty_value, dtype=np.float64)
    if inc.m_pos:
        wsum = np.add.reduceat(W, seg)                                        # :120
        Wn = W / np.repeat(wsum, np.diff(inc.rowptr))                         # :122
        out[inc.pos_edges] = np.add.reduceat(Wn * S0, seg)                    # :123-125
    return out


def cemp(inc: Incidence, S0, max_iter, reweighting, return_hist=False):
    """Algorithms/CEMP.m:98-129 on CSR slot lists.  Returns SVec (length m)."""
    SVec = np.ones(inc.m, dtype=np.float64)
    if inc.m_pos:
        SVec[inc.pos_edges] = np.add.reduceat(S0, inc.rowptr[:-1]) / np.diff(inc.rowptr)   # mean(S0Mat,1), :99
    hist = [SVec.copy()]
    for beta in cemp_betas(max_iter, reweighting):
        SVec = cemp_reweight(inc, S0, SVec, beta)
        hist.append(SVec.copy())
    return (SVec, hist) if return_hist else SVec


def CEMP(Ind, RijMat, CEMP_parameters, seed=0, cycles=None):
    """``SVec = CEMP(Ind, RijMat, CEMP_parameters)`` (Algorithms/CEMP.m:25)."""
    inc = cemp_incidence(Ind, CEMP_parameters["nsample"], seed=seed, cycles=cycles)
    S0 = cycle_inconsistency(inc, RijMat)
    return cemp(inc, S0, CEMP_parameters["max_iter"], CEMP_parameters["reweighting"])


def CEMP_GCW(Ind, RijMat, CEMP_parameters, seed=0, cycles=None):
    """``R_est = CEMP_GCW(Ind, RijMat, CEMP_parameters)`` (Algorithms/CEMP_GCW.m:25)."""
    return gcw(Ind, RijMat, CEMP(Ind, RijMat, CEMP_parameters, seed=seed, cycles=cycles), power=1.0)


# --------------------------------------------------------------------------------------------
# SURVEY 8(f) #4: the make_plots diagnostics of DESC.m:235-239 (per-iteration S_vec error + GCW + alignment)
# --------------------------------------------------------------------------------------------
def pgd_diagnostics(Ind, RijMat, S_hist, ErrVec, R_orig):
    """For every iteration's S_vec: ``mean(abs(ErrVec - S_vec))`` (DESC.m:236), ``GCW`` (:237) and the
    mean / median alignment error in degrees (:238, Utils/GlobalSOdCorrectRight.m == Rotation_Alignment.m)."""
    ErrVec = np.asarray(ErrVec, dtype=np.float64).ravel()
    out = np.zeros((len(S_hist), 3))
    for t, S in enumerate(S_hist):
        R = gcw(Ind, RijMat, S)
        _, _, mean_err, med_err = rotation_alignment(R, R_orig)
        out[t] = [float(np.mean(np.abs(ErrVec - S))), mean_err, med_err]
    return out


# --------------------------------------------------------------------------------------------
# SURVEY 8(f) #3: MPLS on the same incidence (Algorithms/MPLS.m)
# --------------------------------------------------------------------------------------------
def _pad(v, length):
    """MPLS.m:43-63: a short parameter vector is padded with its last element."""
    v = [float(x) for x in np.asarray(v, dtype=np.float64).ravel()]
    return v + [v[-1]] * max(0, length - len(v))


def mst_init(Ind, RijMat, SVec):
    """MPLS.m:152-195: minimum spanning tree of the graph weighted by SVec+1, then R_i by multiplying Rij along
    the tree from node 1 (R_1 = I).  ``minspantree``'s tie-breaking is not documented; here (and on the device) ties
    are broken by the edge index, i.e. the tree is the unique MST under the total order (weight, edge id)."""
    n, ei, ej = check_ind(Ind)
    R = to_internal(RijMat)
    w = np.asarray(SVec, dtype=np.float64).ravel() + 1.0                          # :154
    order = np.lexsort((np.arange(ei.size), w))                                   # Kruskal on (weight, edge id)
    parent = np.arange(n)

    def find(a):
        while parent[a] != a:
            parent[a] = parent[parent[a]]
            a = parent[a]
        return a

    tree = []
    for e in order:
        a, b = find(int(ei[e])), find(int(ej[e]))
        if a != b:
            parent[a] = b
            tree.append(int(e))
            if len(tree) == n - 1:
                break
    if len(tree) != n - 1:
        raise ValueError("graph is not connected (the reference's loop MPLS.m:171 would not terminate)")
    nbr = [[] for _ in range(n)]
    for e in tree:
        nbr[int(ei[e])].append((int(ej[e]), e))
        nbr[int(ej[e])].append((int(ei[e]), e))
    R_est = np.zeros((n, 3, 3))
    R_est[0] = np.eye(3)                                                          # :165-167
    added = np.zeros(n, bool)
    added[0] = True
    roots = [0]
    while roots:                                                                  # :171-186
        new = []
        for r in roots:
            for leaf, e in nbr[r]:
                if added[leaf]:
                    continue
                # edge_leaf = IndMat(leaf, root) > 0 <=> leaf < root: R_leaf = Rij * R_root, else Rij' * R_root
                R_est[leaf] = (R[e] if leaf < r else R[e].T) @ R_est[r]
                added[leaf] = True
                new.append(leaf)
        roots = new
    return to_matlab(R_est), np.array(sorted(tree), dtype=np.int64)


def mpls_refine(Ind, RijMat, inc: Incidence, S0, SVec, R_init, MPLS_parameters, weight_max=1e4, weight_min=1e-4,
                return_info=False):
    """MPLS.m:198-256: the reweighting loop (Weighted_LAA + cycle reweighting of the residuals)."""
    n, ei, ej = check_ind(Ind)
    stop_threshold = float(MPLS_parameters["stop_threshold"])
    maxIters = int(MPLS_parameters["max_iter"])
    beta = _pad(MPLS_parameters["reweighting"], maxIters)                         # :43-47
    tau = _pad(MPLS_parameters["thresholding"], maxIters)                         # :49-53
    alpha = _pad(MPLS_parameters["cycle_info_ratio"], maxIters)                   # :55-59
    S = np.asarray(SVec, dtype=np.float64).ravel()
    RR = np.transpose(np.asarray(RijMat, dtype=np.float64), (1, 0, 2))            # :201
    A = build_amatrix(ei, ej, n)
    Q = R2Q(np.asarray(R_init, dtype=np.float64))
    QQ = R2Q(RR)
    score, it = math.inf, 1
    with np.errstate(divide="ignore"):
        Weights = 1.0 / S ** 0.75                                                 # :211
    Weights[Weights > weight_max] = weight_max                                    # :214
    # S0Mat columns of edges without a cycle are acos(-1/2)/pi (R_cycle = 0, MPLS.m:125-135): HVec = 2/3 there
    empty = float(np.arccos(-0.5) / np.pi)
    scores = []
    while score > stop_threshold and it < maxIters:                              # :219
        Q, W, B, score = weighted_laa(ei, ej, Q, QQ, A, Weights)
        E = A @ W[1:, 1:4] - B                                                    # :222
        ResVec = np.sqrt(np.sum(E * E, axis=1)) / math.pi
        HVec = cemp_reweight(inc, S0, ResVec, beta[it - 1], empty_value=empty)    # :224-238
        RHVec = (1.0 - alpha[it - 1]) * ResVec + alpha[it - 1] * HVec             # :241
        with np.errstate(divide="ignore"):
            Weights = 1.0 / RHVec ** 0.75                                         # :242
        thresh = matlab_quantile(RHVec, tau[it - 1])                              # :244
        Weights[Weights > weight_max] = weight_max
        Weights[RHVec > thresh] = weight_min
        scores.append(score)
        it += 1
    R_est = np.zeros((3, 3, n))
    for i in range(n):
        R_est[:, :, i] = q2R(Q[i])
    if return_info:
        return R_est, dict(scores=np.array(scores), iterations=it - 1)
    return R_est


def MPLS(Ind, RijMat, CEMP_parameters, MPLS_parameters, seed=0, cycles=None, return_info=False):
    """``[R_est, R_init] = MPLS(Ind, RijMat, CEMP_parameters, MPLS_parameters)`` (Algorithms/MPLS.m:28)."""
    inc = cemp_incidence(Ind, CEMP_parameters["nsample"], seed=seed, cycles=cycles)
    S0 = cycle_inconsistency(inc, RijMat)
    SVec = cemp(inc, S0, CEMP_parameters["max_iter"], CEMP_parameters["reweighting"])
    R_init, tree = mst_init(Ind, RijMat, SVec)
    R_est, info = mpls_refine(Ind, RijMat, inc, S0, SVec, R_init, MPLS_parameters, return_info=True)
    if return_info:
        info.update(SVec=SVec, tree=tree)
        return R_est, R_init, info
    return R_est, R_init
