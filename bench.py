#!/usr/bin/env python
"""bench.py -- DESC solve throughput on B200 (metric of BASELINE.json), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg4|cfg2|cfg3|cfg3sc|cfg5]
                    [--dump-outputs DIR]

A "step" is one complete DESC_init-equivalent solve (DESC.m:14-263 + GCW.m) of the workload:
CSR incidence build + cycle inconsistencies + PGD (iterations actually run) + GCW recovery.
Default workload = configs[3] of BASELINE.json (the configuration the metric is quoted on; it fits one GPU):
Uniform_Topology(n=10000, p=0.1, q=0.2, sigma=0.1, 'uniform'), params = {iters=100, Gradient=ConstantStepSize(0.01)}
(Demo/compare_algorithms.m:39-45), reference sampling rule.  Inputs are drawn by the library's own device generators
(csrc/gen.cu, counter-based: every rank draws the identical graph, nothing is broadcast).

value  = 3-cycle evaluations per second over the whole step = m_cycle * iters_run / step time,
         inputs (Ind, RijMat) already resident in HBM; N>1 shards the same problem ("strong").
e2e    = the same through the reference-style call with HOST (pinned) buffers: H2D of Ind/RijMat
         and D2H of S_vec / R_est / history inside the timed region.
roofline = one PGD iteration (its two kernels): algorithmic bytes (40*m_cycle + 12*m_pos + 8*m, SURVEY 8d) / mean
         duration of the pair (CUDA events on the launching stream around each kernel) vs the measured HBM peak.
         `traffic` = DRAM bytes of the pair from the committed ncu capture (profiles/r02_pgd_traffic.json), used only
         when the sha1 of the kernel sources it was captured on equals the current sources (else null + reason).
         `stages` = the same arithmetic for the one-off kernels (incidence build, d_ijk, one GCW SpMV).
cpu_baseline / --impl reference = the C/OpenMP restatement of the reference (oracle/desc_full.c + desc_pgd.c, every
         stage threaded, thread count = the cores this process may run on, set explicitly) on a graph of the
         workload's own family and co-degree regime: the workload's graph itself when the time budget allows,
         otherwise the largest smaller member of the family that fits; its true n / m / m_cycle are in the line.
         All stages run at that size; the PGD loop is timed over k iterations and the whole-solve time is
         fixed stages + iters * per-iteration time (every iteration does the same arithmetic), stated in `sample`.
parity = (N > 1) the N-rank result against a 1-rank solve of the same inputs on rank 0: max |dS_vec|, iters_run,
         mean rotation angle after gauge alignment.
"""
import argparse
import hashlib
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg4": dict(kind="uniform", n=10000, p=0.1, q=0.2, sigma=0.1, model="uniform", iters=100, lr=0.01, n_sample=0,
                 name="Uniform_Topology n=10000 p=0.1 q=0.2 sigma=0.1 uniform, iters=100 ConstantStepSize(0.01)"),
    "cfg2": dict(kind="uniform", n=1000, p=0.5, q=0.3, sigma=0.1, model="uniform", iters=100, lr=0.01, n_sample=0,
                 name="Uniform_Topology n=1000 p=0.5 q=0.3 sigma=0.1 uniform, iters=100 ConstantStepSize(0.01)"),
    # configs[2]: BASELINE.json fixes only n and the corruption type; the rest is SURVEY 8d's proposal, recorded here
    "cfg3": dict(kind="nonuniform", n=2000, p=0.5, p_node_crpt=0.3, p_edge_crpt=0.5, sigma=0.1, sigma_out=0.1,
                 crpt_type="adv", iters=100, lr=0.01, n_sample=0,
                 name="Nonuniform_Topology n=2000 p=0.5 p_node_crpt=0.3 p_edge_crpt=0.5 sigma_in=0.1 sigma_out=0.1 adv, "
                      "iters=100 ConstantStepSize(0.01)"),
    "cfg3sc": dict(kind="nonuniform", n=2000, p=0.5, p_node_crpt=0.3, p_edge_crpt=0.5, sigma=0.1, sigma_out=0.1,
                   crpt_type="self-consistent", iters=100, lr=0.01, n_sample=0,
                   name="Nonuniform_Topology n=2000 p=0.5 p_node_crpt=0.3 p_edge_crpt=0.5 sigma_in=0.1 sigma_out=0.1 "
                        "self-consistent, iters=100 ConstantStepSize(0.01)"),
    # configs[4]: SfM-shaped ring (no reference generator), the reference's large-scale settings compare_algorithms.m:2-5
    # GCW is NOT part of the cfg-5 step: the ring's connection Laplacian has a spectral gap of ~(window/n)^2 ~ 2e-6, the
    # block Lanczos solver (and the reference's eigs, which would also need a 180 GB dense matrix, GCW.m:25) does not
    # converge in thousands of products; the step is the DESC_PGD.m path (incidence + d_ijk + PGD), as the line says
    "cfg5": dict(kind="ring", n=50000, deg=100, window=75, q=0.2, sigma=0.05, iters=30, lr=1.0, n_sample=50, gcw=False,
                 name="Ring_Topology (SfM-shaped) n=50000 mean degree 100 window 75 q=0.2 sigma=0.05, 50 sampled 3-cycles "
                      "per edge, iters=30 ConstantStepSize(1), DESC_PGD path (no GCW: spectral gap ~2e-6)"),
    "small": dict(kind="uniform", n=2000, p=0.1, q=0.2, sigma=0.1, model="uniform", iters=100, lr=0.01, n_sample=0,
                  name="Uniform_Topology n=2000 p=0.1 q=0.2 sigma=0.1 uniform, iters=100 ConstantStepSize(0.01)"),
}
METRIC = "DESC 3-cycle evals/s (whole solve: incidence + d_ijk + PGD + GCW)"
METRIC_PGD = "DESC 3-cycle evals/s (DESC_PGD solve: incidence + d_ijk + PGD; no GCW at this workload)"
UNIT = "evals/s"
PGD_SOURCES = ["desc_b200/csrc/pgd.cu", "desc_b200/csrc/pgd_stream.cuh", "desc_b200/csrc/pgd_passb.cuh"]
TRAFFIC_JSON = os.path.join(ROOT, "profiles", "r02_pgd_traffic.json")


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def captured_traffic(workload, world):
    """DRAM bytes of one PGD iteration from the committed ncu capture, or (None, reason)."""
    if workload != "cfg4" or world != 1:
        return None, "the capture is of cfg4 on one GPU"
    if not os.path.exists(TRAFFIC_JSON):
        return None, "no capture committed"
    try:
        j = json.load(open(TRAFFIC_JSON))
        sha = hashlib.sha1()
        for s in j["sources"]:
            sha.update(open(os.path.join(ROOT, s), "rb").read())
        if sha.hexdigest() != j["sources_sha1"]:
            return None, "kernel sources changed since the capture (%s)" % j.get("report")
        d = j["dram_bytes_per_launch"]
        return sum(v for k, v in d.items() if "k_pgd_stream" in k or "k_pgd_passb" in k), j.get("report")
    except Exception as e:   # noqa: BLE001
        return None, "unreadable capture: %s" % e


class ClockSampler:
    """SM clock and throttle reasons of one GPU every 100 ms while the timed region runs (what the profiling recipe's
    `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.*` line reports), read through NVML in a
    background thread of this process.  A looping `nvidia-smi` child was used first: its start-up and its much larger
    per-sample query set stalled driver calls of the benchmarked process (tens of ms per step on the short cfg-2 /
    cfg-5 steps); it remains the fallback when the NVML binding cannot be imported."""
    NAMES = [("hw_slowdown", "HwSlowdown"), ("hw_thermal_slowdown", "HwThermalSlowdown"),
             ("sw_thermal_slowdown", "SwThermalSlowdown"), ("sw_power_cap", "SwPowerCap")]
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        import threading
        self.p = None
        self.sm, self.mx, self.reasons = [], [], set()
        self.via = "nvml"
        self.period = float(os.environ.get("DESC_BENCH_CLOCK_PERIOD", "0.1"))   # seconds between samples
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].strip().isdigit() else index
            hdl = pynvml.nvmlDeviceGetHandleByIndex(phys)
            masks = [(nm, getattr(pynvml, "nvmlClocksEventReason" + sfx, None) or
                      getattr(pynvml, "nvmlClocksThrottleReason" + sfx)) for nm, sfx in self.NAMES]
            get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(hdl, pynvml.NVML_CLOCK_SM)))

            def loop():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(hdl, pynvml.NVML_CLOCK_SM)))
                        r = int(get_reasons(hdl))
                        for nm, mask in masks:
                            if r & mask:
                                self.reasons.add(nm)
                    except Exception:
                        pass
                    self._stop.wait(self.period)
            self._thread = threading.Thread(target=loop, daemon=True)
            self._thread.start()
        except Exception:
            self.via = "nvidia-smi"
            try:
                self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                           "--format=csv,noheader,nounits", "-lms", "100"],
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            except Exception:
                self.p = None

    def stop(self):
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=2)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "via": "nvml"}
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "via": "nvidia-smi"}


# ------------------------------------------------------------------------------------------
# CPU arm: the C/OpenMP restatement on the workload's own graph family
# ------------------------------------------------------------------------------------------
# thread-seconds per slot as measured on the GPU boxes' hosts (16 threads; the build container is ~2x slower): used
# only to size the sample
CPU_COST_FIXED, CPU_COST_ITER = 4.5e-7, 5.0e-8
_CPU_INPUTS = {}


def workload_estimates(wl):
    """(m, m_cycle) of the workload from its parameters (the CPU arm must not need a GPU to size its sample)"""
    if wl["kind"] == "ring":
        m = wl["n"] * wl["deg"] / 2.0
        p = wl["deg"] / (2.0 * wl["window"])
        codeg = 1.5 * wl["window"] * p * p          # mean common-neighbour count of a window graph (approximate)
    else:
        m = wl["p"] * wl["n"] * (wl["n"] - 1) / 2.0
        codeg = wl["n"] * wl["p"] ** 2
    ns = wl["n_sample"] if wl["n_sample"] > 0 else max(math.ceil(codeg / 4.0), 30)
    return m, m * min(codeg, ns)


def cpu_sample_spec(wl, budget_s, threads, k):
    """the workload's graph itself if its predicted CPU time fits the budget, else the largest smaller member of the
    same family with the same co-degree regime (uniform / nonuniform: p scaled by sqrt(n/n_sub); ring: same degree
    and window)"""
    m, mc = workload_estimates(wl)
    for div in (1, 2, 4, 6, 8, 12, 16, 24, 32, 64):
        n_sub = max(200, wl["n"] // div)
        if wl["kind"] == "ring":
            frac = n_sub / wl["n"]
        else:
            frac = (n_sub / wl["n"]) ** 1.5
        pred = mc * frac * (CPU_COST_FIXED + CPU_COST_ITER * k) / threads * 1.3 + 1.0
        if pred <= budget_s or n_sub == 200:
            spec = dict(wl)
            spec["n"] = n_sub
            if wl["kind"] != "ring":
                spec["p"] = min(0.95, wl["p"] * math.sqrt(wl["n"] / n_sub))
            spec["same_graph"] = div == 1
            spec["predicted_s"] = pred
            return spec
    return None


def cpu_inputs(spec, seed):
    """host inputs of the sample (not timed): graph of the family + the reference model's rotation distribution"""
    import numpy as np
    from oracle import desc_oracle as O
    key = (spec["kind"], spec["n"], spec.get("p"), seed)
    if key in _CPU_INPUTS:
        return _CPU_INPUTS[key]
    rng = np.random.default_rng(seed)
    n = spec["n"]
    if spec["kind"] == "ring":
        w = spec["window"]
        p = spec["deg"] / (2.0 * w)
        rows = []
        for d in range(1, w + 1):                    # pairs at circular distance d
            i = np.nonzero(rng.random(n) < p)[0]
            j = (i + d) % n
            rows.append(np.stack([np.minimum(i, j), np.maximum(i, j)], axis=1))
        e = np.unique(np.concatenate(rows), axis=0)
        ei, ej = e[:, 0], e[:, 1]
    else:
        ei_l, ej_l = [], []
        step = max(1, 20_000_000 // n)
        for a in range(0, n, step):                  # strictly lower triangle in row blocks (Uniform_Topology.m:29-35)
            b = min(n, a + step)
            blk = rng.random((b - a, n)) < spec["p"]
            r, c = np.nonzero(blk)
            keep = c < (r + a)
            ej_l.append(r[keep] + a)
            ei_l.append(c[keep])
        ei, ej = np.concatenate(ei_l), np.concatenate(ej_l)
        o = np.lexsort((ej, ei))
        ei, ej = ei[o], ej[o]
    deg = np.bincount(ei, minlength=n) + np.bincount(ej, minlength=n)
    if (deg == 0).any():
        raise SystemExit("CPU sample graph has an isolated node; use a larger sample")
    m = ei.size
    R = O.proj_so3(rng.standard_normal((n, 3, 3)))
    Rij = R[ei] @ R[ej].transpose(0, 2, 1)
    q, sigma = spec.get("q", 0.2), spec["sigma"]
    corr = rng.random(m) < q
    Rij[~corr] += sigma * rng.standard_normal((int((~corr).sum()), 3, 3))
    Rij[corr] = rng.standard_normal((int(corr.sum()), 3, 3))
    for a in range(0, m, 1_000_000):
        Rij[a:a + 1_000_000] = O.proj_so3(Rij[a:a + 1_000_000])
    Ind = np.stack([ei + 1, ej + 1], axis=1).astype(np.float64)
    out = (Ind, O.to_matlab(Rij))
    _CPU_INPUTS.clear()
    _CPU_INPUTS[key] = out
    return out


def cpu_arm(wl, budget_s, seed=0, k=10):
    """one CPU sample: whole-solve evals/s of the C/OpenMP port, per-stage seconds, and what exactly was run"""
    from oracle import desc_oracle as O
    from oracle import desc_oracle_c as OC
    threads = OC.host_threads()
    k = max(1, min(k, wl["iters"]))
    spec = cpu_sample_spec(wl, budget_s, threads, k)
    Ind, RijMat = cpu_inputs(spec, seed)
    t0 = time.perf_counter()
    r = OC.DESC_init(Ind, RijMat, dict(iters=k, Gradient=O.ConstantStepSize(wl["lr"])),
                     n_sample=(wl["n_sample"] or None), seed=1, threads=threads, full=True, want_R=wl.get("gcw", True))
    wall = time.perf_counter() - t0
    tm, inc = r["timings"], r["inc"]
    per_iter = tm["pgd_s"] / max(r["iters_run"], 1)
    fixed = tm["graph_s"] + tm["build_s"] + tm["cycle_s"] + tm["gcw_s"]
    solve_s = fixed + per_iter * wl["iters"]
    value = inc.m_cycle * wl["iters"] / solve_s
    info = dict(n=int(inc.n), m=int(inc.m), m_cycle=int(inc.m_cycle), n_sample=int(inc.n_sample), threads=threads,
                same_graph=bool(spec["same_graph"]), pgd_iterations_timed=int(r["iters_run"]),
                stage_s={k2: round(v, 4) for k2, v in tm.items()}, pgd_s_per_iteration=per_iter,
                solve_s_at_full_iterations=solve_s, wall_s=wall, pgd_evals_per_s=inc.m_cycle / per_iter,
                p=spec.get("p"))
    text = ("C/OpenMP restatement of DESC.m:14-263 + GCW.m (oracle/desc_full.c, desc_pgd.c; %d threads, every stage threaded) on "
            "%s: n=%d m=%d m_cycle=%d n_sample=%d%s; stages graph %.2f s, build %.2f s, d_ijk %.2f s, GCW %.2f s; PGD timed over %d "
            "iterations (%.3f s each, %.2e evals/s in the loop) and counted %d times: solve = %.1f s"
            % (threads, "the workload's own graph family" + (" at full size" if spec["same_graph"] else
                                                              " at reduced n with the same co-degree regime"),
               inc.n, inc.m, inc.m_cycle, inc.n_sample, "" if spec.get("p") is None else " p=%.4f" % spec["p"],
               tm["graph_s"], tm["build_s"], tm["cycle_s"], tm["gcw_s"], r["iters_run"], per_iter,
               inc.m_cycle / per_iter, wl["iters"], solve_s))
    return value, solve_s, info, text


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    total = max(args.steps, 1)
    budget = max(3.0, min(args.cpu_budget, 300.0 / total))   # the whole run stays within a few minutes
    if args.warmup:
        cpu_arm(dict(wl, n=max(200, wl["n"] // 32), iters=2) if wl["kind"] == "ring" else
                dict(wl, n=max(200, wl["n"] // 32), p=min(0.9, wl["p"] * math.sqrt(32.0)), iters=2), 5.0, k=2)
    vals, times, info, text = [], [], None, ""
    for _ in range(total):
        v, solve_s, info, text = cpu_arm(wl, budget, seed=args.seed)
        vals.append(v)
        times.append(solve_s)
    value = statistics.mean(vals)
    same = info["same_graph"]
    line = {"impl": "reference", "metric": METRIC if wl.get("gcw", True) else METRIC_PGD, "value": value, "unit": UNIT,
            "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(times),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["name"] if same else
                       "%s -- CPU arm on a reduced member of the same family: n=%d p=%s m=%d m_cycle=%d"
                       % (wl["name"], info["n"], info["p"], info["m"], info["m_cycle"]),
                       "same_config": same, "n": info["n"], "m": info["m"], "m_cycle": info["m_cycle"],
                       "n_sample": info["n_sample"]},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["threads"], "kind": "port", "sample": text,
                             "stage_s": info["stage_s"], "pgd_s_per_iteration": info["pgd_s_per_iteration"],
                             "pgd_evals_per_s": info["pgd_evals_per_s"], "same_graph": same},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def make_model(desc_b200, wl, seed, device):
    if wl["kind"] == "uniform":
        return desc_b200.Uniform_Topology(wl["n"], wl["p"], wl["q"], wl["sigma"], wl["model"], seed=seed, device=device,
                                          on_device=True)
    if wl["kind"] == "nonuniform":
        return desc_b200.Nonuniform_Topology(wl["n"], wl["p"], wl["p_node_crpt"], wl["p_edge_crpt"], wl["sigma"],
                                             wl["sigma_out"], wl["crpt_type"], seed=seed, device=device, on_device=True)
    return desc_b200.Ring_Topology(wl["n"], wl["deg"], wl["window"], wl["q"], wl["sigma"], seed=seed, device=device,
                                   on_device=True)


def run_gpu(args, wl):
    import numpy as np
    import torch
    import desc_b200

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    nccl_id = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group(backend="nccl", device_id=dev)
        idt = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            idt = torch.frombuffer(bytearray(desc_b200.nccl_unique_id()), dtype=torch.uint8).to(dev)
        dist.broadcast(idt, 0)
        nccl_id = bytes(idt.cpu().numpy().tobytes())

    # ---- synthetic inputs: the library's device generator; counter-based, so every rank draws the same graph
    mo = make_model(desc_b200, wl, args.seed, local)
    m, n = mo.m, mo.n
    Ind_d, R_d = mo.Ind, mo.RijMat
    # pinned host copies for the end-to-end arm (MATLAB memory layout)
    Ind_h = torch.empty(2 * m, dtype=torch.float64).pin_memory()
    R_h = torch.empty(9 * m, dtype=torch.float64).pin_memory()
    import ctypes as C
    from desc_b200 import _lib
    host = mo.to_host()
    Ind_h.copy_(torch.from_numpy(host["Ind"].ravel(order="F")))
    R_h.copy_(torch.from_numpy(host["RijMat"].ravel(order="F")))
    truth = dict(R_orig=host["R_orig"], ErrVec=host["ErrVec"].ravel().copy(), corrupted=host["corrupted"])
    del host
    Ind_np = Ind_h.numpy().reshape(2, m).T            # (m,2) Fortran view of the pinned buffer
    R_np = R_h.numpy().reshape(m, 3, 3).transpose(2, 1, 0)   # (3,3,m) Fortran view of the pinned buffer
    S_out = torch.empty(m, dtype=torch.float64).pin_memory()
    R_out = torch.empty(9 * n, dtype=torch.float64).pin_memory()
    stream = torch.cuda.current_stream(dev)
    rule = desc_b200.ConstantStepSize(wl["lr"])
    kw = dict(device=local, stream=stream.cuda_stream, rank=rank, world=world, nccl_id=nccl_id)
    state = {}

    def step_resident(fetch=False):
        s = desc_b200.Solver(Ind_d, R_d, n=n, **kw)
        try:
            info = s.build_incidence(n_sample=wl["n_sample"], seed=1)
            s.cycle_inconsistency()
            S_vec, _, iters_run = s.pgd(wl["iters"], rule, want_S=fetch, want_hist=False)
            R_est = s.gcw(want_R=fetch) if wl.get("gcw", True) else None
            state.update(info=info, iters_run=iters_run, timings=s.timings())
            if fetch:
                state.update(S_vec=S_vec, R_est=R_est)
        finally:
            s.close()

    def step_e2e(solver_kw=None):
        s = desc_b200.Solver(Ind_np, R_np, n=n, **(solver_kw or kw))
        try:
            s.build_incidence(n_sample=wl["n_sample"], seed=1)
            s.cycle_inconsistency()
            r = rule._to_c()
            run = C.c_int32(0)
            _lib.check(s._lib.desc_b200_pgd(s._h, wl["iters"], C.byref(r), C.c_void_p(S_out.data_ptr()), None, C.byref(run)))
            if wl.get("gcw", True):
                _lib.check(s._lib.desc_b200_gcw(s._h, None, C.c_void_p(R_out.data_ptr())))
            state.update(e2e_iters=int(run.value))
        finally:
            s.close()

    def timed(fn, steps, **last_kw):
        import gc
        gc.collect()
        gc.disable()            # no collector pauses of the host inside the timed region
        try:
            return _timed(fn, steps, last_kw)
        finally:
            gc.enable()

    def _timed(fn, steps, last_kw):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        launches = 0
        trace = os.environ.get("DESC_BENCH_TRACE") == "1"   # diagnostics: host wall time of every step (adds a sync)
        for i in range(steps):
            t0 = time.perf_counter()
            fn(**(last_kw if i == steps - 1 else {}))
            if trace:
                torch.cuda.synchronize(dev)
                sys.stderr.write("step %s: %.1f ms\n" % (fn.__name__, 1e3 * (time.perf_counter() - t0)))
            launches += state.get("timings", {}).get("total_launches", 0)
        ev1.record(stream)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), launches

    # the clock sampler starts BEFORE the warm-up: nvidia-smi's own start-up (NVML init) must not fall into the timed
    # region (it cost ~10 ms per step on the 35 ms steps of cfg 2)
    sampler = ClockSampler(local) if rank == 0 and os.environ.get("DESC_BENCH_NO_CLOCKS") != "1" else None
    for _ in range(args.warmup):
        step_resident()
    ms_total, launches = timed(step_resident, args.steps, fetch=args.dump_outputs is not None)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, S_vec=state["S_vec"], R_est=state["R_est"])
    ms_step = ms_total / args.steps
    info, iters_run, tm = state["info"], state["iters_run"], state["timings"]
    evals = info["m_cycle"] * iters_run
    value = evals / (ms_step * 1e-3)

    # the refinement stage of the full DESC() call (DESC.m:265-312), reported beside the metric (not in it)
    laa = None
    if world == 1 and not args.no_side and wl.get("gcw", True):
        s = desc_b200.Solver(Ind_d, R_d, n=n, **kw)
        try:
            s.build_incidence(n_sample=wl["n_sample"], seed=1)
            s.cycle_inconsistency()
            s.pgd(wl["iters"], rule, want_S=False, want_hist=False)
            s.gcw(want_R=False)
            s.refine()
            _, sc = s.refine()                       # second call: buffers come from the pool
            t = s.timings()
            laa = {"ms": t["laa_ms"], "irls_iterations": t["laa_iters"], "cg_iterations": t["laa_cg_iters"],
                   "final_score": float(sc[-1]) if len(sc) else None}
        finally:
            s.close()

    # SURVEY 8(f) stages on the same graph, reported beside the metric (not in it); never fatal for the bench line
    side = None
    if world == 1 and not args.no_side and wl["kind"] == "uniform":
        try:
            side = side_stages(desc_b200, Ind_d, R_d, wl, kw, measured_peak()[0], args.seed)
        except Exception as e:   # noqa: BLE001
            side = {"error": "%s: %s" % (type(e).__name__, e)}

    step_e2e()
    ms_e2e_total, _ = timed(step_e2e, args.steps)
    ms_e2e = ms_e2e_total / args.steps
    e2e = {"value": evals / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": (2 * m + 9 * m) * 8,
           "d2h_bytes_per_step": (m + 9 * n) * 8, "ms_per_step": ms_e2e}

    # accuracy of what the timed path returned (S_out / R_out of the last e2e step) against the model's ground truth
    quality = None
    if rank == 0:
        try:
            S_np = S_out.numpy()
            corr = truth["corrupted"]
            mean_err = med_err = float("nan")
            if wl.get("gcw", True):
                Rg = np.asfortranarray(R_out.numpy().reshape(n, 3, 3).transpose(2, 1, 0))
                _, _, mean_err, med_err = desc_b200.Rotation_Alignment(Rg, truth["R_orig"], device=local)
            quality = {"mean_abs_S_minus_ErrVec": float(np.mean(np.abs(S_np - truth["ErrVec"]))),
                       "mean_S_corrupted": float(S_np[corr].mean()) if corr.any() else None,
                       "mean_S_clean": float(S_np[~corr].mean()),
                       "gcw_rotation_error_deg_mean": float(mean_err), "gcw_rotation_error_deg_median": float(med_err)}
        except Exception as e:   # noqa: BLE001
            quality = {"error": "%s: %s" % (type(e).__name__, e)}

    # N > 1: the N-rank result (just computed by step_e2e on every rank) against a 1-rank solve on rank 0
    parity = None
    if world > 1:
        S_N = S_out.numpy().copy()
        R_N = R_out.numpy().copy()
        it_N = state["e2e_iters"]
        if rank == 0:
            step_e2e(dict(device=local, stream=stream.cuda_stream))
            S_1, R_1 = S_out.numpy(), R_out.numpy()
            ang = np.zeros(1)
            if wl.get("gcw", True):
                Ra = np.asfortranarray(R_N.reshape(n, 3, 3).transpose(2, 1, 0))
                Rb = np.asfortranarray(R_1.reshape(n, 3, 3).transpose(2, 1, 0))
                Rab, _, _, _ = desc_b200.Rotation_Alignment(Ra, Rb, device=local)
                D = (np.asarray(Rab) - Rb).reshape(9, n)
                ang = np.degrees(2.0 * np.arcsin(np.minimum(np.sqrt((D ** 2).sum(axis=0)) / (2.0 * math.sqrt(2.0)), 1.0)))
            parity = {"against": "1-rank solve of the same inputs on rank 0", "max_abs_dS_vec": float(np.max(np.abs(S_N - S_1))),
                      "max_rel_dS_vec": float(np.max(np.abs(S_N - S_1) / np.maximum(np.abs(S_1), 1e-12))),
                      "iters_run": [int(it_N), int(state["e2e_iters"])],
                      "mean_rotation_angle_deg": float(ang.mean()),
                      "ok": bool(np.max(np.abs(S_N - S_1) / np.maximum(np.abs(S_1), 1e-12)) <= 1e-10 and
                                 it_N == state["e2e_iters"] and ang.mean() <= 1e-6)}
        dist.barrier()

    per_rank = None
    if world > 1:   # per-rank kernel / collective times of the PGD iteration (load balance)
        mine = [tm.get("pgd_pass1_ms", 0.0), tm.get("pgd_pass2_ms", 0.0), tm.get("pgd_comm_ms", 0.0)]
        allv = [None] * world
        dist.all_gather_object(allv, mine)
        per_rank = {"pass1_ms": [round(v[0], 4) for v in allv], "pass2_ms": [round(v[1], 4) for v in allv],
                    "comm_ms": [round(v[2], 4) for v in allv]}
    if rank == 0:
        peak, peak_src = measured_peak()
        local_slots = info["local_slots"]
        local_edges = info["edge_end"] - info["edge_begin"]
        alg_bytes = 40.0 * local_slots + 12.0 * local_edges + 8.0 * info["m"]
        iter_ms = tm["pgd_iter_ms"]
        achieved = alg_bytes / (iter_ms * 1e-3) / 1e9 if iter_ms > 0 else 0.0
        traffic, traffic_src = captured_traffic(args.workload, world)

        def stage(bytes_, ms):
            return {"algorithmic_bytes": bytes_, "ms": ms, "achieved_gbs": bytes_ / (ms * 1e-3) / 1e9 if ms > 0 else None,
                    "frac": bytes_ / (ms * 1e-3) / 1e9 / peak if ms > 0 else None}
        stages = {"incidence_build": stage(24.0 * info["m"] + 20.0 * local_slots + 4.0 * local_edges, tm["build_ms"]),
                  "d_ijk": stage(72.0 * info["m"] + 20.0 * local_slots + 4.0 * local_edges, tm["cycle_ms"])}
        if tm.get("gcw_spmv_ms", 0) > 0:
            stages["gcw_spmv"] = stage(88.0 * info["m"] + 144.0 * n, tm["gcw_spmv_ms"])
        two_pass = tm.get("pgd_pass2_ms", 0.0) > 0.05 * max(tm.get("pgd_pass1_ms", 0.0), 1e-9)
        roofline = {"bound": "hbm",
                    "kernel": ("PGD iteration = k_pgd_stream (update, smaller endpoints) + k_pgd_passb (tables, larger endpoints)"
                               if two_pass else
                               "PGD iteration = k_pgd_block (update) + k_pgd_scatter (tables): the direct-load kernels the "
                               "library picks for sparse graphs (fewer than 100 own edges per vertex), timed as one span"),
                    "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                    "algorithmic_bytes_per_launch": alg_bytes, "kernel_ms": iter_ms,
                    "kernels_ms": {"k_pgd_stream": tm.get("pgd_pass1_ms"), "k_pgd_passb": tm.get("pgd_pass2_ms")},
                    "comm_ms_per_iteration": tm.get("pgd_comm_ms"),
                    "formula": "40*slots + 12*edges_with_cycles + 8*m (SURVEY 8d), per rank, per iteration (both kernels)",
                    "stages": stages}
        cpu = None
        if world == 1 and not args.no_cpu:
            v, solve_s, ci, text = cpu_arm(wl, args.cpu_budget, seed=args.seed)
            cpu = {"value": v, "unit": UNIT, "cores": ci["threads"], "kind": "port", "sample": text,
                   "stage_s": ci["stage_s"], "pgd_s_per_iteration": ci["pgd_s_per_iteration"],
                   "pgd_evals_per_s": ci["pgd_evals_per_s"], "same_graph": ci["same_graph"],
                   "n": ci["n"], "m": ci["m"], "m_cycle": ci["m_cycle"]}
        line = {"metric": METRIC if wl.get("gcw", True) else METRIC_PGD, "value": value, "unit": UNIT, "n_gpus": world,
                "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic (device generator csrc/gen.cu, seed %d)" % args.seed,
                "config": {"workload": wl["name"], "n": n, "m": m, "m_pos": info["m_pos"],
                           "m_cycle": info["m_cycle"], "n_sample": info["n_sample"], "iters_run": iters_run,
                           "l2": "inputs_exceed_l2 (per-iteration working set %.1f GB)" % (alg_bytes / 1e9),
                           "parallelism": "edge-sharded x%d" % world},
                "solve_s": ms_step * 1e-3,
                "pgd_evals_per_s": evals / (tm["pgd_ms"] * 1e-3) if tm["pgd_ms"] > 0 else None,
                "stages_ms": {k: tm[k] for k in ("graph_ms", "build_ms", "cycle_ms", "pgd_ms", "gcw_ms", "pgd_iter_ms",
                                                 "pgd_pass1_ms", "pgd_pass2_ms", "pgd_comm_ms")},
                "generator_ms": mo.gen_ms,
                "gcw_iters": tm["gcw_iters"], "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
                "cpu_baseline": cpu, "clocks": clocks, "per_rank": per_rank, "parity": parity, "quality": quality,
                "laa_refine": laa, "side_stages": side}
        print(json.dumps(line), flush=True)
    mo.close()
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, **arrays):
    """DIR/<name>.npy of every array a caller of the timed solve receives, in the layout it receives them (float64),
    so that two builds can be compared output for output.  Every workload's outputs fit the size limit as a whole."""
    import numpy as np
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items() if v is not None}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def side_stages(desc_b200, Ind_d, R_d, wl, kw, peak, seed):
    """CEMP / CEMP+GCW / CEMP+MST / MPLS / Spectral (the comparators Demo/compare_algorithms.m runs beside DESC) with
    the demo's parameters on the bench graph; device-timed by the library."""
    import numpy as np
    out = {}
    s = desc_b200.Solver(Ind_d, R_d, n=wl["n"], **kw)
    try:
        info = s.build_incidence(n_sample=50, seed=1)                      # CEMP_parameters.nsample = 50
        s.cycle_inconsistency()
        beta = 2.0 ** np.arange(6)
        s.cemp(6, beta)
        s.cemp(6, beta)                                                     # second call: buffers exist
        t = s.timings()
        per = t["cemp_ms"] / 7.0                                            # initial mean + 6 reweightings
        alg = 16.0 * info["m_cycle"] + 24.0 * info["m"]                     # pk_jk+pk_ki+S0 per slot; rowptr, x in, x out per edge
        out["cemp"] = {"ms": t["cemp_ms"], "m_cycle": info["m_cycle"], "reweightings": 7, "ms_per_reweighting": per,
                       "algorithmic_bytes_per_reweighting": alg, "achieved_gbs": alg / (per * 1e-3) / 1e9,
                       "frac_of_hbm_peak": alg / (per * 1e-3) / 1e9 / peak}
        s.cemp_gcw()
        out["cemp_gcw_ms"] = s.timings()["gcw_ms"]
        s.mst_init()
        out["cemp_mst_ms"] = s.timings()["mst_ms"]
        MP = dict(stop_threshold=1e-3, max_iter=100, reweighting=[32.0], thresholding=[0.95, 0.9, 0.85, 0.8],
                  cycle_info_ratio=1.0 / (np.arange(1, 101) + 1))
        _, sc = s.mpls_refine(MP)
        t = s.timings()
        out["mpls_refine"] = {"ms": t["laa_ms"], "iterations": t["laa_iters"], "cg_iterations": t["laa_cg_iters"],
                              "final_score": float(sc[-1]) if len(sc) else None}
        s.spectral()
        out["spectral_ms"] = s.timings()["gcw_ms"]
    finally:
        s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="desc_b200", choices=["desc_b200", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-budget", type=float, default=25.0,
                    help="seconds of CPU work one CPU sample may take (sizes the sample graph)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-side", action="store_true", help="skip the SURVEY 8(f) side stages (CEMP, MPLS, ...)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (S_vec.npy; R_est.npy when the step runs GCW) to DIR; "
                         "that step also copies them to the host, which the other steps skip")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "desc_b200":
        ap.error("--dump-outputs writes what the GPU solve returns; the reference arm solves a different graph")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_gpu(args, wl)


if __name__ == "__main__":
    main()
