#!/usr/bin/env python
"""bench.py -- RTR iterations/sec on sphere2500 (BASELINE.json metric) + the Q.X SpMV roofline.

    python bench.py --gpus N --steps K --warmup W [--dump-outputs DIR]   (N>1: launched by torch.distributed.run)
    python bench.py --impl reference --steps K --warmup W  (CPU restatement of the reference path)

A "step" is one QuadraticOptimizer::optimize() call with the constants PGOAgent::updateX uses
(ref src/PGOAgent.cpp:1131-1137: RTR, tol 1e-2, 1 outer iteration, <= 10 tCG iterations, radius 100)
and the reference's preconditioner operator (Q + 0.1 I)^-1.  Steps walk the optimisation trajectory from
the chordal initialisation; the iterate is reset to the initial point every CYCLE steps, before the early-exit
tolerance is reached, so every timed step does full work.

 N = 1 : sphere2500 as ONE agent (r = 5).   value = steps/s with the iterate resident in HBM;
         e2e   = the same through QuadraticOptimizer.optimize() with pinned host buffers (H2D + D2H per step).
 N > 1 : sphere2500 split contiguously into 8 agents -- the SAME 8-agent problem at every GPU count, 8/N agents per
         GPU; every round = pack public poses -> one NCCL all-gather -> device-side G rebuild -> the agents of the
         round's colour class take one RTR step (side by side as thread-block clusters while a GPU hosts >= 2 of them).  value = RBCD rounds/s ("strong": fixed work,
         more GPUs); the reference arm runs the same 8-agent coloured RBCD on the host cores.  The N = 1 line carries
         the 1-GPU point of that curve under "multi_agent_1gpu"; torus3D (8 agents) is measured alongside.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DATASET = "sphere2500"
RANK_R = 5
CYCLE = 6            # steps per trajectory before resetting to the initial point (see docstring)
METRIC = "rtr_iters_per_sec_sphere2500"
UNIT = "iter/s"
MULTI_AGENTS = int(os.environ.get("DPGO_BENCH_AGENTS", "16"))   # agents of the multi-GPU workload: FIXED, so that the same algorithm runs at every
                     # GPU count; 16 = two per GPU at 8 GPUs, one of each colour of the 2-colour RBCD, so no GPU idles in a round


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            pk = json.load(open(path))
            return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT = 64 << 20   # bytes, all arrays of one --dump-outputs directory


def dump_outputs(path: str, arrays: dict) -> None:
    """--dump-outputs: what the timed path computed in its last step, one float64 <name>.npy per array, so that two
    builds run with the same arguments (hence the same inputs) can be compared output for output."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def ncu_traffic(kernel: str):
    """DRAM read+write bytes per launch from the committed ncu capture (profiles/traffic.json), else None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel]
        return t["dram_bytes_read"] + t["dram_bytes_write"]
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            f = [x.strip() for x in row.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU legs (the only places that may execute oracle/)
# ------------------------------------------------------------------------------------------------
def cpu_reference_steps(steps: int, warmup: int, sample_desc_only: bool = False):
    """Time the CPU restatement of the reference path on the SAME workload (sphere2500, one agent, r=5,
    RTR with updateX constants, exact (Q+0.1I)^-1 preconditioner).  Returns (steps_per_sec, info)."""
    try:
        from oracle import cpu_port                      # C++ restatement (g++ -O3 -march=native), if built
        have_port = cpu_port.available()
    except Exception:
        cpu_port, have_port = None, False
    from oracle import dpgo_oracle as orc
    meas, n = orc.read_g2o(os.path.join(ROOT, "data", DATASET + ".g2o"))
    Q = orc.construct_connection_laplacian(meas, n)
    X0 = orc.fixed_stiefel_variable(meas.d, RANK_R) @ orc.chordal_initialization(meas, n)
    if have_port:
        # single thread = the reference's default (ENABLE_OPENMP OFF; Eigen's dense*sparse product is serial);
        # a threaded variant (products over columns) is tried as well and the faster one is reported
        runner = cpu_port.Runner(Q, n, meas.d, RANK_R, threads=1)
        best = 1
        try:
            t0 = time.perf_counter(); runner.step(X0); runner.step(X0); t1 = time.perf_counter() - t0
            nthr = max(2, min(8, os.cpu_count() or 2))
            alt = cpu_port.Runner(Q, n, meas.d, RANK_R, threads=nthr)
            t0 = time.perf_counter(); alt.step(X0); alt.step(X0); t2 = time.perf_counter() - t0
            if t2 < 0.9 * t1:
                runner, best = alt, nthr
        except Exception:
            pass
        kind, cores = "port", best
        label = ("C++ restatement of the reference path (scalar-CSR X*Q, min-degree sparse LDL^T solves of Q+0.1I, "
                 "ROPTLIB RTR/tCG restated; 10+j products per call), g++ -O3.  The reference itself cannot be built here (Eigen / "
                 "SuiteSparse / ROPTLIB absent); its CHOLMOD supernodal factor solves are plausibly 2-4x faster than this port's")
    else:
        prob = orc.QuadraticProblem(n, meas.d, RANK_R)
        prob.set_Q(Q)

        class _PyRunner:
            def step(self, X):
                oo = orc.QuadraticOptimizer(prob)
                oo.tr_tolerance, oo.tr_iterations, oo.tr_max_inner, oo.tr_initial_radius = 1e-2, 1, 10, 100.0
                return oo.optimize(X)
        runner = _PyRunner()
        kind, cores, label = "port", 1, "NumPy/SciPy oracle (scipy.sparse SpMM + SuperLU solves), single thread"
    X = X0
    for i in range(warmup):
        X = runner.step(X) if (i + 1) % CYCLE else runner.step(X0)
    X = X0
    t0 = time.perf_counter()
    for i in range(steps):
        if i % CYCLE == 0:
            X = X0
        X = runner.step(X)
    dt = time.perf_counter() - t0
    info = {"value": steps / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{steps} consecutive optimize() steps of the bench workload ({DATASET}, 1 agent, r={RANK_R}, "
                      f"reset every {CYCLE}); {label}", "host_cpus": os.cpu_count()}
    return steps / dt, dt, info


class CpuRBCD:
    """The k-agent coloured RBCD of the multi-GPU arm on the host cores: the C++ restatement of the reference path
    (oracle/cpp/cpu_port.cpp) per agent, G rebuilt per step as the reference does (src/PGOAgent.cpp:783-859, vectorised),
    the agents of one colour class stepping concurrently on a thread pool (the port releases the GIL)."""

    def __init__(self, dataset: str, k: int):
        from concurrent.futures import ThreadPoolExecutor
        from oracle import cpu_port
        from oracle import dpgo_oracle as orc
        self.orc = orc
        meas, n = orc.read_g2o(os.path.join(ROOT, "data", dataset + ".g2o"))
        self.d, self.r, self.k, self.n = meas.d, RANK_R, k, n
        dh = self.d + 1
        drv = orc.MultiRobotDriver(meas, n, k, r=RANK_R, schedule="coloured")
        self.colour, self.ncolours, self.glob = drv.colour, drv.ncolours, drv.glob
        self.X0 = [ag.X.copy() for ag in drv.agents]
        self.X = [x.copy() for x in self.X0]
        self.runners, self.tables = [], []
        for ag in drv.agents:
            self.runners.append(cpu_port.Runner(ag.problem.Q, ag.n, self.d, RANK_R, threads=1))
            sh = ag.shared_lc
            out = sh.r1 == ag.id
            self.tables.append(dict(n=ag.n, out=out, local=np.where(out, sh.p1, sh.p2), nbr_a=np.where(out, sh.r2, sh.r1),
                                    nbr_p=np.where(out, sh.p2, sh.p1), T=orc._homogeneous(sh), Om=orc._omega(sh)))
        self.pool = ThreadPoolExecutor(max_workers=max(1, min(os.cpu_count() or 1, k)))
        self.threads = self.pool._max_workers
        self.round = 0

    def _step_agent(self, a, Xs):
        tb, dh = self.tables[a], self.d + 1
        G = np.zeros((self.r, dh * tb["n"]))
        if len(tb["local"]):
            Xn = np.stack([Xs[int(b)][:, int(q) * dh:(int(q) + 1) * dh] for b, q in zip(tb["nbr_a"], tb["nbr_p"])])   # (m, r, dh)
            L_out = -np.einsum("mrq,mcq->mrc", Xn * tb["Om"][:, None, :], tb["T"])
            L_in = -np.einsum("mrq,mqc->mrc", Xn, tb["T"]) * tb["Om"][:, None, :]
            L = np.where(tb["out"][:, None, None], L_out, L_in)
            Gt = G.reshape(self.r, tb["n"], dh)
            np.add.at(Gt, (slice(None), tb["local"]), np.transpose(L, (1, 0, 2)))
        self.runners[a].set_G(G)
        return self.runners[a].step(Xs[a])

    def run_round(self):
        c = self.round % self.ncolours
        active = [a for a in range(self.k) if self.colour[a] == c]
        snap = list(self.X)
        for a, Xn in zip(active, self.pool.map(lambda a: self._step_agent(a, snap), active)):
            self.X[a] = Xn
        self.round += 1
        return len(active)

    def reset(self):
        self.X = [x.copy() for x in self.X0]
        self.round = 0


def cpu_multi_agent_rounds(dataset: str, k: int, rounds: int, warmup: int):
    """Rounds/s of the k-agent coloured RBCD on the host cores (same workload and reset cycle as the GPU arm)."""
    sim = CpuRBCD(dataset, k)
    cyc = CYCLE * sim.ncolours
    for _ in range(warmup):
        sim.run_round()
    sim.reset()
    steps = 0
    t0 = time.perf_counter()
    for i in range(rounds):
        if i % cyc == 0:
            sim.reset()
        steps += sim.run_round()
    dt = time.perf_counter() - t0
    info = {"value": rounds / dt, "unit": "rounds/s", "cores": sim.threads, "kind": "port",
            "sample": f"{rounds} coloured RBCD rounds of {dataset} split into {k} agents ({sim.ncolours} colours, reset every {cyc} "
                      f"rounds), C++ restatement of the reference path per agent, active agents on {sim.threads} threads",
            "agent_steps": steps, "host_cpus": os.cpu_count()}
    return rounds / dt, dt, info


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    if args.gpus > 1:
        # the multi-GPU arm's workload: sphere2500 split into MULTI_AGENTS agents, coloured RBCD; value = rounds/s
        val, dt, info = cpu_multi_agent_rounds(DATASET, MULTI_AGENTS, steps, min(args.warmup, 4))
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
                "warmup": min(args.warmup, 4), "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "data/sphere2500.g2o (public dataset), chordal init",
                "config": multi_config(DATASET, MULTI_AGENTS, None, "host cores only"), "cpu_baseline": info,
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return
    val, dt, info = cpu_reference_steps(steps, min(args.warmup, 2))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": min(args.warmup, 2), "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "data/sphere2500.g2o (public dataset), chordal init",
            "config": workload_config(1, "host cores only"), "cpu_baseline": info,
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def multi_config(dataset: str, k: int, ncolours, placement: str):
    return {"workload": f"{dataset}.g2o SE(3) split contiguously into {k} agents (fixed at every GPU count), r={RANK_R}, coloured RBCD: "
                        f"per round one boundary-pose exchange, then every agent of the round's colour class takes one RTR step "
                        f"(tol 1e-2, <=10 tCG, radius 100, preconditioner (Q+0.1I)^-1); an iteration = one round",
            "agents": k, "colours": ncolours, "placement": placement, "cycle_reset": CYCLE,
            "l2_policy": "the agents' working sets are L2-resident by nature of the named datasets; the SpMV-roofline inputs exceed L2"}


def workload_config(n_agents: int, schedule: str):
    return {"workload": f"{DATASET}.g2o SE(3), 2500 poses / 4949 edges, {n_agents} agent(s), r={RANK_R}, "
                        f"one RTR step per optimize() (tol 1e-2, <=10 tCG, radius 100), preconditioner (Q+0.1I)^-1",
            "agents": n_agents, "schedule": schedule, "cycle_reset": CYCLE,
            "l2_policy": "sphere2500's working set (Q 1.6 MB, vectors, 29 MB of preconditioner blocks) is L2-resident by nature "
                         "of the named dataset; the SpMV-roofline inputs (605 MB) exceed L2"}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def spmv_roofline(torch, dp, pg, peak_gbs, peak_src, dims=(100, 100, 40), reps=20):
    """Q.X product alone on a synthetic grid far larger than L2 (SURVEY 8d config 5 family)."""
    edges, n, _ = pg.synthetic_grid_graph(*dims, edges_per_pose=4.0, seed=0)
    prob = dp.QuadraticProblem(n, 3, RANK_R, preconditioners=(dp.PRECOND_BLOCK_JACOBI,))
    prob.setQ_blocks(*pg.connection_laplacian_blocks(edges))
    prob.set_stream(torch.cuda.current_stream().cuda_stream)
    X = torch.randn(RANK_R * 4 * n, dtype=torch.float64, device="cuda")
    out = torch.empty_like(X)
    for _ in range(3):
        prob.spmv_device(X.data_ptr(), out.data_ptr(), False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        prob.spmv_device(X.data_ptr(), out.data_ptr(), False)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    nbytes = prob.spmv_algorithmic_bytes(False)
    ach = nbytes / (ms * 1e-3) / 1e9
    res = {"kernel": "k_spmv_tma<5,4,192> (Out = X Q; bulk-TMA producer, predicate-light DMMA consumers)", "workload": f"synthetic grid {dims[0]}x{dims[1]}x{dims[2]} = {n} poses, "
           f"{len(edges)} edges, r={RANK_R}, nb={prob.num_blocks()} blocks", "bound": "hbm", "achieved": ach,
           "peak": peak_gbs, "peak_source": peak_src, "unit": "GB/s", "frac": ach / peak_gbs,
           "algorithmic_bytes_per_launch": nbytes, "us_per_launch": ms * 1e3, "launches_timed": reps,
           "traffic": ncu_traffic("k_spmv_tma")}
    prob.close()
    del X, out
    torch.cuda.empty_cache()
    return res


def run_gpu_arm(args):
    import torch
    import dpo_b200 as dp
    from dpo_b200 import posegraph as pg
    from dpo_b200.agent import DistributedPGO

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    K, W = args.steps, max(args.warmup, 3)
    peak, peak_src = measured_peaks()

    edges, n = pg.read_g2o_file(os.path.join(ROOT, "data", DATASET + ".g2o"))
    d = edges.d
    X0 = pg.fixedStiefelVariable(d, RANK_R) @ pg.chordalInitialization(d, n, edges)
    line = {"metric": METRIC, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "data/sphere2500.g2o (public benchmark pose graph shipped with the reference), chordal initialisation"}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if world == 1:
        prob = dp.QuadraticProblem(n, d, RANK_R, device=local_rank,
                                   preconditioners=(dp.PRECOND_BLOCK_JACOBI, dp.PRECOND_SPARSE_EXACT, dp.PRECOND_DENSE_EXACT))
        prob.setQ_blocks(*pg.connection_laplacian_blocks(edges))
        prob.set_stream(torch.cuda.current_stream().cuda_stream)
        opt = dp.QuadraticOptimizer(prob)
        opt.setTrustRegionTolerance(1e-2)
        opt.setTrustRegionIterations(1)
        opt.setTrustRegionMaxInnerIterations(10)
        opt.setTrustRegionInitialRadius(100)
        PRE = dp.PRECOND_DENSE_EXACT if args.precond == "dense" else dp.PRECOND_SPARSE_EXACT
        opt.setPreconditioner(PRE)
        X0d = torch.from_numpy(np.asfortranarray(X0).ravel(order="F").copy()).to(dev)

        def resident_steps(count, collect=None):
            for i in range(count):
                if i % CYCLE == 0:
                    prob.copy_X_from_device(X0d.data_ptr())
                opt.optimize_resident_async()
                if collect is not None:
                    collect.append(opt.fetch_result())

        # ---- correctness trail of one cycle (also warms everything) ----
        trail = []
        resident_steps(CYCLE, trail)
        resident_steps(W)
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        resident_steps(K)
        e1.record()
        barrier()
        ms_total = e0.elapsed_time(e1)
        outputs = None
        if args.dump_outputs:
            # the iterate and the result record of the last timed step, before the end-to-end leg overwrites them
            rs_last = opt.fetch_result()
            outputs = {"X": prob.download_X(), "f_opt": [rs_last.f_opt], "gradnorm_opt": [rs_last.gradnorm_opt]}
        # ---- end to end: public API, pinned host buffers, H2D + D2H inside the timed region ----
        def pinned():                       # (r, N) Fortran-ordered view of a pinned (N, r) tensor
            t = torch.empty(((d + 1) * n, RANK_R), dtype=torch.float64).pin_memory()
            return t, t.numpy().T
        keep0, X0f = pinned()
        X0f[...] = X0
        keepA, bufA = pinned()
        keepB, bufB = pinned()
        bufs = [bufA, bufB]
        host = X0f
        for i in range(W):
            host = opt.optimize(X0f if i % CYCLE == 0 else host, out=bufs[i & 1])
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            host = opt.optimize(X0f if i % CYCLE == 0 else host, out=bufs[i & 1])
        barrier()
        e2e_dt = time.perf_counter() - t0
        clocks = sampler.stop()
        last = opt.getOptResult()
        vec_bytes = RANK_R * (d + 1) * n * 8
        # ---- roofline of the dominant kernel of the step: the persistent k_optimize launch ----
        spmv_b = prob.spmv_algorithmic_bytes(True)
        N = (d + 1) * n
        pre_b = prob.precond_algorithmic_bytes(PRE)      # bytes of the operator's blocks one application streams
        pre_full = N * N * 8 + 2 * vec_bytes                                # the full dense operator
        per_step, per_step_full, flops = [], [], []
        for rs in trail:
            per_step.append(rs.spmv_passes * spmv_b + rs.precond_applies * pre_b)
            per_step_full.append(rs.spmv_passes * spmv_b + rs.precond_applies * pre_full)
            flops.append(rs.precond_applies * 2.0 * RANK_R * N * N)
        alg_bytes = float(np.mean(per_step))
        alg_full = float(np.mean(per_step_full))
        ms_step = ms_total / K
        ach = alg_bytes / (ms_step * 1e-3) / 1e9
        napply = float(np.mean([rs.precond_applies for rs in trail]))
        npass = float(np.mean([rs.spmv_passes for rs in trail]))
        roof = {"kernel": "k_optimize<5,4> (one persistent launch per step)", "bound": "hbm", "achieved": ach,
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": ach / peak,
                "algorithmic_bytes_per_launch": alg_bytes, "traffic": ncu_traffic("k_optimize_" + args.precond),
                "traffic_note": "dram__bytes of one launch under ncu (caches flushed before the launch): the operator's blocks "
                                "are fetched from HBM once per launch and re-read from L2 by the other applications",
                "precond_applies_per_step": napply, "q_passes_per_step": npass,
                "note": "bytes = q_passes*(132 nb + 4(n+1) + 96 r n) + precond_applies*(P + 16 r N), averaged over the cycle; "
                        + ("P = all dense blocks of the nested-dissection factorisation of Q+0.1I, streamed once per application "
                           "(L2-resident at this size: the launch is bound by the latency of its ~80 grid-wide phases, not by HBM)"
                           if args.precond == "sparse" else
                           "P = unique bytes of the symmetric dense (Q+0.1I)^-1 = 4 N (N+8) (upper-triangle kernel)")}
        if prob.nd_ready():
            roof["nd"] = prob.nd_info()
        if args.precond == "dense":
            roof["full_matrix"] = {"algorithmic_bytes_per_launch": alg_full, "achieved": alg_full / (ms_step * 1e-3) / 1e9,
                                   "frac": alg_full / (ms_step * 1e-3) / 1e9 / peak}
        line.update({
            "value": K / (ms_total * 1e-3), "ms_per_step": ms_step,
            "config": workload_config(1, "single agent"),
            "e2e": {"value": K / e2e_dt, "unit": UNIT, "h2d_bytes_per_step": vec_bytes,
                    "d2h_bytes_per_step": vec_bytes + 96, "ms_per_step": 1e3 * e2e_dt / K,
                    "api": "dpo_b200.QuadraticOptimizer.optimize(Y) -> dpgo_optimize (host buffers)"},
            "gpu_launches": K,
            "clocks": clocks,
            "roofline": roof,
            "trajectory": [{"f": rs.f_opt, "gradnorm": rs.gradnorm_opt, "tcg": rs.tcg_iterations,
                            "status": rs.tcg_status, "spmv_passes": rs.spmv_passes} for rs in trail],
        })
        # ---- extras: Jacobi throughput mode and the RGD step on the same workload ----
        extras = {}
        for name, setter in (("rtr_block_jacobi", lambda: (opt.setAlgorithm(dp.ROPTALG.RTR), opt.setPreconditioner(dp.PRECOND_BLOCK_JACOBI))),
                             ("rgd", lambda: opt.setAlgorithm(dp.ROPTALG.RGD))):
            setter()
            resident_steps(W)
            barrier()
            e0.record()
            resident_steps(K)
            e1.record()
            barrier()
            extras[name + "_iters_per_sec"] = K / (e0.elapsed_time(e1) * 1e-3)
        line["extra"] = extras
        prob.close()
        if not args.no_multi:
            # the multi-GPU arm's workloads with all agents on this one GPU: the 1-GPU point of the scaling curve
            line["multi_agent_1gpu"] = {}
            for ds in (DATASET, "torus3D"):
                m = measure_multi(torch, None, dp, pg, ds, MULTI_AGENTS, 0, 1, local_rank, K, W, peak, peak_src, with_e2e=False)
                line["multi_agent_1gpu"][ds] = {k2: m[k2] for k2 in ("rounds_per_sec", "ms_per_round", "agent_steps_per_sec", "colours", "final",
                                                                     "concurrent_agents", "step_kernel_launch")}
        if not args.no_spmv:
            line["roofline_spmv"] = spmv_roofline(torch, dp, pg, peak, peak_src)
            if not args.no_sweep:
                # SURVEY 8(d) / BASELINE.md section 4: the sweep across the L2 boundary (10k ... 1M poses at 4 edges / pose)
                sweep = []
                for dims in ((25, 20, 20), (40, 30, 25), (50, 50, 40), (100, 60, 50), (100, 100, 100)):
                    rr = spmv_roofline(torch, dp, pg, peak, peak_src, dims=dims, reps=20)
                    sweep.append({"poses": dims[0] * dims[1] * dims[2], "algorithmic_bytes_per_launch": rr["algorithmic_bytes_per_launch"],
                                  "us_per_launch": rr["us_per_launch"], "achieved": rr["achieved"], "frac": rr["frac"]})
                line["roofline_spmv"]["sweep"] = sweep
                line["roofline_spmv"]["sweep_note"] = ("same kernel, inputs from L2-resident (10k-30k poses: 15-45 MB) to far beyond L2 "
                                                       "(1M poses: 1.5 GB); back-to-back launches, so the small sizes are served by L2")
        # ---- CPU restatement of the reference path on the host cores, bounded sample ----
        if not args.no_cpu:
            _, _, info = cpu_reference_steps(2 * CYCLE, 1)
            line["cpu_baseline"] = info
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    else:
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        outputs = {} if args.dump_outputs else None
        res = measure_multi(torch, dist, dp, pg, DATASET, MULTI_AGENTS, rank, world, local_rank, K, W, peak, peak_src, with_e2e=True,
                            outputs=outputs)
        tor = measure_multi(torch, dist, dp, pg, "torus3D", MULTI_AGENTS, rank, world, local_rank, K, W, peak, peak_src, with_e2e=False)
        if rank == 0:
            clocks = sampler.stop()
            line.update({
                "value": res["rounds_per_sec"], "ms_per_step": res["ms_per_round"], "steps": K,
                "config": dict(multi_config(DATASET, MULTI_AGENTS, res["colours"], f"{MULTI_AGENTS // world} agent(s) per GPU, one process per GPU"),
                               rounds=K, launch_mode=res["step_kernel_launch"] + ("; per rank one dpgo_agents_round_async call per round, replayed as a CUDA graph"
                                                                                 if res["concurrent_agents"] else "; eager launches on a side stream"),
                               concurrent_agents=res["concurrent_agents"], parallelism=f"agents{MULTI_AGENTS}/gpus{world}",
                               allgather_bytes_per_rank=res["allgather_bytes_per_rank"]),
                "rounds_per_sec": res["rounds_per_sec"], "agent_steps_per_sec": res["agent_steps_per_sec"],
                "e2e": res["e2e"], "gpu_launches": res["gpu_launches"], "clocks": clocks, "roofline": res["roofline"],
                "final": res["final"],
                "torus3D": {k2: tor[k2] for k2 in ("rounds_per_sec", "ms_per_round", "agent_steps_per_sec", "colours", "final",
                                                    "roofline", "allgather_bytes_per_rank", "concurrent_agents", "step_kernel_launch")},
            })
            print(json.dumps(line))
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)      # every rank writes the iterates of its own agents
        dist.destroy_process_group()


def measure_multi(torch, dist, dp, pg, dataset, k, rank, world, local_rank, K, W, peak, peak_src, with_e2e, outputs=None):
    """K timed coloured RBCD rounds of `dataset` split into k agents spread over `world` ranks (k/world agents per GPU).
    Returns rounds/s (max over ranks of the CUDA-event time), the per-rank roofline of the k_optimize launches of rank 0,
    and optionally the same rounds through the host-level API (host matrices in and out every round).
    outputs: if a dict, receives X_agent<a> = this rank's agents' iterates after the last timed round."""
    from dpo_b200.agent import DistributedPGO
    dev = torch.device("cuda", local_rank)
    edges, n = pg.read_g2o_file(os.path.join(ROOT, "data", dataset + ".g2o"))
    d = edges.d
    dh = d + 1
    X0 = pg.fixedStiefelVariable(d, RANK_R) @ pg.chordalInitialization(d, n, edges)
    distributed = world > 1

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    side = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(side):
        run = DistributedPGO(edges, n, k, r=RANK_R, schedule="coloured", X_init=X0, rank=rank if distributed else None,
                             world=world if distributed else None, device=local_rank, dist=dist if distributed else None)
    mine = run.local_ids
    X0d = {}
    for a in mine:
        cols = (run.glob[a][:, None] * dh + np.arange(dh)[None, :]).ravel()
        X0d[a] = torch.from_numpy(np.asfortranarray(X0[:, cols]).ravel(order="F").copy()).to(dev)
    cyc = CYCLE * run.ncolours

    launches = [0]

    def run_rounds(count, collect=None):
        steps = 0
        with torch.cuda.stream(side):
            for i in range(count):
                c = i % cyc
                if c == 0:
                    for a in mine:
                        run.agents[a].mProblem.copy_X_from_device(X0d[a].data_ptr())
                if run.concurrent:
                    # the active agents of this rank side by side (one thread-block cluster and one stream each): G rebuild ->
                    # RTR step -> pack per agent, then the all-gather; a reset of the iterates re-publishes all tiles
                    if c == 0:
                        run.exchange(build=False)
                    act = [a for a in range(run.k) if run.colour[a] == c % run.ncolours]
                    run._round_concurrent(act)
                    for a in mine:
                        if a in act:
                            steps += 1
                            launches[0] += 3
                            if collect is not None:
                                collect.append((a, run.agents[a].opt.fetch_result()))
                    continue
                run.exchange()
                launches[0] += 2 * len(mine)
                for a in mine:
                    if run.colour[a] == c % run.ncolours:
                        run.agents[a].opt.optimize_resident_async()
                        steps += 1
                        launches[0] += 1
                        if collect is not None:
                            collect.append((a, run.agents[a].opt.fetch_result()))
        return steps

    trail = []
    run_rounds(cyc, trail)                                # correctness / byte accounting trail of one cycle (also warms up)
    run_rounds(max(W, cyc))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with torch.cuda.stream(side):
        e0.record()
    launches[0] = 0
    my_steps = run_rounds(K)
    timed_launches = launches[0]
    with torch.cuda.stream(side):
        e1.record()
    barrier()
    if outputs is not None:
        for a in mine:
            outputs[f"X_agent{a:02d}"] = run.agents[a].mProblem.download_X()
    t = torch.tensor([e0.elapsed_time(e1), float(my_steps)], dtype=torch.float64, device=dev)
    tmax, tsum = t.clone(), t.clone()
    if distributed:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    ms_total, total_steps = float(tmax[0]), float(tsum[1])
    with torch.cuda.stream(side):
        st = run.step(evaluate=True)
    # roofline of this rank's k_optimize launches: algorithmic bytes of one cycle / its share of the timed region
    alg = 0.0
    for a, rs in trail:
        pr = run.agents[a].mProblem
        alg += rs.spmv_passes * pr.spmv_algorithmic_bytes(True) + rs.precond_applies * pr.precond_algorithmic_bytes(dp.PRECOND_SPARSE_EXACT)
    alg_per_round = alg / cyc
    ach = alg_per_round / (ms_total / K * 1e-3) / 1e9
    out = {"rounds_per_sec": K / (ms_total * 1e-3), "ms_per_round": ms_total / K, "agent_steps_per_sec": total_steps / (ms_total * 1e-3),
           "colours": run.ncolours, "allgather_bytes_per_rank": run.plan.pmax * RANK_R * dh * 8 * (k // world),
           "gpu_launches": int(timed_launches), "final": {"cost": st.cost, "gradnorm": st.gradnorm},
           "agents_per_gpu": len(mine), "concurrent_agents": bool(run.concurrent),
           "step_kernel_launch": ("one thread-block cluster of %d CTAs per agent, the round's agents side by side on their own streams"
                                  if run.concurrent else "cooperative grid of %d CTAs, one agent at a time") % run.agents[mine[0]].mProblem.launch_info()[0],
           "roofline": {"kernel": "k_optimize<5,4> launches of rank 0 (its agents' RTR steps)", "bound": "hbm", "achieved": ach,
                        "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": ach / peak,
                        "algorithmic_bytes_per_round": alg_per_round, "traffic": None,
                        "note": "rank 0's launches of an average round against the whole round time (exchange included); the "
                                "agents' working sets are L2-resident, the rounds are latency-bound (grid-wide phases, launches, "
                                "the all-gather), so the HBM fraction is small by construction"}}
    if with_e2e:
        # the same rounds driven through the host-level API (host matrices in and out, public poses packed on the host,
        # H2D / all-gather / D2H inside the timed region)
        for a in mine:
            ag = run.agents[a]
            ag.mProblem.sync()
            cols = (run.glob[a][:, None] * dh + np.arange(dh)[None, :]).ravel()
            ag.X = np.array(X0[:, cols])
        run.round = 0
        with torch.cuda.stream(side):
            for _ in range(2 * run.ncolours):
                run.step_host()
        barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(side):
            for i in range(K):
                if i % cyc == 0:
                    for a in mine:
                        cols = (run.glob[a][:, None] * dh + np.arange(dh)[None, :]).ravel()
                        run.agents[a].X = np.array(X0[:, cols])
                    run.round = 0
                run.step_host()
        barrier()
        e2e_dt = time.perf_counter() - t0
        te = torch.tensor([e2e_dt], dtype=torch.float64, device=dev)
        if distributed:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        h2d, d2h = run.host_bytes_per_step()
        out["e2e"] = {"value": K / float(te[0]), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "rounds": K,
                      "api": "DistributedPGO.step_host(): per round every local agent's X from pinned host memory (H2D), device-side "
                             "exchange (pack -> all-gather -> G rebuild), RTR step of the active agents, their X back to the host (D2H)"
                             + ("; 3 C calls per round (dpgo_agents_host_io_async x2, dpgo_agents_round_async), each replayed as a CUDA graph"
                                if run.concurrent else "")}
    for a in mine:
        run.agents[a].mProblem.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-spmv", action="store_true", help="skip the synthetic SpMV roofline leg")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-multi", action="store_true", help="N = 1: skip the 8-agents-on-one-GPU leg")
    ap.add_argument("--no-sweep", action="store_true", help="N = 1: skip the SpMV size sweep")
    ap.add_argument("--precond", default="sparse", choices=["sparse", "dense"],
                    help="exact preconditioner implementation: nested-dissection block solve (default) or the dense inverse (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float64): "
                         "N = 1: X (the iterate, r x (d+1)n), f_opt, gradnorm_opt; N > 1: X_agent<a> per agent")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
