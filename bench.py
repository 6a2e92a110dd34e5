#!/usr/bin/env python
"""bench.py -- headline metric of BASELINE.json: IPM iterations/sec (+ ms/factorize) on the OPF-10k condensed KKT (fp64).

A "step" = one pass of the hot path over one synthetic interior-point iterate, in the call order of MadNLP's
`regular!` (src/IPM/solver.jl:216-298): compress_jacobian!/compress_hessian! -> set_aug_diagonal! -> build_kkt! ->
factorize! -> inertia -> [regularise + refactor while the inertia is wrong] -> Richardson(solve_kkt! + KKT mat-vec).
Workload: synthetic AC-OPF with the (nbus, nbranch, ngen) counts of pglib case10000_goc (no pglib data offline),
SparseCondensedKKTSystem, 24 distinct iterates (mu: 1e-1 -> 1e-9) cycled; iterate NONCONVEX_AT is nonconvex (wrong inertia
at first) so the regularise -> refactor branch of inertia_correction! runs inside the timed region.

  value : steps/sec with the iterate's inputs already resident in HBM (device-to-device staging only)
  e2e   : same metric through the host-facing path: inputs in pinned HOST memory, H2D of (jac, hess, reg, du_diag,
          l_diag, u_diag, l_lower, u_lower, rhs) and D2H of the step direction d INSIDE the timed region, every step.
          Pipelined (ipm.HostIteratePipeline): the H2D of iterate i+1 and the D2H of direction i-1 run on copy streams
          while step i computes; ONE pair of CUDA events brackets the K steps (pipeline fill, every copy, the final
          drain AND the L2 flush writes are inside it).  `e2e.serial` is the unpipelined figure (copy -> step -> copy,
          per-step events, flush untimed) for callers whose next iterate depends on this step's result.
  --impl reference : the CPU restatement of the reference's path (oracle: the reference's scalar assembly loops in C +
          `LDLSolver` = Davis' LDL^T, sequential like the reference) on the same workload, same --steps/--warmup
  secondary : configs[1], [2], [4] of BASELINE.json measured in the same run (N = 1), and the sharded C5 factorisation (N > 1)

Timing: every step is bracketed by CUDA events on the launching stream; between steps (untimed) L2 is flushed by
writing a 256 MiB buffer; the K steps are bracketed by barrier + synchronize; multi-GPU = max over ranks.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "ipm_iters_per_sec"
UNIT = "iter/s"
N_ITERATES = 24
NONCONVEX_AT = 11
FIELDS = ("jac", "hess", "reg", "du_diag", "l_diag", "u_diag", "l_lower", "u_lower", "rhs")
# below this many flops per factorisation the elimination tree is not sharded: every rank runs the whole (latency-bound)
# factorisation itself, because one NVLink round trip costs more than the work it would save (measured: DESIGN.md section 6)
SHARD_MIN_FLOPS = float(os.environ.get("B2_SHARD_MIN_FLOPS", 2e9))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=240)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="case10000_goc")
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--cpu-sample-steps", type=int, default=60)
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--force-shard", action="store_true", help="shard the elimination tree even below SHARD_MIN_FLOPS")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (step direction, inertia) as DIR/<name>.npy, "
                         "float64; the workload is seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def dump_outputs(dirname, arrays):
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def load_workloads():
    """workloads.py is plain numpy; loaded by PATH so that the reference arm never imports the package (whose __init__
    loads libb200kkt.so)"""
    name = "b2_workloads_standalone"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "madnlp.jl_b200", "workloads.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def make_workload(name):
    W = load_workloads()
    model, st = W.acopf_case(name)
    its = W.ipm_iterates(model, st, N_ITERATES, seed=0)
    bad = W.ipm_iterates(model, st, 1, seed=2, y_scale=1e2, eq_box=(1e-1, 1.0))[0]
    bad.mu = its[NONCONVEX_AT].mu
    its[NONCONVEX_AT] = bad
    return model, st, its


def config_of(args, st, world):
    """identical for both arms (it depends on the arguments and the workload only)"""
    return {"workload": f"acopf_{args.workload}_synthetic_condensed_kkt", "kkt": "SparseCondensedKKTSystem",
            "n": int(st.nvar), "m": int(st.ncon), "iterates": N_ITERATES, "nonconvex_iterates": [NONCONVEX_AT],
            "l2": "flushed between steps (256 MiB write, untimed)" if not args.no_flush else "not flushed",
            "parallelism": (f"{world} GPU(s): elimination tree sharded by subtrees when flops/factorisation >= {SHARD_MIN_FLOPS:.0e}; below it "
                            "(this workload) replicas only -- one independent IPM instance per GPU, no data-path collective, value = all ranks' iterations / s")}


# ----------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """samples nvidia-smi SM clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)"""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

        def run():
            # one nvidia-smi process in loop mode (a sample every 20 ms: the timed region is ~0.7 s); if that does not produce
            # lines (old driver), fall back to one process per sample
            try:
                self._proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "20"],
                                              stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                for line in self._proc.stdout:
                    if self._stop.is_set():
                        break
                    line = line.strip()
                    if line:
                        self.rows.append([x.strip() for x in line.split(",")])
            except Exception:
                pass
            looped = bool(self.rows)
            while not self._stop.is_set() and not looped:
                try:
                    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                         capture_output=True, text=True, timeout=5).stdout.strip()
                    if out:
                        self.rows.append([x.strip() for x in out.split(",")])
                except Exception:
                    pass
                self._stop.wait(0.02)
        self._proc = None
        self._t = threading.Thread(target=run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if getattr(self, "_proc", None) is not None:
            try:
                self._proc.terminate()
            except Exception:
                pass
        if self._t:
            self._t.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 2 + k and r[2 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------- CPU legs (oracle)
def _cpu_replay(st):
    """the reference's CPU path restated: scalar assembly loops (C), LDLSolver (src/LinearSolvers/ldl.jl over Davis' LDL^T, C),
    Richardson + inertia correction (oracle/madnlp_oracle.py::IPMLinearAlgebraCPU).  Sequential, like the reference."""
    import madnlp_oracle as o
    cb = o.Callback(st.nvar, st.ncon, st.jac_I, st.jac_J, st.hess_I, st.hess_J, st.ind_ineq, st.ind_lb, st.ind_ub)
    kkt = o.SparseCondensedKKTSystem(cb, o.LDLSolver)
    kkt.initialize()
    return o.IPMLinearAlgebraCPU(kkt)


def _cpu_run(la, its, warm, steps):
    for i in range(warm):
        la.load_iterate(its[i % len(its)]); assert la.step(mu=its[i % len(its)].mu)
    la.t_factorize = 0.0
    f0 = la.cnt["factorizations"]
    t0 = time.perf_counter()
    for i in range(steps):
        it = its[(warm + i) % len(its)]
        la.load_iterate(it)
        assert la.step(mu=it.mu)
    dt = time.perf_counter() - t0
    return dt, 1e3 * la.t_factorize / max(1, la.cnt["factorizations"] - f0)


CPU_KIND_NOTE = ("oracle port: the reference's scalar assembly/vector loops and its LDLSolver (LDLFactorizations.jl = Davis' LDL^T, "
                 "minimum-degree ordering) restated in C, Richardson + inertia correction in Python; sequential like the reference "
                 "(blas_num_threads = 1 default, src/options.jl:127; fronts <= 47 leave BLAS threads nothing to do)")


def _all_cores_worker(args_tuple):
    name, steps = args_tuple
    model, st, its = make_workload(name)
    la = _cpu_replay(st)
    dt, _ = _cpu_run(la, its, 1, steps)
    return dt


def cpu_all_cores_throughput(name, steps=6):
    """what ALL host cores can deliver on this workload: one independent IPM replay per core (the factorisation itself is
    sequential in the reference), aggregate steps/s.  Not a single-problem speed: a throughput ceiling for context."""
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        dts = pool.map(_all_cores_worker, [(name, steps)] * cores)
    return {"value": cores * steps / max(dts), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{cores} independent replays x {steps} steps in parallel (one per core); aggregate steps/s over the slowest",
            "wall_s": time.perf_counter() - t0}


def run_reference(args, rank, world):
    """--impl reference: rank 0 only; honours --steps/--warmup."""
    if rank != 0:
        return
    model, st, its = make_workload(args.workload)
    la = _cpu_replay(st)
    dt, ms_fac = _cpu_run(la, its, args.warmup, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"direction": la.d.full(), "inertia": la.last_inertia})
    val = args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "ms_per_factorize": ms_fac, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(args, st, args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": f"{args.steps} IPM steps of the same workload; " + CPU_KIND_NOTE},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "counters": la.cnt, "nnz_l_cpu": la.kkt.linear_solver.nnz_l,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_sample(args, st, its):
    la = _cpu_replay(st)
    nstep = max(1, args.cpu_sample_steps)
    dt, ms_fac = _cpu_run(la, its, 2, nstep)
    out = {"value": nstep / dt, "unit": UNIT, "cores": 1, "kind": "port", "ms_per_factorize": ms_fac,
           "sample": f"{nstep} IPM steps of the same workload; " + CPU_KIND_NOTE}
    try:
        out["all_cores"] = cpu_all_cores_throughput(args.workload)
    except Exception as e:      # never let the context number break the bench line
        out["all_cores"] = {"error": repr(e)}
    return out


# ----------------------------------------------------------------------------------------------------- B200 arm
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import madnlp_jl_b200 as pkg
    from madnlp_jl_b200 import kkt as K
    from madnlp_jl_b200.ipm import IPMLinearAlgebra

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model, st, its = make_workload(args.workload)

    class CB:
        pass
    cb = CB()
    cb.nvar, cb.ncon = st.nvar, st.ncon
    cb.jac_I, cb.jac_J, cb.hess_I, cb.hess_J = st.jac_I, st.jac_J, st.hess_I, st.hess_J
    cb.ind_ineq, cb.ind_lb, cb.ind_ub = st.ind_ineq, st.ind_lb, st.ind_ub

    opt = pkg.capi.default_options()
    for env, field in (("B2_FUSE_MAX", "fuse_max_fronts"), ("B2_DEP", "dep_schedule"), ("B2_NEMIN", "nemin")):
        if os.environ.get(env):
            setattr(opt, field, int(os.environ[env]))
    sharded = False
    if world > 1:
        # decide from the symbolic analysis whether sharding the tree can pay at all
        probe = K.create_kkt_system(K.SparseCondensedKKTSystem, cb, None, opt)
        flops = probe.linear_solver.stats()["flops"]
        sharded = args.force_shard or flops >= SHARD_MIN_FLOPS
        if sharded:
            from madnlp_jl_b200.parallel import DistributedSparseSolver
            del probe
            kkt = K.create_kkt_system(K.SparseCondensedKKTSystem, cb,
                                      lambda csc, o_: DistributedSparseSolver(csc, o_, rank=rank, world=world), opt)
        else:
            kkt = probe
    else:
        kkt = K.create_kkt_system(K.SparseCondensedKKTSystem, cb, None, opt)
    kkt.initialize()
    la = IPMLinearAlgebra(kkt, use_cuda_graph=(not sharded and not os.environ.get("B2_NO_STEP_GRAPH")))
    stats = kkt.linear_solver.stats()

    host = [{k: torch.from_numpy(np.ascontiguousarray(getattr(it, k))).pin_memory() for k in FIELDS} for it in its]
    devit = [{k: v.to(dev) for k, v in h.items()} for h in host]
    h2d_bytes = sum(v.numel() * 8 for v in host[0].values())
    d_host = torch.zeros(la.d.values.numel(), dtype=torch.float64).pin_memory()
    d2h_bytes = d_host.numel() * 8
    flush_buf = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream()

    def time_phase(fn, reps=10):
        """median CUDA-event time of one call, L2 flushed before each repeat"""
        ts = []
        for _ in range(reps):
            if not args.no_flush:
                flush_buf.fill_(1.0)
            a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
            a0.record(stream); fn(); a1.record(stream); a1.synchronize()
            ts.append(a0.elapsed_time(a1))
        return float(np.median(ts))

    def one_step(i, e2e):
        if not args.no_flush:
            flush_buf.fill_(1.0)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        if e2e:
            la.load_iterate_host(host, i % N_ITERATES)
        else:
            la.load_iterate(devit[i % N_ITERATES])
        ok = la.step(mu=its[i % N_ITERATES].mu)
        if e2e:
            d_host.copy_(la.d.values, non_blocking=True)
        e1.record(stream)
        e1.synchronize()
        assert ok
        return e0.elapsed_time(e1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_run(e2e):
        for i in range(args.warmup):
            one_step(i, e2e)
        barrier()
        t0 = time.perf_counter()
        ms = [one_step(args.warmup + i, e2e) for i in range(args.steps)]
        barrier()
        wall = time.perf_counter() - t0
        tot = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        return float(tot.item()), wall

    from madnlp_jl_b200.ipm import HostIteratePipeline
    pipe = HostIteratePipeline(la, FIELDS)

    def pipelined_steps(first, count):
        """`count` host-facing steps; copies of neighbouring steps overlap the compute; returns device ms for all of them and
        the index of the pinned host buffer that holds the last step's direction"""
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        slot = pipe.prefetch(host[first % N_ITERATES])
        if not args.no_flush:
            flush_buf.fill_(1.0)                          # (inside the timed region here)
        hs = None
        for j in range(count):
            i = first + j
            pipe.load(slot)
            nxt = [None]
            if j + 1 < count:
                # the next iterate's H2D copies are queued while this step's assembly + factorisation run
                def queue_next(i=i):
                    nxt[0] = pipe.prefetch(host[(i + 1) % N_ITERATES])
            else:
                queue_next = None
            ok = la.step(mu=its[i % N_ITERATES].mu, after_prologue=queue_next)
            assert ok
            if not args.no_flush and j + 1 < count:
                flush_buf.fill_(1.0)                      # L2 flush between steps, queued first so that it runs under the host's hand-over work
            hs = pipe.push_result()
            slot = nxt[0]
        pipe.drain()
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1), hs

    def timed_pipelined():
        pipelined_steps(0, args.warmup)
        barrier()
        t0 = time.perf_counter()
        ms, hs = pipelined_steps(args.warmup, args.steps)
        barrier()
        wall = time.perf_counter() - t0
        tot = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        return float(tot.item()), wall, hs

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    dev_ms, dev_wall = timed_run(False)
    cnt_dev = dict(la.cnt)
    if args.dump_outputs:
        outputs = {"direction": la.d.values.cpu().numpy(), "inertia": la.last_inertia}
    ser_ms, ser_wall = timed_run(True)
    e2e_ms, e2e_wall, e2e_slot = timed_pipelined()
    assert pipe.h2d_bytes == h2d_bytes and pipe.d2h_bytes == d2h_bytes
    if args.dump_outputs and rank == 0:
        outputs["direction_e2e"] = pipe.d_host[e2e_slot].numpy()
        dump_outputs(args.dump_outputs, outputs)

    # phase timings of the hot path's three metrics (SURVEY 8d M1/M2), measured separately from the step loop
    la.load_iterate(devit[0])
    def assemble():
        kkt.compress_jacobian(); kkt.compress_hessian(); kkt.set_aug_diagonal_(); kkt.build_kkt()
    xsol = torch.randn(kkt.n, dtype=torch.float64, device=dev)
    asm_ms = time_phase(assemble)
    fac_ms = time_phase(kkt.linear_solver.factorize)
    sol_ms = time_phase(lambda: kkt.linear_solver.solve_linear_system(xsol))
    clocks = sampler.stop() if sampler else None
    stats = kkt.linear_solver.stats()          # (launch counts are known once the sweeps have been issued)

    secondary = None
    if not args.no_secondary:
        secondary = run_secondary(args, rank, world, dev)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        # algorithmic bytes (SURVEY.md 8d): numeric factorisation 8*(nnz K + nnz L); one solve 2 sweeps x (8+4) B x nnz L
        alg_bytes = 8.0 * (stats["nnz_a"] + stats["nnz_l"])
        achieved = alg_bytes / (fac_ms * 1e-3) / 1e9 if fac_ms else None
        sol_bytes = 24.0 * stats["nnz_l"]
        sol_ach = sol_bytes / (sol_ms * 1e-3) / 1e9 if sol_ms else None
        # replicas (tree not sharded): every rank runs its own IPM instance -> the job processed world x steps iterations
        units = args.steps * (1 if sharded else world)
        value = units / (dev_ms * 1e-3)
        e2e_val = units / (e2e_ms * 1e-3)
        nfac = max(1, cnt_dev["factorizations"])
        solves = cnt_dev["backsolves"] / nfac
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.workload if world == 1 else "", None)
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong" if sharded else "weak",
            "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config_of(args, st, world),
            "solver": {"nnz_kkt": stats["nnz_a"], "nnz_l": stats["nnz_l"], "factor_flops": stats["flops"], "supernodes": stats["n_supernodes"],
                       "levels": stats["n_levels"], "max_front": stats["max_front"], "tree_sharded": bool(sharded),
                       "refinement_solves_per_factorization": solves,
                       "factorizations_per_step": cnt_dev["factorizations"] / float(args.steps + args.warmup)},
            "ms_per_factorize": fac_ms, "ms_per_assemble": asm_ms, "ms_per_solve": sol_ms,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": e2e_ms / args.steps,
                    "mode": "pipelined: H2D of iterate i+1 / D2H of direction i-1 on copy streams during step i; one event pair "
                            "around the K steps, L2 flush writes inside the timed region",
                    "serial": {"value": units / (ser_ms * 1e-3), "ms_per_step": ser_ms / args.steps,
                               "mode": "copy -> step -> copy per step, per-step events, flush untimed"}},
            "per_replica_value": args.steps / (dev_ms * 1e-3),
            # own kernels per step: iterate load (1) + assembly (5) + numeric factorisation + start of the refinement (1) +
            # per refinement step: the triangular sweeps + pre/post/update/mul kernels (6)
            "gpu_launches": int((1 + (5 + stats["n_factor_launches"]) * (cnt_dev["factorizations"] / float(args.steps + args.warmup)) + 1
                                 + solves * (stats["n_solve_launches"] + 6)) * args.steps),
            "roofline": {"kernel": "numeric multifrontal LDL^T of the whole elimination tree (k_factor_dep, one launch)", "bound": "hbm",
                         "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": (achieved / hbm_peak) if achieved else None,
                         "traffic": traffic, "traffic_source": "profiles/traffic.json (ncu --set full dram read+write per launch)",
                         "algorithmic_bytes": alg_bytes, "peak_source": peak_src,
                         "note": "latency-bound: %d fronts of order <= %d in %d levels, %.3g Mflop" % (
                             stats["n_supernodes"], stats["max_front"], stats["n_levels"], stats["flops"] / 1e6)},
            "roofline_solve": {"kernel": "one solve_linear_system! (forward + diagonal + backward sweeps)", "bound": "hbm",
                               "achieved": sol_ach, "peak": hbm_peak, "unit": "GB/s", "frac": (sol_ach / hbm_peak) if sol_ach else None,
                               "algorithmic_bytes": sol_bytes},
            "clocks": clocks,
            "wall_s": {"device_resident": dev_wall, "e2e": e2e_wall, "e2e_serial": ser_wall},
            "counters": la.cnt,
        }
        if secondary is not None:
            line["secondary"] = secondary
        if world == 1 and args.cpu_sample_steps > 0:
            line["cpu_baseline"] = cpu_baseline_sample(args, st, its)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_secondary(args, rank, world, dev):
    """BASELINE.json configs[1], [2], [4] in the driver-run line (median of CUDA-event timings, L2 flushed; see
    tools/bench_configs.py) and, at N > 1, the subtree-sharded C5 factorisation (max over ranks)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    out = {}
    try:
        import bench_configs as BC
        if world == 1:
            out["fp64_peak_tflops"] = {"cublas_dgemm_8192": BC.dgemm_peak(), "dmma_issue_peak": 37.0,
                                       "note": "fp64 roofline denominators (MEASURED_PEAKS.json has none)"}
            out["c2_dense_n4096_m2048"] = BC.config2(cpu=True)
            out["c2_dense_n4096_m2048_neq256"] = BC.config2(n_eq=256, cpu=False, lib=False)
            out["c3_case1354_pegase"] = BC.config_sparse_opf("case1354_pegase")
            out["c5_grid_64"] = BC.config5(64)
        else:
            out["c5_grid_64_sharded"] = BC.config5_dist(64, rank, world)
    except Exception as e:
        import traceback
        out["error"] = repr(e) + " | " + traceback.format_exc(limit=3)
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
