#!/usr/bin/env python
"""bench.py -- headline benchmark: IPM iterations/s (and KKT-solve / refactor ms).

Default workload: BASELINE.json config C4, the configuration the north star quotes its target on (block-angular
sparse QP, n = 1e6 variables, m = 1.5e6 rows, nnz(A) = 8e6; Zero + Nonneg cones).  `--workload c2|c3|c5|expmix`
selects the other configurations.

A "step" is one interior-point iteration = one pass of the hot path: cone
scaling update, KKT value update + static regularisation + numeric LDL^T
refactor, constant-rhs solve, affine + combined KKT solves (each with iterative
refinement), step lengths, iterate update.

  python bench.py --gpus N --steps K --warmup W          our CUDA path
  python bench.py --impl reference ...                   reference algorithm on the host CPU
  python bench.py ... --dump-outputs DIR                 also write the solution of the last timed solve as DIR/*.npy
                                                         (--impl reference: the iterate of its bounded CPU solve)

`value`  : K real iterations (after W untimed warm-up iterations) timed with CUDA
           events on the solver's stream, problem resident in HBM.
`e2e`    : the same metric through the public API from HOST buffers:
           create (equilibrate + order + symbolic analysis + H2D) + solve + solution D2H.
N > 1    : one process per GPU (torchrun).  Default: ONE problem, its LDL^T split over the N GPUs by elimination-tree
           subtrees (DESIGN.md section 6: cut roots' update matrices / vectors and the solution vector meet in NCCL
           all-gathers) -- "scaling": "strong", value = K / max-over-ranks time.  `--replicas`: one independent
           problem per rank (seed+rank), no data-path collective, "scaling": "weak", value = N*K / max time.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
DUMP_CAP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays, cap=DUMP_CAP_BYTES):
    """Write each array as out_dir/<name>.npy in float64, so that two builds can be compared output for output on the
    same seeded inputs.  Past `cap` bytes in all, every array is cut to a fixed, seeded sample of its entries."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64).reshape(-1) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > cap:
            keep = a.size * (cap - 4096 * len(arrays)) // total        # 4 KB per file leaves room for the .npy header
            a = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_workload(name, rank):
    from helpers import workloads
    if name == "c2":
        pr = workloads.random_sparse_qp(n=100_000, m=200_000, nnz_per_row=5, seed=1 + rank, window=200)
        desc = ("random sparse QP n=1e5 m=2e5 nnz(A)=1e6 (5/row, columns drawn inside a sliding 200-column "
                "window), Nonneg(2e5), seed=%d" % (1 + rank))
    elif name == "c2small":
        pr = workloads.random_sparse_qp(n=10_000, m=20_000, nnz_per_row=5, seed=1 + rank, window=200)
        desc = "random sparse QP n=1e4 m=2e4 nnz(A)=1e5, Nonneg, seed=%d" % (1 + rank)
    elif name == "c2u":
        # SURVEY 8(d)'s wording of C2 (columns of A drawn uniformly from all n columns: the KKT graph is an expander and the
        # factor essentially dense) at a tenth of the size -- at full size a single CPU refactorisation would take a day
        # (DESIGN.md section 7); the window variant above is the headline C2
        pr = workloads.random_sparse_qp(n=10_000, m=20_000, nnz_per_row=5, seed=1 + rank, window=None)
        desc = "random sparse QP n=1e4 m=2e4 nnz(A)=1e5, columns drawn uniformly (expander), Nonneg, seed=%d" % (1 + rank)
    elif name == "c3":
        pr = workloads.portfolio_socp(seed=2 + rank)
        desc = "portfolio SOCP 5000 assets, 200 SOC(26), seed=%d" % (2 + rank)
    elif name == "c4":
        pr = workloads.block_angular_qp(seed=3 + rank)
        desc = "block-angular sparse QP n=1e6 m=1.5e6, seed=%d" % (3 + rank)
    elif name == "c5":
        pr = workloads.block_sdp(seed=4 + rank)
        desc = "block-diagonal SDP: 500 PSD(20) + linear constraints, n=2e4, seed=%d" % (4 + rank)
    elif name == "expmix":
        pr = workloads.entropy_power_mix(k_exp=100_000, k_pow=50_000, n_eq=10, seed=6 + rank)
        desc = ("entropy maximisation + geometric-mean allocation: 1e5 exponential cones, 5e4 power cones, "
                "11 equality rows, seed=%d" % (6 + rank))
    else:
        raise SystemExit("unknown workload " + name)
    return pr, desc


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def aggregate_over_ranks(dist, world, steps_local, seconds_local, device=None):
    """Whole-job throughput: units processed by all ranks / max-over-ranks time (bench contract).
    Works with any torch.distributed backend (nccl on GPUs, gloo in the CPU tests)."""
    if world <= 1 or dist is None:
        return steps_local / seconds_local, seconds_local, steps_local
    import torch
    t = torch.tensor([seconds_local], dtype=torch.float64, device=device)
    k = torch.tensor([float(steps_local)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(k, op=dist.ReduceOp.SUM)
    return float(k.item()) / float(t.item()), float(t.item()), float(k.item())


def algorithmic_bytes(li, N, nnzK):
    """Bytes one launch sequence must move at minimum.  `survey`: SURVEY.md section 8(d) / BASELINE.md section 5, the
    reference's own data structures (CSC factor with indices: 24 B per entry of L over the two sweeps) -- the figure
    the roofline fraction is quoted on.  `stored`: what this implementation actually has to read (dense panels
    without indices, 8 B per STORED entry per sweep, zero padding of relaxed supernodes included)."""
    survey = {"refactor": 12 * nnzK + 12 * li.nnzL + 16 * N, "solve": 24 * li.nnzL + 96 * N}
    stored = {"refactor": 20 * nnzK + 8 * li.nnzL_stored + 16 * N, "solve": 2 * 8 * li.nnzL_stored + 40 * N}
    return survey, stored


def pin_rank(local_rank, local_world):
    """Give every rank of a multi-process run its own slice of the host cores (and thereby size the thread pools of
    the one-time analysis, csrc/symbolic.cpp host_threads()): ranks that each assume the whole box fight over it."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        if local_world <= 1 or len(cores) < 2 * local_world:
            return len(cores)
        per = len(cores) // local_world
        mine = cores[local_rank * per:(local_rank + 1) * per]
        os.sched_setaffinity(0, mine)
        return len(mine)
    except Exception:
        return os.cpu_count()


def run_ours(args, rank, world):
    import torch
    import clarabel_rs_b200 as cb
    dev_index = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(dev_index)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev_index))
    shard = world > 1 and not args.replicas
    # default for N > 1: ONE problem, its LDL^T split over the N GPUs (subtree sharding, DESIGN section 6); every rank
    # builds the same data and runs the same iterations.  --replicas: one independent problem per rank.
    host_threads = pin_rank(dev_index, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    pr, desc = load_workload(args.workload, 0 if shard else rank)
    P, q, A, b, cones = pr["P"], pr["q"], pr["A"], pr["b"], pr["cones"]
    n, m = P.shape[0], A.shape[0]
    h2d_bytes = (P.data.nbytes + P.indices.size * 4 + A.data.nbytes * 2 + A.indices.size * 8 + 8 * (n + m) * 2)

    # ---------------- e2e through the public API from host buffers ----------------
    # warm the process (CUDA module load, allocator pools) on a tiny problem so that the end-to-end number below
    # is the cost of a new problem in a running process, not of the first CUDA call
    from helpers import workloads as _wl
    _pw = _wl.random_sparse_qp(n=300, m=500, nnz_per_row=4, seed=99, window=40)
    for _ in range(0 if args.no_process_warmup else 2):
        _sw = cb.CudaSolver(_pw["P"], _pw["q"], _pw["A"], _pw["b"], _pw["cones"], device=dev_index)
        _sw.solve()
        _sw.close()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    # C2's sliding-window structure is a nested-dissection case; the other configs let the backend compare AMD and ND
    ordering = cb.ORDER_ND if args.workload.startswith("c2") else cb.ORDER_BEST
    solver = cb.CudaSolver(P, q, A, b, cones, ordering=ordering, device=dev_index,
                           shard=(world, rank) if shard else None)
    t_setup = time.perf_counter() - t0
    res = solver.solve()                      # includes the D2H of (x, z, s)
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    iters_e2e = res["iterations"]
    li = solver.linear_solver_info()
    info = solver.info
    d2h_bytes = 8 * (n + 2 * m)

    # ---------------- device-resident K iterations after W warm-up iterations ----------------
    W, K = args.warmup, args.steps
    clocks = ClockSampler(dev_index)
    launches0 = cb.launch_count()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks.start()
    durations, launches_timed, first = [], 0, True
    status_all = [res["status"]]
    while len(durations) < K:
        l0 = cb.launch_count()
        r = solver.solve()
        l1 = cb.launch_count()
        status_all.append(r["status"])
        d = np.diff(solver.iter_ms)[:r["iterations"]]      # per-iteration device time (ms)
        if len(d) == 0:
            raise SystemExit("solver made no iterations")
        per_iter_launch = (l1 - l0) / max(len(d), 1)
        if first:
            d = d[W:] if len(d) > W else d[-1:]
            first = False
        take = d[:K - len(durations)]
        durations.extend(take.tolist())
        launches_timed += int(per_iter_launch * len(take))
    torch.cuda.synchronize()
    # re-solve with new data on the same handle (DefaultSolver::update_data): host buffers in, solution out,
    # symbolic analysis / plans / equilibration reused -- the parametric (MPC-style) use of the backend
    t_r0 = time.perf_counter()
    solver.update_data(P=P, q=q * 1.01, A=A, b=b)
    r_re = solver.solve()
    torch.cuda.synchronize()
    t_resolve = time.perf_counter() - t_r0
    if world > 1:
        dist.barrier()
    clk = clocks.stop()
    t_local = float(np.sum(durations)) / 1e3
    value, t_max, _ = aggregate_over_ranks(dist, world, K, t_local, "cuda")
    e2e_value, t_e2e, _ = aggregate_over_ranks(dist, world, iters_e2e, t_e2e, "cuda")
    if shard:      # one job, not N: the units are not summed over the ranks
        value, e2e_value = value / world, e2e_value / world
        # the kernel-level timings below are collective in a sharded run: every rank takes part
        shard_ms = (solver.time_ms("refactor", 5), solver.time_ms("ldl_solve", 20), solver.time_ms("kkt_solve", 5))

    out = None
    if rank == 0:
        # ---------------- kernel-level timings + roofline (live, CUDA events) ----------------
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        if shard:
            refactor_ms, ldl_solve_ms, kkt_solve_ms = shard_ms
        else:
            refactor_ms = solver.time_ms("refactor", 5)
            ldl_solve_ms = solver.time_ms("ldl_solve", 20)
            kkt_solve_ms = solver.time_ms("kkt_solve", 5)
        b_survey, b_stored = algorithmic_bytes(li, solver.N, int(info.nnzK))
        b_ref, b_sol = b_survey["refactor"], b_survey["solve"]
        solves_per_iter = info.n_ldl_solve / max(info.n_refactor, 1)
        share_ref = refactor_ms
        share_sol = ldl_solve_ms * solves_per_iter
        acct = ("algorithmic bytes per SURVEY.md 8(d): %s; the bytes this implementation has to read "
                "(dense panels, padding included) are in algorithmic_bytes_stored / frac_stored")
        rf_ref = {"kernel": "k_factor_level (tree level 0) + k_factor_df + k_invert_pivots: one numeric LDL^T refactor", "bound": "hbm",
                  "achieved": b_ref / (refactor_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                  "frac": b_ref / (refactor_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                  "algorithmic_bytes": b_ref, "algorithmic_bytes_stored": b_stored["refactor"],
                  "frac_stored": b_stored["refactor"] / (refactor_ms * 1e-3) / 1e9 / hbm_peak,
                  "accounting": acct % "12 nnzK + 12 nnzL + 16 N", "ms": refactor_ms, "share_of_step_ms": share_ref,
                  "fp64_gflops": li.flops / (refactor_ms * 1e-3) / 1e9, "peak_source": peak_src}
        rf_sol = {"kernel": "k_solve2<fwd> + k_solve2<bwd> (+ leaf kernels, permutation): one LDL solve, both sweeps", "bound": "hbm",
                  "achieved": b_sol / (ldl_solve_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                  "frac": b_sol / (ldl_solve_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                  "algorithmic_bytes": b_sol, "algorithmic_bytes_stored": b_stored["solve"],
                  "frac_stored": b_stored["solve"] / (ldl_solve_ms * 1e-3) / 1e9 / hbm_peak,
                  "accounting": acct % "24 nnzL + 96 N", "ms": ldl_solve_ms, "share_of_step_ms": share_sol,
                  "peak_source": peak_src}
        # DRAM traffic per launch from the committed ncu --set full capture of this workload (profiles/), if any
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json"))).get(args.workload, {})
            rf_ref["traffic"] = tr.get("refactor_dram_bytes")
            rf_sol["traffic"] = tr.get("solve_dram_bytes")
            rf_ref["traffic_source"] = rf_sol["traffic_source"] = tr.get("source")
        except Exception:
            pass
        # `roofline` is the triangular-solve launch sequence: the kernel the north star's roofline target names, and half
        # of the step together with the refactor (the two shares are within a few per cent of each other on C2 and C4)
        dominant, other = rf_sol, rf_ref
        rf_sol["share_of_step"] = share_sol / max(share_sol + share_ref, 1e-30)
        rf_ref["share_of_step"] = share_ref / max(share_sol + share_ref, 1e-30)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline(pr, args.workload, sample_iters=args.cpu_sample_iters, perm=solver.kkt_perm())
        out = {
            "metric": "ipm_iterations_per_sec", "value": value, "unit": "iterations/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": 1e3 * t_max / K, "higher_is_better": True,
            "scaling": "strong" if shard else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc, "n": n, "m": m, "nnzA": int(A.nnz), "nnzP_triu": int(P.nnz),
                       "kkt_dim": solver.N, "nnzK": int(info.nnzK), "nnzL": int(li.nnzL),
                       "nnzL_stored": int(li.nnzL_stored), "levels": int(li.n_levels),
                       "supernodes": int(li.n_supernodes), "ordering": "nested dissection (hub separators, AMD leaves)",
                       "host_threads_per_rank": host_threads,
                       "cache": "working set larger than L2 (factor panels %.0f MB)" % (li.nnzL_stored * 8 / 1e6),
                       "parallelism": ("one problem, subtree-sharded LDL x%d (NCCL all-gather of cut-root update matrices / vectors and of x)" if shard else "replicas x%d") % world},
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "iterations/s", "h2d_bytes_per_step": h2d_bytes / max(iters_e2e, 1),
                    "d2h_bytes_per_step": d2h_bytes / max(iters_e2e, 1), "setup_s": t_setup,
                    "total_s": t_e2e, "iterations": iters_e2e,
                    "note": "create (equilibrate+order+symbolic+H2D) + solve + solution D2H, from host numpy buffers"},
            "e2e_resolve": {"value": r_re["iterations"] / t_resolve, "unit": "iterations/s", "total_s": t_resolve,
                            "iterations": r_re["iterations"], "status": r_re["status"],
                            "note": "update_data(P, q, A, b from host) + solve + solution D2H on the existing handle"},
            "gpu_launches": launches_timed,
            "roofline": dominant, "roofline_other": other,
            "kkt_solve_ms": kkt_solve_ms, "ldl_solve_ms": ldl_solve_ms, "refactor_ms": refactor_ms,
            "other_ms_per_step": max(0.0, 1e3 * t_max / K - refactor_ms - ldl_solve_ms * solves_per_iter) if not shard else None,
            "collectives": ({"transport": "stream-ordered ncclAllGather issued by the library" if getattr(solver, "nccl_direct", False) else "torch.distributed all_gather_into_tensor (callback)",
                             "count_total": int(cb._lib2().cipm_collective_count(solver._h))} if shard else None),
            "ldl_solves_per_iteration": solves_per_iter,
            "status": status_all[0], "iterations": iters_e2e,
            "cpu_baseline": cpu,
        }
    solver.close()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: r[k] for k in ("x", "z", "s")})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


def one_core():
    """Pin the calling process to one core for the single-thread CPU legs (BASELINE.md section 3); returns a restore function."""
    try:
        old = os.sched_getaffinity(0)
        os.sched_setaffinity(0, {sorted(old)[len(old) // 2]})
        return lambda: os.sched_setaffinity(0, old)
    except Exception:
        return lambda: None


def cpu_solve(pr, workload, max_iter, perm=None):
    """Reference algorithm on the host: oracle IPM + oracle qdldl (line-faithful C port, oracle/), ONE thread pinned to
    one core.  Ordering: the reference orders with AMD at dense-scale 1.5 (the `amd` crate is not vendored; the
    repo's own AMD stands in).  On C4 that ordering costs the CPU 2.7e12 flops per refactorisation (about half an
    hour, measured once: profiles/r02_cpu_c4_amd_container.json), so the CPU leg there gets the nested-dissection
    ordering the GPU path uses -- 1.5e10 flops, the cheapest ordering known for the reference algorithm: a
    conservative baseline."""
    import clarabel_rs_b200 as cb
    import oracle
    os.environ.setdefault("ORACLE_NATIVE", "1")       # -O3 -march=native build of the port on this host, if gcc is here
    t0 = time.perf_counter()
    ipm = oracle.IPM(pr["P"], pr["q"], pr["A"], pr["b"], pr["cones"],
                     settings=oracle.default_settings(max_iter=max_iter))
    N, cp, rv, _, _ = ipm.kkt()
    if workload == "c4":
        order = "nested dissection (the GPU path's ordering; the reference's own AMD costs 180x the flops here)"
        if perm is None:
            perm = cb.SymbolicAnalysis(N, cp, rv, ordering=cb.ORDER_ND).perm
    elif workload == "c5":
        # plain AMD smears the 500 dense 210 x 210 Hs blocks into each other (nnzL 4.9e9): the CPU leg gets the block-aware
        # ordering of the GPU path (every dense block contracted to one vertex, csrc/symbolic.cpp order_with_groups)
        order = "block-aware minimum degree (the GPU path's ordering; plain AMD gives nnzL 4.9e9 here)"
        if perm is None:
            perm = cb.order_groups(N, cp, rv, pr["cones"], pr["P"].shape[0])
    else:
        order = "AMD (dense scale 1.5)"
        perm = cb.order(N, cp, rv, cb.ORDER_AMD, 1.5)
    ipm.set_perm(perm)
    t_setup = time.perf_counter() - t0
    restore = one_core()
    try:
        r = ipm.solve()
    finally:
        restore()
    t_total = time.perf_counter() - t0
    return ipm, r, t_setup, t_total, order


def cpu_baseline(pr, workload, sample_iters=0, perm=None):
    if sample_iters <= 0:
        sample_iters = 2 if workload in ("c4", "c5") else 3
    ipm, r, t_setup, t_total, order = cpu_solve(pr, workload, sample_iters, perm)
    i = r["info"]
    return {"value": r["iterations"] / i.solve_time, "unit": "iterations/s", "cores": 1, "kind": "port",
            "sample": "first %d IPM iterations of the same problem (oracle IPM + oracle qdldl, 1 pinned thread); ordering: %s"
                      % (r["iterations"], order),
            "host_cores_available": os.cpu_count(), "solve_s": i.solve_time, "setup_s": t_setup,
            "refactor_ms": 1e3 * i.t_kkt_update / max(i.n_refactor, 1), "nnzL": int(i.nnzL),
            "kkt_solve_ms": 1e3 * i.t_kkt_solve / max(2 * r["iterations"], 1), "oracle_build": _oracle_build()}


def _oracle_build():
    try:
        import oracle
        return oracle.build_flags()
    except Exception:
        return None


def run_reference(args, rank, world):
    if rank != 0:
        return None
    pr, desc = load_workload(args.workload, 0)
    W, K = args.warmup, args.steps
    # bounded sample: the whole arm has to end within a few minutes; an iteration of the port costs ~12 s on C4
    cap = {"c4": 6, "c5": 4}.get(args.workload, W + K)
    ipm, r, t_setup, t_total, order = cpu_solve(pr, args.workload, min(W + K, cap))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: r[k] for k in ("x", "z", "s")})
    i = r["info"]
    iters = r["iterations"]
    value = iters / i.solve_time
    return {
        "impl": "reference", "metric": "ipm_iterations_per_sec", "value": value, "unit": "iterations/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": 1e3 * i.solve_time / max(iters, 1),
        "higher_is_better": True, "scaling": "strong" if (world > 1 and not args.replicas) else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "n": ipm.n, "m": ipm.m, "kkt_dim": ipm.N, "nnzK": int(i.nnzK),
                   "nnzL": int(i.nnzL), "ordering": order, "parallelism": "1 host thread"},
        "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": 1, "kind": "port",
                         "sample": "first %d IPM iterations (min(W+K, %d)) of the same problem; the reference is Rust "
                                   "and cannot be built here, so this is the line-faithful C port (oracle/), one pinned thread"
                                   % (iters, cap),
                         "host_cores_available": os.cpu_count(), "setup_s": t_setup,
                         "refactor_ms": 1e3 * i.t_kkt_update / max(i.n_refactor, 1),
                         "kkt_solve_ms": 1e3 * i.t_kkt_solve / max(2 * iters, 1), "oracle_build": _oracle_build()},
        "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "iterations": iters, "status": r["status"],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4")
    ap.add_argument("--cpu-sample-iters", type=int, default=0, help="0 = per workload (2 on c4, 3 elsewhere)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--shard", action="store_true", help="(default for --gpus N > 1; kept for old command lines)")
    ap.add_argument("--replicas", action="store_true",
                    help="with --gpus N > 1: N independent problems (weak scaling) instead of ONE problem split over the N GPUs")
    ap.add_argument("--no-process-warmup", action="store_true",
                    help="skip the tiny warm-up problem (for ncu launch lists: keeps the capture on the workload)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write x, z and s of the last timed solve as DIR/<name>.npy (float64); "
                         "with --impl reference: the iterate where its bounded solve stopped (min(W+K, 6) iterations "
                         "on c4, min(W+K, 4) on c5), which is not converged and so not comparable with the CUDA arm's")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    import __graft_entry__
    if not (os.path.exists(os.path.join(ROOT, "clarabel.rs_b200", "libclarabel_b200.so"))
            and os.path.exists(os.path.join(ROOT, "oracle", "liboracle.so"))):
        if rank == 0:
            __graft_entry__.build()
    # libraries (NCCL, torchrun) may write banners to stdout: keep fd 1 clean for the ONE JSON line
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        out = run_reference(args, rank, world) if args.impl == "reference" else run_ours(args, rank, world)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    if rank == 0 and out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the benchmark writes nothing into the source tree (it may be read-only)
    main()
