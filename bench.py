#!/usr/bin/env python
"""bench.py — path-QP solves/s on B200 (contract in the task statement).

One "step" = one pass of the hot path (assemble + OSQP-style ADMM to the reference's
eps = 2e-3 + solution write-back, i.e. one `BaseSolver::solve` per instance) over one batch
of synthetic instances. Default workload: BASELINE.json configs[2] — batch 8192 paths,
240 knots, per-instance clearance bounds — per GPU (weak scaling: configs[3] = 8 x 8192).

  value      : solves/s, inputs resident in HBM, kernel launched through the C ABI's
               device-pointer entry point, CUDA events on the launching stream, max over ranks
  e2e        : same metric through the host-buffer C ABI call (pinned host buffers, H2D + D2H
               inside the timed region)
  roofline   : algorithmic bytes (SURVEY.md §8d: 104 n + 56 per cold solve) / kernel time vs the
               measured HBM peak (MEASURED_PEAKS.json)
  cpu_baseline: the oracle port (OSQP-algorithm restatement) on the host cores, bounded sample
  config.fp64 / config.secondary : the same metric with the FP64 instantiation of the kernel (the
               reference's OSQP is FP64), and the other BASELINE configs (configs[0] one path through
               the C++ drop-in incl. handle creation, configs[1] shared map, configs[4] receding horizon)

`--impl reference` times that CPU path alone (kind "port": OSQP itself is not available).
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from path_optimizer_2_b200 import abi, synthetic  # noqa: E402

METRIC = "path-QP solves/sec (N knots, batch B)"
UNIT = "solves/s"
CFG_ID = 3


# --------------------------------------------------------------------------------------- workloads
def make_workload(args, batch, first, device=None):
    """(HostBatch, description, extras) of `batch` instances starting at global index `first`.
    Shared-map workload: the clearance bounds come from the CUDA bounds kernel (pqp_bounds.h) on
    `device`; with device=None (the CPU reference arm) from the oracle's numpy restatement."""
    if args.workload == "sharedmap":
        from path_optimizer_2_b200 import sharedmap
        dmap = sharedmap.DistanceMap()
        lines = sharedmap.make_lines(batch, args.n, first=first, dmap=dmap)
        extras = {}
        if device is None:
            from oracle import bounds_oracle
            t0 = time.perf_counter()
            bnd = np.zeros((batch, 6, args.n))
            nv = np.zeros(batch, dtype=np.int32)
            for b in range(batch):
                bnd[b], nv[b] = bounds_oracle.update_bounds(dmap.dist, dmap.res, lines.spline_rows(b), *lines.states[b])
            extras["bounds_cpu_s"] = time.perf_counter() - t0
        else:
            extras = bounds_stage(args, dmap, lines, device)
            bnd, nv = extras.pop("bounds"), extras.pop("n_valid")
        hb = lines.to_host_batch(bnd, nv)
        extras["_lines"], extras["_dmap"] = lines, dmap  # for the front-end stages (popped before the line is printed)
        return hb, ("BASELINE configs[1] per GPU: batch %d paths x %d knots through ONE shared obstacle map "
                    "(gridmap.png distance layer; clearance bounds = updateBoundsImproved, "
                    "reference_path_impl.cpp:177-312), cold BaseSolver::solve (configs[0] is batch 1 of the "
                    "same)" % (batch, args.n)), extras
    hb = synthetic.make_batch(CFG_ID, batch, args.n, first=first)
    return hb, ("BASELINE configs[2] per GPU: batch %d paths, %d knots, per-instance clearance "
                "bounds, cold BaseSolver::solve (configs[3] = 8 GPUs x 8192)" % (batch, args.n)), {}


def bounds_stage(args, dmap, lines, device):
    """SURVEY.md §8 rows f-2 + f-1 on the GPU: reference states from the splines, then the
    clearance bounds, for the whole batch through the C ABI with device-resident buffers; timed
    with CUDA events on the launching stream and checked against the oracle on a sample."""
    import torch
    from oracle import bounds_oracle
    from path_optimizer_2_b200 import bounds
    dev = torch.device("cuda", device)
    pbn = bounds.PathBounds(dmap.dist, dmap.res, device=device)
    B, n = lines.batch, lines.n_max
    max_s = np.array([lines.spline_rows(b)[0, -1] for b in range(B)])
    d_spline, d_k, d_maxs = (torch.from_numpy(v).to(dev) for v in (lines.spline, lines.k, max_s))
    d_states = torch.zeros((B, 4, n), dtype=torch.float64, device=dev)
    d_curv = torch.zeros((B, n), dtype=torch.float64, device=dev)
    d_n, d_nv = (torch.zeros(B, dtype=torch.int32, device=dev) for _ in range(2))
    d_bounds = torch.zeros((B, 6, n), dtype=torch.float64, device=dev)
    si = bounds.StatesIn(B, n, lines.k_max, d_spline.data_ptr(), d_k.data_ptr(), d_maxs.data_ptr(), 0.15, 0.3, 1)
    so = bounds.StatesOut(d_states.data_ptr(), d_curv.data_ptr(), d_n.data_ptr(), None, None)
    bi = bounds.BoundsIn(B, n, lines.k_max, d_states.data_ptr(), d_n.data_ptr(), d_spline.data_ptr(), d_k.data_ptr())
    bo = bounds.BoundsOut(d_bounds.data_ptr(), d_nv.data_ptr(), None)
    stream = torch.cuda.current_stream().cuda_stream
    reps = 10
    ms = {}
    for name, fn in (("states", lambda: pbn.build_states_device(si, so, stream=stream)),
                     ("bounds", lambda: pbn.compute_device(bi, bo, stream=stream))):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms[name] = e0.elapsed_time(e1) / reps
    states, bnd, nv = d_states.cpu().numpy(), d_bounds.cpu().numpy(), d_nv.cpu().numpy()
    assert np.max(np.abs(states - lines.states)) < 1e-9, "reference-states kernel disagrees with the workload's states"
    sample = min(B, 64)
    t0 = time.perf_counter()
    worst = 0.0
    for b in range(sample):
        ob, onv = bounds_oracle.update_bounds(dmap.dist, dmap.res, lines.spline_rows(b), *lines.states[b])
        d = np.abs(ob - bnd[b])
        worst = max(worst, float(d[d < 0.04].max()))
        assert onv == nv[b], "bounds kernel and oracle cut path %d differently" % b
    cpu_s = time.perf_counter() - t0
    plan = plan_pipeline(args, pbn, lines, d_spline, d_k, d_maxs, device)
    pbn.close()
    # algorithmic bytes per state: 32 B state + 48 B bounds + the path's share of its spline
    alg = B * n * 80 + lines.spline.nbytes + dmap.dist.nbytes
    return {"bounds": bnd, "n_valid": nv,
            "bounds_kernel": {"kernel": "clearance_bounds_kernel", "ms_per_batch": ms["bounds"],
                              "states_per_s": B * n / (ms["bounds"] * 1e-3), "rays_per_s": 3 * B * n / (ms["bounds"] * 1e-3),
                              "algorithmic_bytes": int(alg), "achieved_GBps": alg / (ms["bounds"] * 1e-3) / 1e9,
                              "gpu_launches_per_batch": 2, "max_abs_diff_vs_oracle": worst,
                              "cpu_oracle_states_per_s": sample * n / cpu_s, "cpu_oracle_sample": sample},
            "states_kernel": {"kernel": "reference_states_kernel", "ms_per_batch": ms["states"],
                              "states_per_s": B * n / (ms["states"] * 1e-3)},
            "plan_pipeline": plan}


def plan_pipeline(args, pbn, lines, d_spline, d_k, d_maxs, device):
    """The reference's whole PathOptimizer::optimizePath sequence (path_optimizer.cpp:124-161) for the
    batch, device-resident through the C ABI: reference states from the splines -> clearance bounds
    -> BaseSolver::solve -> re-linearise -> updateProblemFormulationAndSolve. One plan = two solves."""
    import torch
    from path_optimizer_2_b200 import bounds, solver
    dev = torch.device("cuda", device)
    B, n = lines.batch, lines.n_max
    f64 = dict(dtype=torch.float64, device=dev)
    d_inst = torch.from_numpy(lines.inst).to(dev)
    d_states, d_curv = torch.zeros((B, 4, n), **f64), torch.zeros((B, n), **f64)
    d_knots, d_bounds = torch.zeros((B, abi.NFIELDS, n), **f64), torch.zeros((B, 6, n), **f64)
    d_sol, d_cost = torch.zeros((B, 4, n), **f64), torch.zeros(B, **f64)
    d_n, d_nv, d_status, d_iters = (torch.zeros(B, dtype=torch.int32, device=dev) for _ in range(4))
    sv = solver.PathQpSolver(abi.default_params(reserved=args.option_bits & ~128), n_max=n, batch_max=B, device=device)
    si = bounds.StatesIn(B, n, lines.k_max, d_spline.data_ptr(), d_k.data_ptr(), d_maxs.data_ptr(), 0.15, 0.3, 1)
    so = bounds.StatesOut(d_states.data_ptr(), d_curv.data_ptr(), d_n.data_ptr(), None, d_knots.data_ptr())
    bi = bounds.BoundsIn(B, n, lines.k_max, d_states.data_ptr(), d_n.data_ptr(), d_spline.data_ptr(), d_k.data_ptr())
    bo = bounds.BoundsOut(d_bounds.data_ptr(), d_nv.data_ptr(), d_knots.data_ptr())
    qi = abi.PqpBatchIn(B, n, d_knots.data_ptr(), d_inst.data_ptr(), d_nv.data_ptr(), None)
    qo = abi.PqpBatchOut(d_sol.data_ptr(), d_cost.data_ptr(), d_status.data_ptr(), d_iters.data_ptr(), None, None, None, None)
    stream = torch.cuda.current_stream().cuda_stream

    def plan():
        pbn.build_states_device(si, so, stream=stream)
        pbn.compute_device(bi, bo, stream=stream)
        sv.solve_device(qi, qo, stream=stream)
        sv.relinearise_device(B, d_sol.data_ptr(), d_knots.data_ptr(), stream=stream)
        sv.solve_device(qi, qo, stream=stream, warm=True)

    for _ in range(3):
        plan()
    torch.cuda.synchronize()
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        plan()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    status, iters2 = d_status.cpu().numpy(), d_iters.cpu().numpy()
    sv.close()
    return {"what": "states -> bounds -> solve -> relinearise -> warm re-solve, device-resident (PathOptimizer::optimizePath)",
            "ms_per_batch": ms, "plans_per_s": B / (ms * 1e-3), "launches_per_plan": 8,
            "solved_fraction": float(np.mean(status == abi.PQP_SOLVED)), "mean_second_solve_iters": float(np.mean(iters2))}


def algorithmic_bytes(n, warm=False):
    return (296 * n + 72) if warm else (104 * n + 56)


def measured_traffic(n, instances, cold_only):
    """DRAM bytes per launch from the ncu --set full capture committed in the same round
    (profiles/r2/traffic_*.json, written by profiles/traffic_from_ncu.py), or None."""
    name = "traffic_cold_n%d%s.json" % (n, "_coldonly" if cold_only else "")
    try:
        with open(os.path.join(ROOT, "profiles", "r2", name)) as f:
            return float(json.load(f)["dram_bytes_per_instance"]) * instances
    except Exception:
        return None


def measured_issue(n, cold_only):
    """What actually bounds the kernel, from the same capture: warp instructions per launch and the share of cycles
    in which a scheduler issued (one warp per scheduler: the kernel is latency / issue bound, not HBM bound)."""
    name = "traffic_cold_n%d%s.json" % (n, "_coldonly" if cold_only else "")
    try:
        with open(os.path.join(ROOT, "profiles", "r2", name)) as f:
            r = json.load(f)
        if r.get("issue_active_pct") is None:
            return None
        return {"warp_instructions_per_launch": r["warp_instructions"], "issue_active_pct": r["issue_active_pct"],
                "registers_per_thread": r.get("registers_per_thread"), "batch": r["batch"],
                "source": "ncu --set full capture of this round (profiles/r2/%s)" % name}
    except Exception:
        return None


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# --------------------------------------------------------------------------------------- CPU arm
def host_cores():
    """Cores this process can really use: the scheduler affinity mask, capped by the cgroup CPU quota
    (a container may see 128 CPUs in its mask and be entitled to a fraction of them: round 1's CPU arm
    differed 5.5x between two boxes that both reported 128 cores)."""
    try:
        affinity = len(os.sched_getaffinity(0))
    except AttributeError:
        affinity = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2: "<quota|max> <period>"
            q, p = f.read().split()
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    eff = affinity if quota is None else max(1, min(affinity, int(math.ceil(quota))))
    return {"affinity": affinity, "nproc": os.cpu_count(), "cgroup_quota": quota, "effective": eff}


def pick_threads(params, hb, cores):
    """Short sweep of OpenMP thread counts on a slice of the workload (torchrun's OMP_NUM_THREADS=1 is
    ignored: the count is passed explicitly); returns (best thread count, {threads: solves/s})."""
    from oracle import oracle
    cand = sorted({t for t in (1, 8, 16, 32, 64, 96, 128, 192, 256, cores["effective"], cores["affinity"])
                   if 1 <= t <= cores["affinity"]})
    sub = hb.slice(0, min(hb.batch, 2048))
    oracle.solve_batch(params, sub.slice(0, min(64, sub.batch)), nthreads=cand[-1])  # warm the thread pool
    sweep = {}
    for t in cand:
        # long enough (a few hundred ms) to run into the cgroup's CPU quota: a short burst may use more cores than
        # the container is entitled to and would pick a thread count that the full batch cannot sustain
        s = sub.slice(0, min(sub.batch, 64 if t == 1 else 2048))
        _, secs = oracle.solve_batch(params, s, nthreads=t, mode=0, dense_assembly=False)
        sweep[t] = s.batch / secs
    multi = {t: v for t, v in sweep.items() if t > 1} or sweep
    best = max(multi, key=multi.get)
    return best, {str(t): round(v, 1) for t, v in sweep.items()}


def cpu_baseline(params, hb, sample):
    """Oracle port on the host cores. `value` is the OSQP-algorithm cost alone (direct CSC
    assembly, the conservative figure); the reference's own plumbing additionally zero-fills
    and scans dense m x nv / nv x nv temporaries per solve (base_solver.cpp:122,145,159,210),
    timed separately and quoted in `sample`."""
    from oracle import oracle
    cores = host_cores()
    threads, sweep = pick_threads(params, hb, cores)
    sub = hb.slice(0, min(sample, hb.batch))
    res, secs = oracle.solve_batch(params, sub, nthreads=threads, mode=0, dense_assembly=False)
    dsub = sub.slice(0, min(256, sub.batch))
    _, dsecs = oracle.solve_batch(params, dsub, nthreads=threads, mode=0, dense_assembly=True)
    solved = int(np.sum(res.status == abi.PQP_SOLVED))
    return {"value": sub.batch / secs, "unit": UNIT, "cores": threads, "kind": "port",
            "host": cores, "thread_sweep_solves_per_s": sweep,
            "sample": "%d instances of the same workload, oracle port (OSQP-algorithm restatement, FP64, "
                      "sparse LDL'), %d OpenMP threads (fastest of the sweep; cgroup quota %s, affinity %d), %.2f s "
                      "wall, %d solved; 1 thread: %s solves/s; with the reference-style dense assembly temporaries: "
                      "%.0f solves/s on %d threads"
                      % (sub.batch, threads, cores["cgroup_quota"], cores["affinity"], secs, solved, sweep.get("1"),
                         dsub.batch / dsecs, threads)}


def run_reference(args, rank, world):
    """--impl reference: the CPU path alone (rank 0 only under torchrun), on the FULL batch of the
    b200 arm's config every step, with the fastest OpenMP thread count of a short sweep."""
    if rank != 0:
        return
    from oracle import oracle
    params = abi.default_params()
    cores = host_cores()
    sample = args.batch if args.cpu_sample is None else args.cpu_sample
    hb, workload, _ = make_workload(args, sample, 0)
    threads, sweep = pick_threads(params, hb, cores)
    for _ in range(max(1, min(args.warmup, 2))):
        oracle.solve_batch(params, hb.slice(0, min(sample, 8 * threads)), nthreads=threads)
    t_tot = 0.0
    for _ in range(args.steps):
        res, secs = oracle.solve_batch(params, hb, nthreads=threads, mode=0, dense_assembly=False)
        t_tot += secs
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"sol": res.sol, "cost": res.cost, "status": res.status, "iters": res.iters})
    value = sample * args.steps / t_tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload, "n_knots": args.n, "batch_per_gpu": sample, "batch_per_step": sample,
                   "global_batch": sample, "cold_solve": True, "eps_abs": params.eps_abs, "eps_rel": params.eps_rel,
                   "max_iter": params.max_iter,
                   "note": "CPU arm: rank 0 alone, one GPU-rank's batch per step whatever --gpus says"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "host": cores,
                         "thread_sweep_solves_per_s": sweep,
                         "sample": "%d instances per step (the whole batch of one GPU rank), OSQP-algorithm restatement "
                                   "with direct CSC assembly, %d OpenMP threads = fastest of the sweep (real OSQP is not "
                                   "vendored by the reference and not installable here; the reference's dense assembly "
                                   "temporaries are NOT included)" % (sample, threads)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------- GPU arm
class GatherPipe:
    """The only exchange of the multi-GPU path - an all-gather of {cost f64, status i32, iters i32} =
    16 B per instance - taken off the solve stream: the records are packed by one library kernel
    (pqp_pack_results_device) and gathered over NCCL on a side stream while the next batch already
    solves, so a rank is no longer held in lock step with the slowest rank's launch tail every step
    (round 1: blocking gather + 6 eager torch launches per step, efficiency 0.92 at 8 GPUs)."""

    def __init__(self, sv, B, world, dev):
        import torch
        from path_optimizer_2_b200 import multi
        self.torch, self.multi, self.sv, self.B, self.world = torch, multi, sv, B, world
        self.side = torch.cuda.Stream(device=dev)
        self.packed = torch.zeros(B * 16, dtype=torch.uint8, device=dev)
        self.gathered = torch.zeros(world * B * 16, dtype=torch.uint8, device=dev)
        self.ev_solved, self.ev_packed = torch.cuda.Event(), torch.cuda.Event()

    def submit(self, d_cost, d_status, d_iters, stream=None):
        """Call right after the solve was queued on `stream` (default: the current stream)."""
        import torch.distributed as dist
        torch = self.torch
        main = stream if stream is not None else torch.cuda.current_stream()
        self.ev_solved.record(main)
        with torch.cuda.stream(self.side):
            self.side.wait_event(self.ev_solved)
            self.multi.pack_results_device(self.sv, self.B, d_cost.data_ptr(), d_status.data_ptr(), d_iters.data_ptr(),
                                           self.packed.data_ptr(), stream=self.side.cuda_stream)
            self.ev_packed.record(self.side)
            dist.all_gather_into_tensor(self.gathered, self.packed)
        main.wait_event(self.ev_packed)  # the next solve overwrites cost/status/iters: wait for the 2 us pack only

    def finish(self):
        self.torch.cuda.current_stream().wait_stream(self.side)

    def table(self):
        return self.gathered.cpu().numpy().view(self.multi.RESULT_REC)


def reduce_max(value, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_scalars(value, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64, device=dev)
    if world == 1:
        return [float(value)]
    out = torch.zeros(world, dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(out, t)
    return [float(v) for v in out.cpu().numpy()]


def barrier(world):
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def bind_to_gpu_numa_node(local_rank):
    """One process per GPU: run this rank's host threads on the CPUs of the GPU's NUMA node, so that the pinned
    host buffers it allocates (local allocation policy) sit behind the memory controllers next to its PCIe root.
    Eight ranks move 8 x 205 MB of host memory per 5.7 ms step end to end; from one socket's memory that stops at
    ~170 GB/s (profiles/r2/scale_r2_builder.txt). Returns the node, or None when the topology is not exposed."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:  # noqa: BLE001 - no sysfs / no permission: keep the default placement
        return None


DUMP_BYTES = 64_000_000  # what --dump-outputs may write in all


def dump_outputs(out_dir, arrays):
    """--dump-outputs: the per-instance arrays the timed path's caller received in the last timed step, one
    <out_dir>/<name>.npy each in float64. Beyond DUMP_BYTES the same seeded sample of instances is taken from
    every array; instance.npy lists the instances written."""
    batch = len(arrays["cost"])
    per_instance = 8 * (1 + sum(a[0].size for a in arrays.values()))
    keep = min(batch, (DUMP_BYTES - 4096) // per_instance)  # 4096: room for the .npy headers
    idx = np.arange(batch) if keep == batch else np.sort(np.random.default_rng(0).choice(batch, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in dict({k: v[idx] for k, v in arrays.items()}, instance=idx).items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def sv_uses_tmem(n, batch):
    """The library's storage policy (DESIGN.md §4): tensor memory for n_max >= 64."""
    return n >= 64


def measure_cold(args, hb, option_bits, steps, warmup, e2e_steps, local_rank, world, dev, gather=True, clocks=False,
                 inflight=1, dump_dir=None):
    """Cold solves of this rank's batch `hb`: device-resident value, end-to-end value, kernel time.
    inflight = 2: consecutive steps alternate between two handles on two streams, so the next batch's CTAs take
    over SMs as the previous batch's persistent CTAs run out of work (iteration counts are heavy-tailed: 10 % of a
    lone launch is tail). Every step is still one full batch; the timed region covers all of them.
    dump_dir: rank 0 writes the last timed step's results there (dump_outputs)."""
    import torch
    from path_optimizer_2_b200 import solver
    params = abi.default_params(reserved=option_bits)
    B, n = hb.batch, hb.n_max
    K = max(1, int(inflight))
    svs = [solver.PathQpSolver(params, n_max=n, batch_max=B, device=local_rank) for _ in range(K)]
    sv = svs[0]
    # inputs smaller than L2 (the shared-map config): evict them between timed steps
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if hb.knots.nbytes < (160 << 20) else None
    d_knots, d_inst, d_n = (torch.from_numpy(v).to(dev) for v in (hb.knots, hb.inst, hb.n))
    outs = []
    for _ in range(K):
        d_sol = torch.zeros((B, 4, n), dtype=torch.float64, device=dev)
        d_cost = torch.zeros(B, dtype=torch.float64, device=dev)
        d_status, d_iters = (torch.zeros(B, dtype=torch.int32, device=dev) for _ in range(2))
        outs.append((d_sol, d_cost, d_status, d_iters,
                     abi.PqpBatchOut(d_sol.data_ptr(), d_cost.data_ptr(), d_status.data_ptr(), d_iters.data_ptr(), None, None, None, None)))
    bin_s = abi.PqpBatchIn(B, n, d_knots.data_ptr(), d_inst.data_ptr(), d_n.data_ptr(), None)
    main = torch.cuda.current_stream()
    streams = [main] if K == 1 else [torch.cuda.Stream(device=dev) for _ in range(K)]
    pipes = [GatherPipe(svs[k], B, world, dev) if (gather and world > 1) else None for k in range(K)]

    def step(i, ev=None):
        k = i % K
        st = streams[k]
        if ev is not None:
            ev[0].record(st)
        svs[k].solve_device(bin_s, outs[k][4], stream=st.cuda_stream)
        if ev is not None:
            ev[1].record(st)
        if pipes[k]:
            pipes[k].submit(outs[k][1], outs[k][2], outs[k][3], stream=st)

    def join():
        for k in range(K):
            if pipes[k]:
                with torch.cuda.stream(streams[k]):
                    pipes[k].finish()
            if streams[k] is not main:
                main.wait_stream(streams[k])

    def fork():
        for st in streams:
            if st is not main:
                st.wait_stream(main)

    fork()
    for i in range(warmup):
        step(i)
    join()
    barrier(world)
    # launch duration of the dominant kernel, timed alone (one launch at a time) - the roofline's denominator
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(steps, 5))]
    for i in range(len(kev)):
        if flush is not None:
            flush.fill_(i & 255)
        kev[i][0].record(main)
        svs[0].solve_device(bin_s, outs[0][4], stream=main.cuda_stream)
        kev[i][1].record(main)
    barrier(world)
    kernel_ms = float(np.median([a.elapsed_time(b) for a, b in kev]))
    sampler = ClockSampler(local_rank) if clocks else None
    if sampler:
        sampler.start()
    launches0 = sum(s_.launch_count for s_ in svs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    e0.record(main)
    fork()
    for i in range(steps):
        if flush is not None:
            with torch.cuda.stream(streams[i % K]):
                flush.fill_(i & 255)
        step(i)
    join()  # the timed region ends when the last solve and the last gather have landed
    e1.record(main)
    barrier(world)
    launches = sum(s_.launch_count for s_ in svs) - launches0
    clk = sampler.stop() if sampler else None
    my_ms = e0.elapsed_time(e1)
    total_ms = reduce_max(my_ms, dev, world)
    last = (steps - 1) % K
    status, iters = outs[last][2].cpu().numpy(), outs[last][3].cpu().numpy()
    if dump_dir and int(os.environ.get("RANK", "0")) == 0:
        dump_outputs(dump_dir, {"sol": outs[last][0].cpu().numpy(), "cost": outs[last][1].cpu().numpy(),
                                "status": status, "iters": iters})
    for k in range(K):  # every handle solved the same batch: identical results
        assert np.array_equal(outs[k][2].cpu().numpy(), status) or steps <= k
    if pipes[last]:  # the gathered table holds every rank's records; this rank's block must equal its own results
        tab = pipes[last].table()
        rank = int(os.environ.get("RANK", "0"))
        mine = tab[rank * B:(rank + 1) * B]
        assert np.array_equal(mine["status"], status) and np.array_equal(mine["iters"], iters), "gathered table is wrong"
    # ---- e2e: host buffers through the public host-pointer call (H2D + kernel + D2H timed). With K batches in
    # flight the caller drives K handles from K host threads (a handle is single-threaded, handles are independent):
    # every step is still one synchronous pqp_solve of a whole batch from pinned host memory into pinned host memory.
    pin = lambda a: torch.from_numpy(a).pin_memory()  # noqa: E731
    p_knots, p_inst, p_n = pin(hb.knots), pin(hb.inst), pin(hb.n)
    hbp = abi.HostBatch(p_knots.numpy(), p_inst.numpy(), p_n.numpy())
    hress, keep = [], []
    for _ in range(K):
        hres = abi.HostResult(B, n, full=False, info=False)
        p_sol, p_cost = pin(hres.sol), pin(hres.cost)
        p_status, p_iters = pin(hres.status), pin(hres.iters)
        hres.sol, hres.cost, hres.status, hres.iters = p_sol.numpy(), p_cost.numpy(), p_status.numpy(), p_iters.numpy()
        hress.append(hres)
        keep.append((p_sol, p_cost, p_status, p_iters))
    for k in range(K):
        for _ in range(2):
            svs[k].solve(hbp, out=hress[k])
    errs = []

    def host_worker(k):
        try:
            torch.cuda.set_device(local_rank)
            for _ in range(k, e2e_steps, K):
                svs[k].solve(hbp, out=hress[k])  # synchronous: returns after the D2H copy completed
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    barrier(world)
    t0 = time.perf_counter()
    if K == 1:
        host_worker(0)
    else:
        import threading
        ths = [threading.Thread(target=host_worker, args=(k,)) for k in range(K)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
    torch.cuda.synchronize()
    e2e_s = reduce_max(time.perf_counter() - t0, dev, world)
    if errs:
        raise errs[0]
    hres = hress[0]
    for k in range(1, K):
        assert np.array_equal(hress[k].status, hres.status) and np.array_equal(hress[k].sol, hres.sol)
    h2d = int(hb.knots.nbytes + hb.inst.nbytes + hb.n.nbytes)
    d2h = int(hres.sol.nbytes + hres.cost.nbytes + hres.status.nbytes + hres.iters.nbytes)
    if not (option_bits & 2):  # the host call escalates suspected-infeasible instances to FP64, the device call cannot
        assert np.array_equal(hres.status, status), "host-API and device-API runs disagree"
    info = sv.kernel_info
    kms = gather_scalars(kernel_ms, dev, world)
    for s_ in svs:
        s_.close()
    return {"value": world * B * steps / (total_ms * 1e-3), "ms_per_step": total_ms / steps, "kernel_ms": kernel_ms, "inflight": K,
            "kernel_ms_per_rank": kms, "e2e_value": world * B * e2e_steps / e2e_s, "e2e_steps": e2e_steps,
            "h2d": h2d, "d2h": d2h, "launches": int(launches), "clocks": clk, "status": status, "iters": iters,
            "info": info, "params": params, "flushed": flush is not None, "steps": steps}


def run_receding(args, rank, local_rank, world, dev, dump_dir=None):
    """BASELINE configs[4]: receding-horizon warm re-solves (SURVEY.md §8d config 5). One step =
    one tick: advance the window by one knot (pqp_advance_window_device, one launch),
    re-linearise about the previous solution, warm re-solve with max_iter = 50 through
    pqp_resolve_device; x, z, y, rho stay resident in the handle between ticks.
    dump_dir: rank 0 writes the last timed tick's results there (dump_outputs)."""
    import torch
    from path_optimizer_2_b200 import solver

    B, n = args.batch, args.n
    ticks = args.warmup + args.steps
    params = abi.default_params(max_iter=50)
    ext = synthetic.make_batch(5, B, n + ticks + 1, first=rank * B)
    sv = solver.PathQpSolver(params, n_max=n, batch_max=B, device=local_rank)
    d_ext = torch.from_numpy(ext.knots).to(dev)
    d_knots = d_ext[:, :, :n].contiguous()
    d_inst = torch.from_numpy(ext.inst).to(dev)
    d_n = torch.full((B,), n, dtype=torch.int32, device=dev)
    d_sol = torch.zeros((B, 4, n), dtype=torch.float64, device=dev)
    d_cost = torch.zeros(B, dtype=torch.float64, device=dev)
    d_status = torch.zeros(B, dtype=torch.int32, device=dev)
    d_iters = torch.zeros(B, dtype=torch.int32, device=dev)
    bout_s = abi.PqpBatchOut(d_sol.data_ptr(), d_cost.data_ptr(), d_status.data_ptr(), d_iters.data_ptr(),
                             None, None, None, None)
    pipe = GatherPipe(sv, B, world, dev) if world > 1 else None
    stream = torch.cuda.current_stream().cuda_stream
    bin_w = abi.PqpBatchIn(B, n, d_knots.data_ptr(), d_inst.data_ptr(), d_n.data_ptr(), None)
    ext_len = int(d_ext.shape[2])

    def tick_device(t):
        # window bookkeeping in one launch of the library's own kernel, in place: the previous
        # tick's solve has consumed d_knots / d_inst (same stream), d_sol holds its result
        sv.advance_window_device(B, ext_len, t, d_ext.data_ptr(), d_sol.data_ptr(), d_knots.data_ptr(),
                                 d_inst.data_ptr(), stream=stream)

    sv.solve_device(bin_w, bout_s, stream=stream, warm=False)  # tick 0: cold
    tick = 0
    for _ in range(args.warmup):
        tick += 1
        tick_device(tick)
        sv.solve_device(bin_w, bout_s, stream=stream, warm=True)
        if pipe:
            pipe.submit(d_cost, d_status, d_iters)
    if pipe:
        pipe.finish()
    barrier(world)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = sv.launch_count
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    e0.record()
    for i in range(args.steps):
        tick += 1
        tick_device(tick)
        kev[i][0].record()
        sv.solve_device(bin_w, bout_s, stream=stream, warm=True)
        kev[i][1].record()
        if pipe:
            pipe.submit(d_cost, d_status, d_iters)
    if pipe:
        pipe.finish()
    e1.record()
    barrier(world)
    launches = sv.launch_count - launches0
    clocks = sampler.stop()
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    total_ms = reduce_max(e0.elapsed_time(e1), dev, world)
    value = world * B * args.steps / (total_ms * 1e-3)
    status = d_status.cpu().numpy()
    iters = d_iters.cpu().numpy()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"sol": d_sol.cpu().numpy(), "cost": d_cost.cpu().numpy(), "status": status, "iters": iters})
    kms = gather_scalars(kernel_ms, dev, world)

    # e2e: the same tick through the host-pointer call (pinned host buffers, H2D + D2H timed);
    # the window bookkeeping runs on the host in numpy and is part of the timed region
    hb = abi.HostBatch(ext.knots[:, :, :n].copy(), ext.inst, np.full(B, n, dtype=np.int32))
    sv2 = solver.PathQpSolver(params, n_max=n, batch_max=B, device=local_rank)
    hres = abi.HostResult(B, n, full=False, info=False)
    sv2.solve(hb, out=hres)
    inst_h, tick2 = ext.inst, 0
    e2e_steps = args.e2e_steps or args.steps
    barrier(world)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        tick2 += 1
        k_h, inst_h = synthetic.shift_window(ext.knots, inst_h, hres.sol, tick2, n)
        sv2.resolve(abi.HostBatch(k_h, inst_h, hb.n), out=hres)
    e2e_s = reduce_max(time.perf_counter() - t0, dev, world)
    e2e_value = world * B * e2e_steps / e2e_s
    info = sv.kernel_info
    sv.close()
    sv2.close()
    peak, peak_src = hbm_peak()
    bytes_per_launch = B * algorithmic_bytes(n, warm=True)
    achieved = bytes_per_launch / (kernel_ms * 1e-3) / 1e9
    return {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": "BASELINE configs[4] per GPU: receding-horizon warm re-solve, batch %d, %d knots, "
                        "50-iteration cap, window advances one knot per step" % (B, n),
            "n_knots": n, "batch_per_gpu": B, "global_batch": world * B, "parallelism": "dp%d" % world,
            "max_iter": 50, "l2_policy": "inputs %.0f MB per step (smaller than L2; each step reads freshly "
                                         "written window buffers)" % (d_knots.numel() * 8 / 1e6),
            "collective": "all_gather of {cost,status,iters} (16 B/instance) on a side stream, overlapping the next "
                          "tick's solve" if world > 1 else "none",
            "mean_admm_iters": float(np.mean(iters)),
            "solved_fraction": float(np.mean(status == abi.PQP_SOLVED)),
            "warps_per_sm": info["warps_per_sm"], "smem_per_warp": info["smem_per_warp"],
            "kernel_ms_per_rank": {"min": min(kms), "max": max(kms)},
        },
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT,
                "h2d_bytes_per_step": int(hb.knots.nbytes + hb.inst.nbytes + hb.n.nbytes),
                "d2h_bytes_per_step": int(hres.sol.nbytes + hres.cost.nbytes + hres.status.nbytes + hres.iters.nbytes),
                "steps": e2e_steps},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                     "kernel": "pqp_admm_kernel_tmem (warm)", "kernel_ms": kernel_ms,
                     "algorithmic_bytes_per_launch": bytes_per_launch},
    }


def dropin_single_path(n=120, plans=200):
    """BASELINE configs[0]: ONE path of ~120 knots through the C++ drop-in (include/pqp_base_solver.hpp),
    driven like PathOptimizer::optimizePath at 30 Hz (path_optimizer.cpp:138-153): a BaseSolver object
    is constructed per plan, solve() + updateProblemFormulationAndSolve(), destructed. Wall time per
    plan INCLUDING construction/destruction; the first plan pays pqp_create, later ones borrow the
    pooled handle."""
    from path_optimizer_2_b200 import sharedmap
    from tests import test_dropin
    exe = test_dropin._build(False)
    dmap = sharedmap.DistanceMap()
    lines = sharedmap.make_lines(1, n, dmap=dmap)
    from oracle import bounds_oracle
    bnd, nv = bounds_oracle.update_bounds(dmap.dist, dmap.res, lines.spline_rows(0), *lines.states[0])
    hb = lines.to_host_batch(bnd[None], np.array([nv], dtype=np.int32))
    nn = int(hb.n[0])
    ref = np.stack([lines.states[0][1], lines.states[0][2], lines.states[0][3]])
    with tempfile.TemporaryDirectory() as tmp:  # the tree may be read-only
        path = os.path.join(tmp, "dropin_instance.txt")
        test_dropin._write_instance(path, hb.knots[0], hb.inst[0], nn, ref, 0.0, constraint_end_heading=0)
        out = subprocess.run([exe, path, str(plans)], capture_output=True, text=True, check=True).stdout.strip().split("\n")
    tok = out[0].split()
    if tok[0] != "plans":
        return {"error": out[0]}
    st = {tok[i]: float(tok[i + 1]) for i in range(0, 10, 2)}
    sg = {tok[i]: float(tok[i + 1]) for i in range(11, len(tok) - 1, 2)}
    return {"what": "BASELINE configs[0]: one path, %d knots, gridmap.png clearance bounds, C++ drop-in BaseSolverT "
                    "constructed per plan (solve + updateProblemFormulationAndSolve = 2 solves per plan)" % nn,
            "plans": int(st["plans"]), "first_plan_ms_incl_pqp_create": st["first_ms"], "later_plan_ms": st["later_ms"],
            "plans_per_s": 1e3 / st["later_ms"], "solves_per_s": 2e3 / st["later_ms"],
            "handle_pool": {"creates": int(st["creates"]), "hits": int(st["hits"])},
            "last_call_stage_ms": sg}


def front_end_stages(lines, dmap, device):
    """SURVEY.md §8 rows f-4 and f-3 on the GPU for the shared-map batch: lattice DP search over the smoothed
    references, then the post-smooth QP on the DP's corridor, and the tension-smoother QP on the references resampled
    at 1 m - each one launch through its C ABI (host-pointer call; the kernel time is the CUDA-event time between the
    copies). Checked against the oracles on a sample."""
    from oracle import bounds_oracle as bo, dp_oracle, smoother_oracle
    from path_optimizer_2_b200 import bounds, dp, smoother
    B = lines.batch
    length = np.array([lines.spline_rows(b)[0, lines.k[b] - 1] + 3.0 for b in range(B)])
    start = np.zeros((B, 3))
    rng = np.random.default_rng(11)
    for b in range(B):
        sp = bo.Spline2(lines.spline_rows(b))
        x, y = dp_oracle._xy(sp, 0.5)
        h = dp_oracle.heading(sp, 0.5)
        off = rng.uniform(-1.0, 1.0)
        start[b] = x - off * np.sin(h), y + off * np.cos(h), h
    pbn = bounds.PathBounds(dmap.dist, dmap.res, device=device)
    ds = dp.DpSearch(pbn, layers_max=64, batch_max=B)
    for _ in range(2):
        r = ds.search(lines.spline, lines.k, length, start, tables=False)
    dp_ms = ds.last_kernel_ms
    ok = r.status == dp.DP_OK
    for b in np.nonzero(ok)[0][:8]:
        o = dp_oracle.graph_search_dp(dmap.dist, dmap.res, lines.spline_rows(b), length[b], start[b])
        assert np.array_equal(r.chosen[b, :r.n_out[b]], o["chosen"]), "DP kernel and oracle chose different nodes"
    out = {"dp_search": {"kernel": "dp_search_kernel", "paths": int(B), "ok_fraction": float(ok.mean()),
                         "mean_layers": float(r.n_layers.mean()), "ms_per_batch": dp_ms, "paths_per_s": B / (dp_ms * 1e-3),
                         "algorithmic_bytes": int(lines.spline.nbytes + 3 * 8 * B + r.n_out.sum() * 28 + 40 * B)}}
    idx = np.nonzero(ok & (r.n_out >= 4))[0]
    sm = smoother.Smoother(p_max=64, batch_max=B, device=device)
    ls = [r.layer_s[b, :r.n_out[b]] for b in idx]
    lo = [r.lower[b, :r.n_out[b]] for b in idx]
    up = [r.upper[b, :r.n_out[b]] for b in idx]
    vl = r.vehicle_l[idx]
    for _ in range(2):
        pr = sm.post(ls, lo, up, vl)
    post_ms = sm.last_kernel_ms
    for j in range(min(4, len(idx))):
        okp, off, g = smoother_oracle.post_smooth(ls[j], lo[j], up[j], vl[j])
        assert pr["status"][j] == g.status and pr["iters"][j] == g.iters and np.allclose(pr["offsets"][j, :len(off)], off, atol=1e-6)
    out["post_smooth_qp"] = {"kernel": "smoother_kernel (postSmooth QP)", "qps": int(len(idx)), "ms_per_batch": post_ms,
                             "qps_per_s": len(idx) / (post_ms * 1e-3), "mean_iters": float(pr["iters"].mean()),
                             "solved_fraction": float(np.mean(pr["status"] == abi.PQP_SOLVED)),
                             "algorithmic_bytes": int(sum(len(v) for v in ls) * 32 + 16 * len(idx))}
    sm.close()
    # tension smoother: the references resampled at 1 m (segmentRawReference) with a little noise as the raw input
    xs, ys, an, ks, ss = [], [], [], [], []
    for b in range(B):
        sp = bo.Spline2(lines.spline_rows(b))
        s = np.arange(0.0, lines.spline_rows(b)[0, lines.k[b] - 1], 1.0)
        x, dx, ddx = sp.x(s)
        y, dy, ddy = sp.y(s)
        xs.append(x + rng.normal(0, 0.03, len(s)))
        ys.append(y + rng.normal(0, 0.03, len(s)))
        an.append(np.arctan2(dy, dx))
        ks.append((dx * ddy - dy * ddx) / np.power(dx * dx + dy * dy, 1.5))
        ss.append(s)
    pmax = max(len(v) for v in xs)
    sm = smoother.Smoother(p_max=max(pmax, 8), batch_max=B, device=device)
    for _ in range(2):
        tr = sm.tension(xs, ys, an, ks, ss)
    t_ms = sm.last_kernel_ms
    for j in range(3):
        okt, rx, ry, rs, g = smoother_oracle.osqp_smooth(xs[j], ys[j], an[j], ks[j], ss[j])
        assert tr["status"][j] == g.status and tr["iters"][j] == g.iters and np.allclose(tr["x"][j, :len(rx)], rx, atol=1e-6)
    out["tension_smoother_qp"] = {"kernel": "smoother_kernel (TensionSmoother2 QP)", "qps": int(B), "mean_points": float(np.mean([len(v) for v in xs])),
                                  "ms_per_batch": t_ms, "qps_per_s": B / (t_ms * 1e-3), "mean_iters": float(tr["iters"].mean()),
                                  "solved_fraction": float(np.mean(tr["status"] == abi.PQP_SOLVED)),
                                  "algorithmic_bytes": int(sum(len(v) for v in xs) * 64 + 12 * B)}
    sm.close()
    ds.close()
    pbn.close()
    return out


def secondary(args, rank, local_rank, world, dev, hb_primary):
    """The other BASELINE configs and the FP64 instantiation, measured in the same run (short loops)."""
    sec = {}
    # the like-for-like precision against FP64 OSQP: the same kernel instantiated in double (option bit 2)
    steps = max(2, min(args.steps, 3))
    r = measure_cold(args, hb_primary, 2, steps, 1, 2, local_rank, world, dev, gather=False)
    fp64 = {"value": r["value"], "unit": UNIT, "e2e": r["e2e_value"], "kernel_ms": r["kernel_ms"], "steps": steps,
            "mean_admm_iters": float(np.mean(r["iters"])), "solved_fraction": float(np.mean(r["status"] == abi.PQP_SOLVED)),
            "what": "same workload, pqp_params.reserved = 2: iterates, factorisation and residuals in FP64 "
                    "(reproduces the FP64 oracle's iterates to 1e-8, tests/test_gpu_parity.py)"}
    # configs[4] at this N
    a4 = argparse.Namespace(**vars(args))
    a4.batch, a4.n, a4.steps, a4.warmup, a4.e2e_steps = 512, 240, 20, 3, 5
    l4 = run_receding(a4, rank, local_rank, world, dev)
    sec["configs[4]"] = {"workload": l4["config"]["workload"], "value": l4["value"], "unit": UNIT, "n_gpus": world,
                         "ms_per_step": l4["ms_per_step"], "e2e": l4["e2e"]["value"], "kernel_ms": l4["roofline"]["kernel_ms"],
                         "mean_admm_iters": l4["config"]["mean_admm_iters"], "solved_fraction": l4["config"]["solved_fraction"],
                         "kernel_ms_per_rank": l4["config"]["kernel_ms_per_rank"]}
    if world == 1:
        a1 = argparse.Namespace(**vars(args))
        a1.workload, a1.batch, a1.n = "sharedmap", 1024, 120
        hb1, wl1, ex1 = make_workload(a1, 1024, 0, device=local_rank)
        lines1, dmap1 = ex1.pop("_lines"), ex1.pop("_dmap")
        r1 = measure_cold(a1, hb1, args.option_bits, min(args.steps, 10), 3, 6, local_rank, world, dev, gather=False,
                          inflight=args.inflight)
        sec["configs[1]"] = {"workload": wl1, "value": r1["value"], "unit": UNIT, "e2e": r1["e2e_value"],
                             "batches_in_flight": r1["inflight"],
                             "ms_per_step": r1["ms_per_step"], "kernel_ms": r1["kernel_ms"],
                             "mean_admm_iters": float(np.mean(r1["iters"])),
                             "solved_fraction": float(np.mean(r1["status"] == abi.PQP_SOLVED)),
                             "l2_policy": "L2 flushed between timed steps", **ex1}
        try:
            sec["front_end"] = front_end_stages(lines1, dmap1, local_rank)
        except Exception as e:  # report rather than lose the bench line
            sec["front_end"] = {"error": repr(e)}
        if rank == 0:
            try:
                sec["configs[0]"] = dropin_single_path()
            except Exception as e:  # the drop-in binary needs g++ on the box; report rather than lose the line
                sec["configs[0]"] = {"error": repr(e)}
    return fp64, sec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8192, help="instances per GPU per step")
    ap.add_argument("--n", type=int, default=240, help="knots per path")
    ap.add_argument("--cpu-sample", type=int, default=None,
                    help="instances of the CPU baseline leg (default: 2048 inside the b200 arm, the whole batch "
                         "for --impl reference)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip config.fp64 / config.secondary")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--inflight", type=int, default=2,
                    help="batches in flight in the device-resident loop: 2 = consecutive steps alternate between two handles "
                         "on two streams (hides the launch tail of the persistent kernel); 1 = one launch at a time")
    ap.add_argument("--option-bits", type=int, default=128,
                    help="pqp_params.reserved: 2 FP64 iterates, 4 no FP64 escalation, 8 state in tensor memory, "
                         "16 state in shared memory, 32 increment-form ADMM step, 64 textbook form, 128 cold-only "
                         "handle (default for the cold workloads: nothing is ever re-solved, so no warm state is written)")
    ap.add_argument("--workload", default="cold", choices=["cold", "receding", "sharedmap"],
                    help="cold: BASELINE configs[2]/[3] (default); receding: configs[4], warm re-solves with a "
                         "50-iteration cap on a window that advances one knot per step; sharedmap: configs[1], "
                         "1024 paths x 120 knots through the shared obstacle map")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned for rank 0's batch (solution, "
                         "cost, status, iterations) as DIR/<name>.npy in float64, at most 64 MB in all (a seeded "
                         "sample of instances beyond that; DIR/instance.npy lists them)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.workload == "receding" and args.batch == 8192:
        args.batch = 512  # configs[4]: 4096 instances over 8 GPUs
    if args.workload == "sharedmap":
        if args.batch == 8192:
            args.batch = 1024
        if args.n == 240:
            args.n = 120
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    if args.workload == "receding":
        line = run_receding(args, rank, local_rank, world, dev, dump_dir=args.dump_outputs)
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    B, n = args.batch, args.n
    # this rank's shard of the global batch (weak scaling: B instances per GPU)
    hb, workload, extras = make_workload(args, B, rank * B, device=local_rank)
    extras.pop("_lines", None)
    extras.pop("_dmap", None)
    r = measure_cold(args, hb, args.option_bits, args.steps, args.warmup, args.e2e_steps or args.steps, local_rank,
                     world, dev, gather=True, clocks=True, inflight=args.inflight, dump_dir=args.dump_outputs)
    fp64, sec = (None, None) if args.no_secondary else secondary(args, rank, local_rank, world, dev, hb)

    if rank == 0:
        params, info = r["params"], r["info"]
        peak, peak_src = hbm_peak()
        bytes_per_launch = B * algorithmic_bytes(n)
        achieved = bytes_per_launch / (r["kernel_ms"] * 1e-3) / 1e9
        cold_only = bool(args.option_bits & 128)
        line = {
            "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": workload,
                **extras,
                "n_knots": n, "batch_per_gpu": B, "global_batch": world * B, "parallelism": "dp%d" % world,
                "eps_abs": params.eps_abs, "eps_rel": params.eps_rel, "max_iter": params.max_iter,
                "l2_policy": ("inputs larger than L2 (%.0f MB per step vs 126 MB)" % (hb.knots.nbytes / 1e6))
                if not r["flushed"] else "L2 flushed between timed steps (256 MB fill inside the timed region)",
                "collective": ("all_gather of {cost,status,iters} (16 B/instance): one pack kernel + NCCL on a side "
                               "stream, overlapping the next step's solve; the timed region ends after the last gather")
                if world > 1 else "none",
                "mean_admm_iters": float(np.mean(r["iters"])),
                "solved_fraction": float(np.mean(r["status"] == abi.PQP_SOLVED)),
                "warps_per_sm": info["warps_per_sm"], "smem_per_warp": info["smem_per_warp"],
                "kernel_ms_per_rank": {"min": min(r["kernel_ms_per_rank"]), "max": max(r["kernel_ms_per_rank"]),
                                       "all": r["kernel_ms_per_rank"]},
                "option_bits": args.option_bits,
                "batches_in_flight": r["inflight"],
                "step_overlap": ("consecutive steps run on two handles / two streams: the next batch takes over SMs as the "
                                 "previous batch's persistent CTAs drain (each step is one full batch; `roofline.kernel_ms` is a "
                                 "launch timed alone)") if r["inflight"] > 1 else "none: one launch at a time",
                "warm_state": "not kept (cold-only handle, option bit 128: these batches are solved once)" if cold_only
                else "kept per instance for pqp_resolve",
                "admm_step": ("increment form (dx solve, carried row values)"
                              if (args.option_bits & 32) or (not (args.option_bits & (64 | 2)) and n >= 64)
                              else "textbook form"),
                "state_storage": ("tensor memory (tcgen05.ld/st), persistent CTAs; %d KB of shared memory per warp for the groups "
                                  "that do not fit the warp's columns" % (info["smem_per_warp"] // 1024))
                                 if sv_uses_tmem(n, B) else "shared memory",
            },
            "clocks": r["clocks"],
            "e2e": {"value": r["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                    "steps": r["e2e_steps"], "batches_in_flight": r["inflight"], "host_numa_node": numa,
                    "how": "every step = one synchronous pqp_solve of the whole batch, pinned host inputs -> pinned host "
                           "results; %d handle(s), one host thread per handle" % r["inflight"]},
            "gpu_launches": r["launches"],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": measured_traffic(n, B, cold_only), "peak_source": peak_src,
                         "kernel": "pqp_admm_kernel_tmem", "kernel_ms": r["kernel_ms"],
                         "algorithmic_bytes_per_launch": bytes_per_launch,
                         "issue": measured_issue(n, cold_only),
                         "note": "per-iteration state is on-chip (tensor memory / shared memory); the path is "
                                 "latency/issue bound, not HBM bound (see DESIGN.md)"},
        }
        if fp64 is not None:
            line["config"]["fp64"] = fp64
            line["config"]["secondary"] = sec
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(params, hb, args.cpu_sample or 2048)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
