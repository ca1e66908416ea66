#!/usr/bin/env python
"""bench.py — IK solves/s of the bio2_memetic population loop (BASELINE.json metric).

One "step" = one pass of the hot path over one batch: B independent PR2-like 7-DOF PoseGoal queries,
pop=128, 200 generations per species (= 25 solver step()s), on each GPU (weak scaling: every rank
solves its own B-query shard; N>1 adds one NCCL all-gather of the result slab per pass).

  value      device-resident inputs, CUDA-event timed, max over ranks          (whole-job solves/s)
  e2e        the public host-buffer API (bioik_solve_batch): pinned host inputs, H2D + D2H inside
  roofline   dominant kernel vs the bound that binds it, the FP64 pipe: algorithmic flops (SURVEY.md §8(d)) / its CUDA-event time
             over the measured DFMA peak (profiles/fp64_peak.json); the HBM view (real DRAM traffic / time) beside it
  other_configs (N=1, cfg2 run only)   BASELINE.json configs[2..4]: GPU value, e2e, CPU arm, ratio, FP64 fraction
  cpu_baseline / --impl reference   the reference's own bio2_memetic code compiled with its Release flags
             (oracle/_ref/libbioik_ref_fast.so, kind "reference"; child pool re-sized to pop=128 by the harness),
             else the oracle port (kind "port"); all usable host threads, bounded sample of the same workload
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

METRIC = "IK solves/sec (PR2 7-DOF, pop=128, 200 gens)"
UNIT = "solves/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2")
    ap.add_argument("--batch", type=int, default=10000)
    ap.add_argument("--population", type=int, default=128)
    ap.add_argument("--solver-steps", type=int, default=25)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-other-configs", action="store_true", help="skip the cfg3/cfg4/cfg5 table of the default cfg2 run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed pass returned (solutions, fitness, success, steps of every query) "
                                                          "as DIR/<name>.npy in float64, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, slab, n_vars, B):
    """The answers a caller of the timed path receives, from its [B][n_vars + 3] result slab (all ranks' queries in query order).
    Above DUMP_MAX_BYTES only a fixed, seeded sample of the queries is written, their indices in query_index.npy."""
    from bio_ik_b200.distributed import unpack_slab
    os.makedirs(out_dir, exist_ok=True)
    out = unpack_slab(slab, n_vars, B)
    rows = DUMP_MAX_BYTES // ((n_vars + 4) * 8)
    if B > rows:
        idx = np.sort(np.random.default_rng(0).choice(B, rows, replace=False))
        out = {k: v[idx] for k, v in out.items()}
        out["query_index"] = idx
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons while the timed region runs (NVML every 20 ms; nvidia-smi fallback)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.mx, self.reasons, self._stop_evt = index, [], [], set(), threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml, self.handle = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        self.sm.append(float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
        self.mx.append(float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)))
        get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        r = get(h)
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        for k, b in bits.items():
            if r & b:
                self.reasons.add(k)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
        f = [x.strip() for x in out.split(",")]
        self.sm.append(float(f[0]))
        self.mx.append(float(f[1]))
        for i, k in enumerate(self.NAMES):
            if f[2 + i].lower().startswith("active"):
                self.reasons.add(k)

    def run(self):
        while not self._stop_evt.is_set():
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            self._stop_evt.wait(0.02 if self.nvml else 0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons), "samples": len(self.sm),
                "source": "nvml" if self.nvml else "nvidia-smi"}


def make_workload(args, fk):
    from bio_ik_b200 import workloads
    f, cid = workloads.CONFIGS[args.config]
    w = f(args.batch) if args.config != "cfg1" else f()
    return w, cid


def usable_cpus():
    """CPUs this process may actually use: min(affinity, cgroup cpu.max quota).  The GPU box exposes 128 hardware
    threads but its container is capped (cpu.max) — oversubscribing the quota only slows the CPU arm down."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(round(int(quota) / int(period)))))
    except Exception:
        pass
    return n


def cpu_solver():
    """(object with .solve(...), kind): the reference's own code built with its Release flags when oracle/_ref/ holds
    it (built here from /root/reference by __graft_entry__.build(); the prebuilt .so travels to the GPU box), else the
    oracle port built with the same flags."""
    import oracle_lib
    if os.path.exists(oracle_lib.ref_lib_path("fast")) and not os.environ.get("BIOIK_BENCH_CPU_PORT"):
        try:
            return oracle_lib.Reference("fast"), "reference"
        except OSError:
            pass
    o = oracle_lib.Oracle("fast")
    o.tables(1)
    return o, "port"


def cpu_rate(args, w_small, seconds, config=None):
    """Times the CPU implementation on all usable host threads over a bounded sample of the workload.
    Returns (solves/s, threads, kind, sample description)."""
    import oracle_lib
    o, kind = cpu_solver()
    cfg = oracle_lib.make_cfg(population=args.population)
    threads = usable_cpus()
    n0 = min(len(w_small.seeds), max(64, 16 * threads))
    dt0 = None
    for _ in range(2):  # the first call builds the solver prototype and its lookup tables (set-up, not solving): calibrate on the second
        t0 = time.perf_counter()
        o.solve(w_small.robot, w_small.problem, cfg, w_small.goal_params[:n0], w_small.seeds[:n0], w_small.rng_seeds[:n0], args.solver_steps, nthreads=threads)
        dt0 = time.perf_counter() - t0
    n1 = int(max(n0, seconds / max(dt0, 1e-6) * n0))
    reps = -(-n1 // len(w_small.seeds))
    gp, sd, rs = (np.concatenate([a] * reps)[:n1] for a in (w_small.goal_params, w_small.seeds, w_small.rng_seeds))
    t0 = time.perf_counter()
    res = o.solve(w_small.robot, w_small.problem, cfg, gp, sd, rs, args.solver_steps, nthreads=threads)
    dt = time.perf_counter() - t0
    quality = {"success_rate": float(np.mean(res["success"])), "median_fitness": float(np.median(res["fitness"]))}
    return n1 / dt, threads, kind, f"{n1} queries drawn from the {config or args.config} batch, {args.solver_steps} steps, pop {args.population}, {threads} threads, {dt:.1f} s", quality


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores - its own
    ik_evolution_2.cpp / problem.cpp / forward_kinematics.h compiled with its Release flags (oracle/_ref, see
    oracle/Makefile) when present, else the oracle port; all usable threads, each step a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_lib
    o = oracle_lib.Oracle("strict")
    w, cid = make_workload(args, None)
    threads = usable_cpus()
    sample = int(min(args.batch, max(256, 256 * threads)))
    w.generate(lambda rm, pr, v: o.fk(rm, pr, v), B=sample, cfg_id=cid, seed_noise=(0.1 if args.config == "cfg4" else None))
    fast, kind = cpu_solver()
    cfg = oracle_lib.make_cfg(population=args.population)
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res = fast.solve(w.robot, w.problem, cfg, w.goal_params, w.seeds, w.rng_seeds, args.solver_steps, nthreads=threads)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = sample / (ms / 1e3)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": w.name, "batch_per_step": sample, "population": args.population, "solver_steps": args.solver_steps, "generations": 8 * args.solver_steps,
                   "note": ("the reference's own solver sources compiled with its Release flags (oracle/_ref)" if kind == "reference" else "CPU port of the reference path (oracle/_ref absent)")
                           + "; each step = bounded sample of the batch"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": f"{sample} queries per step x {args.steps} steps", "host_hw_threads": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "quality": {"success_rate": float(np.mean(res["success"])), "median_fitness": float(np.median(res["fitness"]))},
    }
    print(json.dumps(line), flush=True)


# algorithmic FP64 flops of one individual-evaluation (SURVEY.md §8(d), FMA = 2) and, where an ncu capture exists, the flops the
# generation kernel's opcode mix really executes per child (profiles/r01_k_evolve_fast_v7.txt: K1's r * rate * span is tabulated)
FLOPS_PER_UNIT = {"cfg1": 252.0, "cfg2": 252.0, "cfg3": 540.0, "cfg4": 1300.0, "cfg5": 924.0}
EXECUTED_FLOPS_PER_UNIT = {"cfg1": 183.0, "cfg2": 183.0}


def fp64_peak(clocks):
    """(TFLOP/s, source): the FP64-pipe peak measured by profiles/fp64_peak.cu on this pool's B200 (independent DFMA chains, all
    SMs, CUDA events), else the nominal pipe width at the sampled clock."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "fp64_peak.json")))
        return float(d["fp64_tflops"]), f"profiles/fp64_peak.json (measured with profiles/fp64_peak.cu: independent DFMA chains on every SM at {d['sm_mhz_during_peak']:.0f} MHz; nominal {d['nominal_tflops_at_that_clock']:.1f})"
    except Exception:
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        return 148 * 64 * 2 * mhz * 1e6 / 1e12, "fallback: nominal 148 SMs x 64 FP64 FMA lanes x 2 x sampled SM clock (profiles/fp64_peak.json absent)"


def measure(args, config, B, steps, warmup, env, cpu_seconds, full, dump_dir=None):
    """One bench measurement of `config` at B queries per GPU: device-resident value, host-buffer e2e, kernel timing, CPU arm.
    env = dict(torch, dist, world, rank, local_rank, dev, stream).  dump_dir: where rank 0 writes the results of the last timed pass."""
    torch, dist, world, rank, dev, stream = env["torch"], env["dist"], env["world"], env["rank"], env["dev"], env["stream"]
    from bio_ik_b200 import workloads
    from bio_ik_b200.distributed import DeviceShardedSolver
    from bio_ik_b200.solver import IKSolver
    f, cid = workloads.CONFIGS[config]
    w = f(B) if config != "cfg1" else f()
    solver = IKSolver(w.robot, mode="bio2_memetic", population=args.population, random_seed=1, device=env["local_rank"]).initialize(w.problem)
    S = args.solver_steps
    n_vars, n, G = w.robot.n_vars, len(w.problem.active_variables), w.problem.n_goals

    # distinct synthetic batches per iteration (targets made reachable by the GPU's own exact FK), resident in HBM
    n_batches = min(steps + warmup, 8)
    batches = []
    for k in range(n_batches):
        w.generate(lambda rm, pr, v: solver.fk(v), B=B, cfg_id=cid + 100 * k + 1000 * rank, seed_noise=(0.1 if config == "cfg4" else None))
        batches.append((w.goal_params.copy(), w.seeds.copy(), w.rng_seeds.copy()))
    d_batches = [(torch.from_numpy(g).to(dev), torch.from_numpy(s).to(dev), torch.from_numpy(r.view(np.int32)).to(dev)) for g, s, r in batches]
    sharded = DeviceShardedSolver(solver, B, dev, stream)  # solve + pack + (N > 1) one all-gather of the result slab per pass
    flush = env["flush"]

    def one_pass(k):
        g, s, r = d_batches[k % n_batches]
        sharded.solve(g, s, r, S)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(env["local_rank"]) if full else None  # started before the warm-up: the timed region itself is only ~0.1 s long
    if sampler:
        sampler.start()
    for k in range(warmup):
        one_pass(k)
    barrier()
    solver.kernel_time(reset=True)
    launches0 = solver.launch_count()
    evs = []
    barrier()
    t_wall0 = time.perf_counter()
    for k in range(steps):
        flush.zero_()  # evict L2 between timed iterations (outside the event pair)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        one_pass(warmup + k)
        b.record(stream)
        evs.append((a, b))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if sampler else None
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, sharded.gathered.cpu().numpy(), n_vars, world * B)
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    launches = solver.launch_count() - launches0
    ev_ms, ev_n, ser_ms, ser_n = solver.kernel_time(reset=True)
    kernel_name = solver.kernel_name()
    success_rate = float(sharded.succ.float().mean().item())
    median_fitness = float(sharded.fit.median().item())
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / steps
    value = world * B / (ms_per_step / 1e3)

    # e2e: the public host-buffer API with pinned host memory; H2D + D2H inside the timed region; at N > 1 also the all-gather of the
    # result slabs (results back to the device, one NCCL all-gather, the full slab read back by every rank)
    def pinned(a):
        tns = torch.from_numpy(a.copy()).pin_memory()
        return tns, tns.numpy()
    hb = [tuple(pinned(x) for x in (g, s, r)) for g, s, r in batches]
    out = dict(solutions=torch.empty((B, n_vars), dtype=torch.float64).pin_memory(), fitness=torch.empty(B, dtype=torch.float64).pin_memory(),
               success=torch.empty(B, dtype=torch.int32).pin_memory(), steps=torch.empty(B, dtype=torch.int32).pin_memory())
    out_np = {k: v.numpy() for k, v in out.items()}
    if world > 1:
        out_np["slab"] = torch.empty((B, n_vars + 3), dtype=torch.float64).pin_memory()
        out_np["gathered"] = torch.empty((world * B, n_vars + 3), dtype=torch.float64).pin_memory()
    solver.kernel_time(disable=True)  # no per-launch events in the end-to-end leg: repeated solves replay a CUDA graph
    for k in range(max(warmup, 3)):
        g, s, r = hb[k % n_batches]
        sharded.solve_host(g[1], s[1], r[1], S, out_np)
    barrier()
    t0 = time.perf_counter()
    for k in range(steps):
        g, s, r = hb[(warmup + k) % n_batches]
        sharded.solve_host(g[1], s[1], r[1], S, out_np)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    e2e_value = world * B * steps / e2e_s
    slab_bytes = B * (n_vars + 3) * 8
    h2d = B * (G * 12 * 8 + n_vars * 8 + 4) + (slab_bytes if world > 1 else 0)
    d2h = B * (n_vars * 8 + 8 + 4 + 4) + (world * slab_bytes if world > 1 else 0)
    res = dict(workload=w.name, robot=w.robot.name, value=value, ms_per_step=ms_per_step, e2e_value=e2e_value, h2d=int(h2d), d2h=int(d2h), launches=int(launches), clocks=clocks,
               quality={"success_rate": success_rate, "median_fitness": median_fitness}, wall_s=t_wall, n=n, n_vars=n_vars, G=G)
    if rank != 0:
        return res

    # Roofline of the dominant kernel.  The population never leaves the chip (genes, gradients, fitness live in registers, the
    # mutation table in L2), so the FP64 pipe binds, not HBM: achieved = algorithmic flops of the generation work / the kernel's
    # CUDA-event time, peak = the measured DFMA peak.  The HBM view is kept beside it: real DRAM traffic of the kernel (ncu) / its time.
    units = B * 2 * 8 * (args.population - 2) * S * steps       # individual-evaluations inside the timed region (per GPU)
    flops_unit = FLOPS_PER_UNIT.get(config, 252.0)
    peak_tf, peak_src = fp64_peak(clocks)
    roofline = None
    if ev_n:
        ach_tf = units * flops_unit / (ev_ms * 1e-3) / 1e12
        persistent = kernel_name.startswith("k_persist")
        roofline = {"bound": "fp64", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf, "traffic": None, "peak_source": peak_src,
                    "kernel": kernel_name, "kernel_launches": int(ev_n), "kernel_ms_per_launch": ev_ms / ev_n, "kernel_share_of_step": ev_ms / total_ms if total_ms else None,
                    "other_kernels_ms_per_step": ser_ms / max(steps, 1), "algorithmic_flops_per_unit": flops_unit, "units_per_step": units // steps,
                    "note": "unit = one individual-evaluation (reproduce + approximate phenotype + goal fitness), SURVEY.md §8(d); "
                            + ("the kernel also carries the memetic line search, exact FK, Jacobian and species block of every step, which the algorithmic count does not credit"
                               if persistent else "one launch per step(); the per-task serial work runs in the other kernels")}
        if config in EXECUTED_FLOPS_PER_UNIT:
            ex = units * EXECUTED_FLOPS_PER_UNIT[config] / (ev_ms * 1e-3) / 1e12
            roofline["executed"] = {"flops_per_unit": EXECUTED_FLOPS_PER_UNIT[config], "achieved": ex, "frac": ex / peak_tf,
                                    "note": "flops of the instructions really issued per child (opcode mix of the ncu capture): K1's r * rate * span is tabulated once per problem"}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm = {"peak": hbm_peak, "unit": "GB/s", "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s", "achieved": None, "frac": None,
               "algorithmic_bytes_per_unit": 24 * n + 8, "note": "not the bound: the state is L2/shared-memory resident by design; achieved = measured DRAM bytes of the kernel / its time"}
        tp = os.path.join(ROOT, "profiles", "evolve_traffic.json")
        if os.path.exists(tp) and config == "cfg2" and args.population == 128 and B == 10000:  # the shape the committed ncu capture was taken on
            try:
                tr = json.load(open(tp))
                if tr.get("kernel", "").split("<")[0] == kernel_name.split("<")[0]:
                    roofline["traffic"] = tr.get("dram_bytes_per_launch")
                    hbm["achieved"] = roofline["traffic"] / (ev_ms / ev_n * 1e-3) / 1e9
                    hbm["frac"] = hbm["achieved"] / hbm_peak
                    hbm["traffic_source"] = tr.get("source")
            except Exception:
                pass
        roofline["hbm"] = hbm
    res["roofline"] = roofline

    cpu = None
    if cpu_seconds > 0 and world == 1:  # the contract asks for it on rank 0 at N=1 only
        wcpu = f(B) if config != "cfg1" else f()
        wcpu.goal_params, wcpu.seeds, wcpu.rng_seeds = batches[0][0], batches[0][1], batches[0][2]
        rate, threads, kind, desc, cpu_quality = cpu_rate(args, wcpu, cpu_seconds, config)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": kind, "sample": desc, "host_hw_threads": os.cpu_count(), "quality": cpu_quality}
    res["cpu_baseline"] = cpu
    solver.close()
    return res


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; bio_ik_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build_cuda()

    stream = torch.cuda.Stream(device=dev)  # the solve, the L2 flush, the events and NCCL all run on this stream
    torch.cuda.set_stream(stream)
    env = dict(torch=torch, dist=dist, world=world, rank=rank, local_rank=local_rank, dev=dev, stream=stream,
               flush=torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev))  # > 126 MB L2
    m = measure(args, args.config, args.batch, args.steps, args.warmup, env, 0.0 if args.no_cpu_baseline else args.cpu_seconds, True, dump_dir=args.dump_outputs)

    # BASELINE.json's other configurations on the same box (N = 1 only): GPU value, e2e, the reference's CPU arm and the bound fraction
    others = None
    if world == 1 and args.config == "cfg2" and not args.no_other_configs:
        others = {}
        for name, b in (("cfg3", 4096), ("cfg4", 2048), ("cfg5", 8192)):
            try:
                o = measure(args, name, b, 3, 3, env, 0.0 if args.no_cpu_baseline else min(args.cpu_seconds, 6.0), False)
                c, r = o.get("cpu_baseline"), o.get("roofline")
                others[name] = {"workload": o["workload"], "batch": b, "value": o["value"], "ms_per_step": o["ms_per_step"], "e2e": o["e2e_value"],
                                "cpu": c["value"] if c else None, "cpu_cores": c["cores"] if c else None, "cpu_kind": c["kind"] if c else None,
                                "e2e_over_cpu": (o["e2e_value"] / c["value"]) if c else None, "fp64_frac": r["frac"] if r else None, "kernel": r["kernel"] if r else None,
                                "success_rate": o["quality"]["success_rate"], "cpu_success_rate": c["quality"]["success_rate"] if c else None}
            except Exception as e:  # a parity configuration must not take the headline line down
                others[name] = {"error": repr(e)}
        if "cfg5" in others and "error" not in others["cfg5"]:
            others["cfg5"]["note"] = "BASELINE configs[4] is 65 536 queries over 8 GPUs = 8192 per GPU: this is the per-GPU shard"
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    B, S = args.batch, args.solver_steps
    line = {
        "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": m["workload"], "batch_per_gpu": B, "population": args.population, "solver_steps": S, "generations": 8 * S, "species": 2, "memetic": "q",
                   "robot": f"{m['robot']} (synthetic link table, no URDF offline)", "l2": "flushed (256 MiB memset) between timed iterations",
                   "parallelism": f"query-sharded x{world}" + (", one NCCL all-gather of the result slab per pass" if world > 1 else ""),
                   "legs": "value: inputs resident in HBM, CUDA events around each pass, L2 flushed before it; e2e: bioik_solve_batch with pinned host buffers (H2D + D2H inside), "
                           "back-to-back passes replaying a CUDA graph with a warm L2 - two different experiments, which is why e2e can exceed value"},
        "clocks": m["clocks"], "gpu_launches": m["launches"],
        "e2e": {"value": m["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"]},
        "roofline": m.get("roofline"), "cpu_baseline": m.get("cpu_baseline"),
        "quality": m["quality"], "wall_s_timed_region": m["wall_s"],
    }
    if others is not None:
        line["other_configs"] = others
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
