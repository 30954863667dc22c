#!/usr/bin/env python
"""Benchmark of the hot path: batched ``Integrator.step`` on B200.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU reference arm
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # + the outputs as .npy

Headline workload (BASELINE.json configs[1], "C1"): dense-mass Euclidean leapfrog on Neal's
funnel, D = 128, 8192 chains per GPU, step size 0.01.  One bench "step" = one launch of
``LEAPFROG_PER_LAUNCH`` fused leapfrog steps over the whole batch (the trajectory loop of
``transitions.py:289-291``).  Metric: aggregate leapfrog steps / s = chains x leapfrog steps /
time.  Prints ONE JSON line (rank 0).

The same line carries, under ``"workloads"``, the other GPU configurations of BASELINE.json
(C2 SoftAbs implicit leapfrog, C3 constrained leapfrog on the torus, C4 dense Riemannian D = 512,
8192 chains per GPU -- 65 536 over 8 GPUs), each with its own CUDA-event time, roofline entry
and (at N = 1) a CPU baseline from the same worker pool, and under ``"strong_scaling"`` the C1
launch with the 8192 chains divided over the N ranks.

CPU arm: the UNMODIFIED reference (``mici``, imported from ``/root/reference/src`` or from the
copy ``oracle/build_ref.sh`` places under ``oracle/_ref``) stepping chains in a process pool with
one worker per usable core (``oracle/ref_baseline.py``).
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# the benchmark writes nothing into the tree (which may be read-only): no bytecode caches, here
# or in the CPU baseline's spawned workers (they inherit the environment)
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

METRIC = "leapfrog steps/sec (aggregate over chains)"
UNIT = "leapfrog steps/s"
WORKLOAD = "C1: dense-mass Euclidean leapfrog, Neal's funnel D=128, 8192 chains per GPU"
N_CHAINS = 8192
DIM = 128
LEAPFROG_PER_LAUNCH = 50
HBM_FALLBACK_GBS = 6650.0
# FP64 peaks of this pool's B200 measured with profiles/tools/fp64_peak.cu
# (profiles/r01_fp64_peak.txt; = 148 SMs x 64 FMA/clk x 1.965 GHz); not in MEASURED_PEAKS.json.
FP64_DMMA_PEAK_TFLOPS = 37.1
FP64_DFMA_PEAK_TFLOPS = 34.1
FP64_PEAK_SOURCE = "constant: profiles/r01_fp64_peak.txt (builder-measured microbenchmark)"

# The other GPU configurations of BASELINE.json.  `launch`: leapfrog steps fused per launch;
# `reps`: timed launches; `cpu`: (chains per worker, steps, seconds) of the CPU sample.
WORKLOADS = {
    "C2": dict(cfg="C2", kwargs={}, launch=2, reps=5, cpu=(2, 2, 4.0),
               label="C2: SoftAbs Riemannian implicit leapfrog, banana D=64, 2048 chains"),
    "C2_dense_hessian": dict(cfg="C6", kwargs={}, launch=2, reps=3, cpu=(2, 2, 4.0),
                             label="C2 with a DENSE Hessian: SoftAbs implicit leapfrog on the "
                                   "quartic target |q|^2/2 + sum_m (a_m.q)^4/4, D=64, 2048 "
                                   "chains (the banana's Hessian is 2x2 block diagonal)"),
    "C3": dict(cfg="C3", kwargs={}, launch=50, reps=10, cpu=(8, 50, 3.0),
               label="C3: constrained leapfrog (RATTLE + Newton), torus D=3 C=1, 4096 chains"),
    "C4": dict(cfg="C4", kwargs={"n_chains": 8192}, launch=1, reps=2, cpu=(1, 1, 5.0),
               label="C4: dense Riemannian implicit leapfrog, quadratic D=512, 8192 chains per "
                     "GPU; metric B + c q q^T factorised per chain (blocked DMMA Cholesky, "
                     "explicit inverse: the reference's algorithm)"),
    "C4_low_rank": dict(cfg="C4", kwargs={"n_chains": 8192}, launch=1, reps=3, cpu=None,
                        metric_overrides={"force_low_rank_form": True},
                        label="C4 with the OPTIONAL Sherman-Morrison policy for the rank-1 "
                              "registry metric (O(D^2) per metric, no factorisation)"),
    "C5": dict(cfg="C5", kwargs={"n_chains": 8192}, launch=1, reps=2, cpu=(1, 1, 5.0),
               label="C5: as C4 with the full-rank metric B + c (q q^T) o S (no low-rank "
                     "shortcut exists), D=512, 8192 chains per GPU"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--leapfrog-per-launch", type=int, default=LEAPFROG_PER_LAUNCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-workloads", action="store_true",
                    help="headline workload only (skip C2 / C3 / C4 and strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed launch returned on "
                         "rank 0 (pos, mom, status, n_done of its chains) as DIR/<name>.npy in "
                         "float64; the inputs are seeded, so runs with the same arguments can "
                         "be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the outputs of the CUDA arm")
    return args


def dump_outputs(out_dir, state):
    """``state``'s arrays as float64 ``out_dir/<name>.npy`` (8192 chains, D = 128: 16 MB)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name in ("pos", "mom", "status", "n_done"):
        arr = getattr(state, name).detach().cpu().numpy().astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:  # noqa: BLE001
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(name):
    """dram bytes per launch of the dominant kernel from the committed ncu capture of this
    workload (profiles/r02_traffic.json, written by profiles/tools/ncu_traffic.py), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            return json.load(f).get(name)
    except Exception:  # noqa: BLE001
        return None


class ClockSampler:
    """Samples SM clock / clock-event reasons during the timed region through NVML (no
    subprocesses: forking from the benchmark process would stall the launch thread)."""

    REASONS = {
        "hw_slowdown": 0x8,
        "sw_power_cap": 0x4,
        "sw_thermal_slowdown": 0x20,
        "hw_thermal_slowdown": 0x40,
    }

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._nvml = None
        try:  # initialise NVML here, outside any timed region
            import pynvml

            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._max = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
            self._nvml = pynvml
        except Exception:  # noqa: BLE001
            pass

    def _run(self):
        pynvml, h, mx = self._nvml, getattr(self, "_h", None), getattr(self, "_max", None)
        if pynvml is None:
            return
        while not self._stop.is_set():
            try:
                self.rows.append((
                    pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), mx,
                    pynvml.nvmlDeviceGetCurrentClocksEventReasons(h),
                    pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0,
                ))
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.004)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=10)

    def summary(self):
        sm = sorted(r[0] for r in self.rows)
        reasons = sorted(k for k, bit in self.REASONS.items() if any(r[2] & bit for r in self.rows))
        return {
            "sm_mhz": sm[len(sm) // 2] if sm else None,
            "sm_max_mhz": self.rows[0][1] if self.rows else None,
            "reasons": reasons,
            "samples": len(self.rows),
            "power_w_max": max((r[3] for r in self.rows), default=None),
        }


# ------------------------------------------------------------------------------- CPU arm


def _cpu_entry(res):
    return {
        "value": res["value"],
        "unit": UNIT,
        "cores": res["cores"],
        "kind": res["kind"],
        "sample": res["sample"],
        "per_core": res["per_core"],
        "probe_per_core": res["probe_per_core"],
        "starved": res["starved"],
        "schedulable_cpus": res["schedulable_cpus"],
        "cgroup_cpu_quota": res["cgroup_cpu_quota"],
        "failed_chains": res["failed_chains"],
        "seconds": res["seconds"],
    }


def cpu_baselines(names, leapfrog_per_launch):
    """CPU samples of C1 and of the workloads in `names` from ONE worker pool (before CUDA is
    initialised in this process)."""
    from oracle import ref_baseline as rb

    pool = rb.Pool()
    out = {}
    try:
        out["C1"] = _cpu_entry(rb.run("C1", {"dim": DIM}, 4, leapfrog_per_launch, 10.0, pool=pool))
        for name in names:
            w = WORKLOADS[name]
            kw = {k: v for k, v in w["kwargs"].items() if k != "n_chains"}
            if w["cpu"] is None:
                continue
            cpw, ns, budget = w["cpu"]
            out[name] = _cpu_entry(rb.run(w["cfg"], kw, cpw, ns, budget, pool=pool))
    finally:
        pool.close()
    return out


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path on all usable host
    cores; every bench step is a bounded sample (1.5 s) of the C1 workload."""
    if rank != 0:
        return
    from oracle import ref_baseline as rb

    pool = rb.Pool()
    vals, res = [], None
    t0 = time.perf_counter()
    try:
        for i in range(args.warmup + args.steps):
            if i == args.warmup:
                t0 = time.perf_counter()
            res = rb.run("C1", {"dim": DIM}, 4, args.leapfrog_per_launch, 1.5, pool=pool,
                         probe=(i == 0))
            if i == 0:
                probe = res["probe_per_core"]
            if i >= args.warmup:
                vals.append(res["value"])
        wall = time.perf_counter() - t0
        extra = {}
        if not args.no_workloads:
            for name, w in WORKLOADS.items():
                if w["cpu"] is None:
                    continue
                kw = {k: v for k, v in w["kwargs"].items() if k != "n_chains"}
                cpw, ns, budget = w["cpu"]
                extra[name] = _cpu_entry(rb.run(w["cfg"], kw, cpw, ns, budget, pool=pool))
    finally:
        pool.close()
    value = sum(vals) / len(vals)
    cores = res["cores"]
    cpu = {"value": value, "unit": UNIT, "cores": cores, "kind": res["kind"],
           "sample": res["sample"] + f"; mean of {args.steps} samples",
           "per_core": value / cores, "probe_per_core": probe,
           "starved": bool(probe and value / cores < 0.5 * probe),
           "schedulable_cpus": res["schedulable_cpus"],
           "cgroup_cpu_quota": res["cgroup_cpu_quota"]}
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": WORKLOAD},
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "workloads": extra,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- CUDA arm


def bind_to_gpu_numa_node(index):
    """Pin this rank's host threads (and therefore its pinned buffers' first touch and its copy
    submission) to the CPUs of the NUMA node the GPU hangs off.  At N = 8 the end-to-end path is
    eight processes pushing cudaMemcpyAsync traffic through the host at once; crossing the
    socket interconnect costs bandwidth.  Returns a short description, or None if unavailable."""
    try:
        import pynvml

        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:  # nvml prints an 8-digit PCI domain, sysfs a 4-digit one
            bus = bus[4:]
        base = f"/sys/bus/pci/devices/{bus}"
        with open(base + "/local_cpulist") as f:
            spec = f.read().strip()
        with open(base + "/numa_node") as f:
            node = int(f.read())
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus)}
    except Exception:  # noqa: BLE001
        pass
    return None


def time_launches(torch, fn, reps, flush=None, park_ms=0.0):
    """Per-launch CUDA-event times (ms) of `fn`, L2 optionally flushed between launches.  With
    `park_ms` the GPU is held busy while the host enqueues all launches, so that the event pairs
    of sub-millisecond kernels contain device time only (no host launch gaps)."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(reps)]
    out = None
    if park_ms > 0.0:
        torch.cuda._sleep(int(park_ms * 1e-3 * 1.9e9))
    for i, (a, b) in enumerate(ev):
        if flush is not None:
            flush.fill_(float(i))
        a.record()
        out = fn()
        b.record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev], out


def run_workload(name, torch, dist, dev, rank, world, flush, hbm_peak):
    """One of the non-headline configurations on this rank; returns a dict (rank 0) with
    aggregate throughput (max launch time over ranks) and the roofline entry."""
    from mici_b200 import engine, problems

    w = WORKLOADS[name]
    kw = dict(w["kwargs"])
    base_seed = {"C2": 2, "C3": 3, "C4": 4, "C5": 7, "C6": 9}[w["cfg"]]
    prob = problems.make_problem(w["cfg"], seed=problems.BASE_SEED + base_seed + 1000 * rank, **kw)
    if w.get("metric_overrides"):
        prob.metric_params = dict(prob.metric_params, **w["metric_overrides"])
    integ = engine.build_integrator(prob)
    state = engine.build_state(prob, dev)
    n, dim = state.pos.shape
    L = w["launch"]
    integ.step_n(state, L)  # warm-up
    integ.step_n(state, L)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    times, out = time_launches(torch, lambda: integ.step_n(state, L), w["reps"], flush,
                               park_ms=10.0 if name == "C3" else 0.0)
    t = torch.tensor([sum(times) / len(times)], dtype=torch.float64, device=dev)
    done = out.n_done.sum().to(torch.float64).reshape(1)
    ok = (out.status == 0).sum().to(torch.float64).reshape(1)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(done)
        dist.all_reduce(ok)
    ms = float(t.item())
    steps_done = float(done.item())
    value = steps_done / (ms * 1e-3)
    iters = None
    if out.solver_iters is not None:
        it = out.solver_iters.to(torch.float64)
        iters = it.mean(0).tolist() if it.ndim > 1 else float(it.mean().item())
    # what the kernels evaluated per leapfrog step, tallied by the kernels themselves
    # (mb200_set_call_counters) in one more untimed launch on this rank
    integ.count_calls()
    cnt_out = integ.step_n(state, L)
    torch.cuda.synchronize(dev)
    cnt_steps = max(1.0, float(cnt_out.n_done.sum().item()))
    counted = {k: v / cnt_steps for k, v in integ.call_count_totals().items()}
    integ.count_calls(False)
    b_alg = prob.algorithmic_bytes_per_chain_step
    res = {
        "workload": w["label"],
        "value": value,
        "unit": UNIT,
        "ms_per_launch": ms,
        "leapfrog_steps_per_launch": L,
        "chains_per_gpu": n,
        "n_gpus": world,
        "dim": dim,
        "ok_fraction": float(ok.item()) / (n * world),
        "mean_solver_iters_last_step": iters,
        "kernel_counted_per_step": counted,
    }
    hbm_gbs = value / world * b_alg / 1e9
    if name in ("C2", "C2_dense_hessian"):
        # metric builds (eigendecompositions) per step: _step_a + every iteration of the two
        # position fixed points + _step_b_adj; quadratic-form gradients: every iteration of the
        # two momentum fixed points + 1.  F_alg = builds * 9 D^3 + quad * 2 D^3 (SURVEY 8(d)).
        builds, quads = counted["metric"], counted["quad_form_vjp"]
        f_alg = builds * 9.0 * dim**3 + quads * 2.0 * dim**3
        tf = value / world * f_alg / 1e12
        res["roofline"] = {
            "bound": "fp64 (scalar pipe: Jacobi eigensolver)", "achieved": tf,
            "peak": FP64_DFMA_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": tf / FP64_DFMA_PEAK_TFLOPS,
            "peak_source": FP64_PEAK_SOURCE, "traffic": ncu_traffic(name),
            "flops_per_chain_step": f_alg, "metric_builds_per_step": builds,
            "formula": "builds*9*D^3 + quad_grads*2*D^3; builds, quad_grads counted in the kernel",
            "hbm_frac": hbm_gbs / hbm_peak,
            "kernel": "implicit_leapfrog_kernel<%s, SoftAbsMetric>"
                      % ("BananaRTarget" if name == "C2" else "QuarticRTarget"),
        }
    elif name == "C3":
        res["roofline"] = {
            "bound": "latency / issue (B_alg = 96 B per chain-step)", "achieved": hbm_gbs,
            "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak,
            "traffic": ncu_traffic(name),
            "kernel": "constrained_torus_thread_kernel (one thread per chain)",
            "newton_iterations_per_step": iters,
        }
    elif name in ("C4", "C5"):
        # per metric build: Cholesky D^3/3 (+ fill); per position fixed-point iteration one
        # M^-1 p = two triangular solves 2 D^2; two explicit inverses per step (the two _step_a
        # kicks need grad_log_abs_det = M^-1): L^-1 (D^3/3) and X^T X (D^3/3); per momentum
        # fixed-point iteration one M^-1 p and the model's VJP (2 D^2)
        builds, quads = counted["metric"], counted["quad_form_vjp"]
        f_exec = (builds * (dim**3 / 3.0 + 2.0 * dim**2) + 2.0 * (2.0 * dim**3 / 3.0)
                  + quads * 4.0 * dim**2 + 2.0 * 2.0 * dim**2)
        tf = value / world * f_exec / 1e12
        res["roofline"] = {
            "bound": "fp64 tensor pipe (DMMA: blocked Cholesky, L^-1, X^T X)", "achieved": tf,
            "peak": FP64_DMMA_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": tf / FP64_DMMA_PEAK_TFLOPS,
            "peak_source": FP64_PEAK_SOURCE, "traffic": ncu_traffic(name),
            "flops_per_chain_step": f_exec, "metric_builds_per_step": builds,
            "formula": "builds*(D^3/3 + 2 D^2) + 2*(2 D^3/3) + quad_grads*4 D^2 + 4 D^2",
            "hbm_frac": hbm_gbs / hbm_peak,
            "kernel": "implicit_leapfrog_kernel<QuadraticRTarget, GlobalDenseMetricT<...>>",
        }
    elif name == "C4_low_rank":
        # the Sherman-Morrison policy never factorises: per metric build 2 D^2 (B^-1 q), per
        # M^-1 v 2 D^2, per target gradient 2 D^2; counted from the iteration counts
        builds, quads = counted["metric"], counted["quad_form_vjp"]
        matvecs = 2.0 * builds + quads + 2.0  # build + M^-1 p per build; M^-1 p per quad; 2 grads
        f_exec = matvecs * 2.0 * dim**2
        f_ref = builds * dim**3 / 3.0 + matvecs * 2.0 * dim**2
        tf = value / world * f_exec / 1e12
        res["roofline"] = {
            "bound": "fp64 (L2-resident mat-vecs against the shared B^-1, P)", "achieved": tf,
            "peak": FP64_DFMA_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": tf / FP64_DFMA_PEAK_TFLOPS,
            "peak_source": FP64_PEAK_SOURCE, "traffic": ncu_traffic(name),
            "flops_per_chain_step_executed": f_exec,
            "flops_per_chain_step_reference_algorithm": f_ref,
            "metric_builds_per_step": builds, "hbm_frac": hbm_gbs / hbm_peak,
            "kernel": "implicit_leapfrog_kernel<QuadraticRTarget, Rank1WoodburyMetric>",
        }
    return res


def run_nuts(torch, dist, dev, rank, world):
    """Row N4: whole dynamic-HMC (NUTS) transitions on C1 -- momentum refresh excluded, one
    launch per transition for all chains (`nuts_dmma_kernel`: 8 chains per CTA in lock-step, the
    mat-vec of every leaf on the tensor pipe).  Leapfrog steps inside the trees per second."""
    from mici_b200 import engine, problems, transitions

    out = {}
    for depth in (6, 8):
        prob = problems.make_problem("C1", n_chains=N_CHAINS, dim=DIM,
                                     seed=problems.BASE_SEED + 11 + 1000 * rank)
        prob.step_size = 0.01
        integ = engine.build_integrator(prob)
        state = engine.build_state(prob, dev)
        gen = torch.Generator(device=dev)
        gen.manual_seed(rank)
        tr = transitions.MultinomialDynamicIntegrationTransition(integ.system, integ,
                                                                 max_tree_depth=depth)
        mom = transitions.IndependentMomentumTransition(integ.system)
        for _ in range(2):
            state, _ = mom.sample(state, gen)
            state, st = tr.sample(state, gen)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        reps, ms, steps = 5, 0.0, 0.0
        for _ in range(reps):
            state, _ = mom.sample(state, gen)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            state, st = tr.sample(state, gen)
            b.record()
            torch.cuda.synchronize(dev)
            ms += a.elapsed_time(b)
            steps += float(st["n_step"].sum().item())
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        sdone = torch.tensor([steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(sdone)
        out[f"max_tree_depth_{depth}"] = {
            "value": float(sdone.item()) / (float(t.item()) * 1e-3), "unit": UNIT,
            "ms_per_transition": float(t.item()) / reps,
            "mean_leapfrog_steps_per_transition": float(sdone.item()) / reps / (N_CHAINS * world),
            "mean_tree_depth": float(st["tree_depth"].double().mean().item()),
            "accept_stat": float(st["accept_stat"].mean().item()),
        }
    return {
        "workload": "N4: MultinomialDynamicIntegrationTransition (NUTS) on C1 (funnel D=128, dense "
                    "metric, 8192 chains per GPU, step size 0.01), uniforms generated on device",
        "kernel": "nuts_dmma_kernel<NealFunnelTarget, 2, 1>",
        "chains_per_gpu": N_CHAINS, "n_gpus": world, "dim": DIM,
        "value": out["max_tree_depth_6"]["value"], "unit": UNIT,
        "roofline": {
            "bound": "tensor (fp64 DMMA: one M^-1 grad product per leaf, 2 D^2 flop)",
            "achieved": out["max_tree_depth_6"]["value"] / world * 2.0 * DIM * DIM / 1e12,
            "peak": FP64_DMMA_PEAK_TFLOPS, "unit": "TFLOP/s",
            "frac": out["max_tree_depth_6"]["value"] / world * 2.0 * DIM * DIM / 1e12
                    / FP64_DMMA_PEAK_TFLOPS,
            "peak_source": FP64_PEAK_SOURCE, "traffic": ncu_traffic("nuts_c1"),
            "formula": "leapfrog steps/s x 2 D^2 (the INIT / START products of a transition are "
                       "not counted)",
        },
        **out,
    }


def run_cuda(args, rank, local_rank, world):
    cpu = None
    extra_names = [] if args.no_workloads else list(WORKLOADS)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baselines(extra_names, args.leapfrog_per_launch)  # before CUDA is initialised

    import numpy as np
    import torch
    import torch.distributed as dist

    from mici_b200 import engine, parallel, problems

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        # NCCL prints its version banner / debug lines to stdout: keep stdout for the JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    L = args.leapfrog_per_launch
    prob = problems.make_problem("C1", n_chains=N_CHAINS, dim=DIM,
                                 seed=problems.BASE_SEED + 1 + 1000 * rank)
    integ = engine.build_integrator(prob)
    state = engine.build_state(prob, dev)
    n, dim = state.pos.shape

    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)  # > 126 MB L2

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- device-resident throughput (value) + per-launch kernel time
    for _ in range(args.warmup):
        integ.step_n(state, L)
    sync_all()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    with sampler as clocks:
        for _ in range(2):  # sampler thread is running: absorb its start-up before timing
            integ.step_n(state, L)
        sync_all()
        out = state
        # Park the GPU while the host enqueues the whole timed sequence, so that the per-launch
        # event pairs contain device time only (no host launch gaps).  If the host was slower
        # than the parking time the measurement is repeated once with a longer park.
        park_ms = 3.0 * args.steps + 10.0
        for attempt in range(2):
            t_host = time.perf_counter()
            torch.cuda._sleep(int(park_ms * 1e-3 * 1.9e9))
            # one more untimed launch right behind the parking kernel: the first kernel after an
            # idle-spin runs a few percent slower (clock / power state), which is not the
            # steady state the K timed launches are meant to show
            flush.fill_(-1.0)
            integ.step_n(state, L)
            for i in range(args.steps):
                flush.fill_(float(i))  # evict q, p, M^-1 from L2 between timed launches
                ev[i][0].record()
                out = integ.step_n(state, L)
                ev[i][1].record()
            host_ms = (time.perf_counter() - t_host) * 1e3
            sync_all()
            if host_ms < 0.8 * park_ms:
                break
            park_ms = 2.0 * host_ms + 10.0
    times_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(times_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    assert int((out.status != 0).sum().item()) == 0 and bool(torch.isfinite(out.pos).all())
    # every timed launch steps the same initial state, so `out` does not depend on how many
    # launches ran before it
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)

    # ---------------- end-to-end through the public API with HOST buffers
    pos_h = torch.as_tensor(prob.pos).pin_memory()
    mom_h = torch.as_tensor(prob.mom).pin_memory()
    pos_o = torch.empty_like(pos_h).pin_memory()
    mom_o = torch.empty_like(mom_h).pin_memory()
    st_o = torch.empty(n, dtype=torch.int32).pin_memory()

    def e2e_step():
        integ.step_n_host(pos_h, mom_h, L, out_pos=pos_o, out_mom=mom_o, out_status=st_o,
                          device=dev, n_chunks=6)

    def timed_e2e(fn):
        for _ in range(args.warmup):
            fn()
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        sync_all()
        wall_ms = (time.perf_counter() - t0) * 1e3
        ms = torch.tensor([max(e0.elapsed_time(e1), wall_ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    e2e_ms = timed_e2e(e2e_step)

    # the same call with PAGEABLE NumPy-backed inputs and outputs (what the reference's
    # ChainState holds, states.py:160-305): no pre-pinned buffers anywhere
    pos_p, mom_p = torch.from_numpy(np.array(prob.pos)), torch.from_numpy(np.array(prob.mom))

    def e2e_pageable_step():
        integ.step_n_host(pos_p, mom_p, L, device=dev, n_chunks=8)

    e2e_pageable_ms = timed_e2e(e2e_pageable_step)

    # ---------------- the other configurations and strong scaling
    hbm_peak, peak_src = measured_hbm_peak()
    workloads = {}
    strong = None
    if not args.no_workloads:
        # C2 / C3 are 1-GPU configurations; C4 is the 8-GPU one (65 536 chains over 8 GPUs)
        names = extra_names if world == 1 else ["C4", "C4_low_rank"]
        for name in names:
            res = run_workload(name, torch, dist, dev, rank, world, flush, hbm_peak)
            if cpu is not None and name in cpu:
                res["cpu_baseline"] = cpu[name]
            workloads[name] = res
        workloads["N4_nuts_C1"] = run_nuts(torch, dist, dev, rank, world)
        # strong scaling: the 8192 chains of C1 divided over the ranks
        n_s = N_CHAINS // world
        sprob = problems.make_problem("C1", n_chains=N_CHAINS, dim=DIM,
                                      seed=problems.BASE_SEED + 1)
        sstate = engine.build_state(sprob, dev, chains=slice(rank * n_s, (rank + 1) * n_s))
        integ.step_n(sstate, L)
        sync_all()
        st_times, _ = time_launches(torch, lambda: integ.step_n(sstate, L), 10, flush,
                                    park_ms=20.0)
        st_ms = torch.tensor([sum(st_times) / len(st_times)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(st_ms, op=dist.ReduceOp.MAX)
        strong = {"total_chains": n_s * world, "chains_per_gpu": n_s,
                  "ms_per_launch": float(st_ms.item()),
                  "value": n_s * world * L / (float(st_ms.item()) * 1e-3), "unit": UNIT}

    # ---------------- write-out: the one collective (outside the timed step path)
    if world > 1:
        gathered = parallel.gather_state(out, n * world, dst=0)
        if rank == 0:
            assert gathered["pos"].shape[0] == n * world

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    chain_steps_per_launch = n * L
    value = world * chain_steps_per_launch * args.steps / (total_ms * 1e-3)
    e2e_value = world * chain_steps_per_launch * args.steps / (e2e_ms * 1e-3)
    e2e_pageable = world * chain_steps_per_launch * args.steps / (e2e_pageable_ms * 1e-3)
    b_alg = prob.algorithmic_bytes_per_chain_step  # 32 * D = 4096 B
    avg_launch_s = (sum(times_ms) / len(times_ms)) * 1e-3
    achieved_gbs = b_alg * chain_steps_per_launch / avg_launch_s / 1e9
    flops = (2.0 * dim * dim) * chain_steps_per_launch / avg_launch_s
    n_launches = args.steps + (sum(w["reps"] for k, w in WORKLOADS.items() if k in workloads))
    if "N4_nuts_C1" in workloads:
        n_launches += 10  # 5 timed transitions at each of the two depths
    line = {
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps,
        "ms_per_step_min_median_max": [min(times_ms), sorted(times_ms)[len(times_ms) // 2],
                                       max(times_ms)],
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic",
        "config": {
            "workload": WORKLOAD,
            "chains_per_gpu": n,
            "dim": dim,
            "leapfrog_steps_per_launch": L,
            "integrator": "LeapfrogIntegrator",
            "metric": "dense (explicit M^-1, shared)",
            "step_size": prob.step_size,
            "l2": "flushed between timed launches (256 MB fill)",
            "parallelism": f"chains sharded over {world} GPU(s), no collective on the step path",
        },
        "roofline": {
            "bound": "hbm",
            "achieved": achieved_gbs,
            "peak": hbm_peak,
            "unit": "GB/s",
            "frac": achieved_gbs / hbm_peak,
            "traffic": ncu_traffic("C1") if (n, dim) == (8192, 128) else None,
            "traffic_source": "profiles/r02_traffic.json (ncu --set full capture of this command)",
            "peak_source": peak_src,
            "kernel": "leapfrog_dmma_kernel<NealFunnelTarget,128>",
            "algorithmic_bytes_per_chain_step": b_alg,
            "fp64_tflops": flops / 1e12,
            "fp64_peak_tflops": FP64_DMMA_PEAK_TFLOPS,
            "fp64_peak_source": FP64_PEAK_SOURCE,
            "fp64_frac": flops / 1e12 / FP64_DMMA_PEAK_TFLOPS,
        },
        "e2e": {
            "value": e2e_value,
            "unit": UNIT,
            "h2d_bytes_per_step": int(2 * n * dim * 8),
            "d2h_bytes_per_step": int(2 * n * dim * 8 + n * 4),
            "buffers": "pinned host tensors in and out",
            "pageable": {"value": e2e_pageable, "unit": UNIT,
                         "buffers": "pageable NumPy-backed tensors in, fresh pageable out"},
            "host_binding": numa,
        },
        "gpu_launches": n_launches,
        "clocks": clocks.summary(),
        "workloads": workloads,
        "strong_scaling": strong,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu["C1"]
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_cuda(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
