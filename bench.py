#!/usr/bin/env python
"""bench.py — agent-env-steps/sec of the gather-trade-build step (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path (random-policy action sampling -> dynamics -> observations) over one batch
of synthetic env replicas: at N GPUs every rank steps its own `envs_per_gpu` replicas (weak scaling, no
collective on the step path).  Rank 0 prints ONE JSON line.

  value     whole-job agent-env-steps/s, inputs and outputs resident in HBM, K steps timed on the device
            (CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks)
  sustained the same K-step region repeated until >= ~1 s of device time has been measured: median over repeats
            (the driver's K is small; this is the number that does not depend on one 3 ms window)
  e2e       the same metric through the C-ABI host entry point with HOST (pinned) buffers: actions copied H2D and
            every observation / mask / reward / done tensor delivered to host memory inside the timed region
  roofline  per-kernel algorithmic bytes / CUDA-event duration against MEASURED_PEAKS.json (HBM)
  cpu_baseline  the CPU oracle (oracle/, a C port of the reference step) on this box's host cores
  workloads the other BASELINE configs (c3, c4 = COVID, c5) measured the same way in the same process (headline c2 only)

Episode phases are staggered before anything is timed (replica e starts at t = e*T/E and one full episode of steps is
run untimed), so every timed window sees the whole episode distribution - full order books, houses, tax days and the
per-step share of auto-resets - instead of 8192 replicas in lock-step at t = 5..25.

--impl reference times the CPU oracle alone (the reference itself is Python and cannot travel to the box).
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

METRIC = "agent-env-steps/sec gather-trade-build"
UNIT = "agent-env-steps/s"

WORKLOADS = {
    # BASELINE.json configs[1]: gather-trade-build, 4 agents, 25x25, 8192 env replicas per B200
    "c2": dict(cfg="c1_tutorial", envs_per_gpu=8192, agents=4, world=[25, 25], steps=None,
               desc="gather-trade-build (layout_from_file/simple_wood_and_stone: Build+CDA+Gather), 4 agents, "
                    "25x25, 8192 env replicas per GPU, uniformly random unmasked actions",
               l2="no explicit flush: each step rewrites 296 MB of observations (> 126 MB L2) and touches 46 MB of state"),
    # BASELINE.json configs[2]: + PeriodicBracketTax planner, 10 agents, 40x40, 65536 envs over 8 GPUs = 8192 per GPU
    "c3": dict(cfg="c3_paper_tax", envs_per_gpu=8192, agents=10, world=[40, 40], steps=100,
               desc="gather-trade-build + PeriodicBracketTax, 10 agents, 40x40, 8192 env replicas per GPU",
               l2="no explicit flush: each step rewrites 390 MB of observations (> 126 MB L2) and touches 87 MB of state"),
    # BASELINE.json configs[3]: COVID-19 scenario (51 US-state agents + federal planner), 4096 envs per GPU
    "c4": dict(cfg="covid", envs_per_gpu=4096, agents=51, world=[1, 1], steps=540,
               desc="COVID-19 + economy (CovidAndEconomySimulation: ControlUSStateOpenCloseStatus + "
                    "FederalGovernmentSubsidy + VaccinationCampaign), 51 state agents + planner, 4096 env replicas per GPU",
               l2="no explicit flush: per-step footprint 163 MB (stringency history re-read every step) > 126 MB L2"),
    # BASELINE.json configs[4]: ContinuousDoubleAuction stress, 64 agents, 64x64, deep book, 16384 envs over 8 GPUs
    "c5": dict(cfg="c5_full", envs_per_gpu=2048, agents=64, world=[64, 64], steps=60, device_reset="snapshot",
               desc="CDA stress (uniform/simple_wood_and_stone: Build+CDA(max_num_orders=50)+Gather, multi-action agents), "
                    "64 agents, 64x64, 2048 env replicas per GPU",
               l2="no explicit flush: each step rewrites 740 MB of observations (> 126 MB L2) and touches 126 MB of state"),
}


# what a caller of the step receives, per workload family (the stepper's output buffers)
GTB_OUTPUTS = ["obs_agent_map", "obs_agent_idx", "obs_agent_flat", "mask_agent", "obs_planner_map", "obs_planner_idx",
               "obs_planner_flat", "obs_planner_agents", "mask_planner", "obs_time", "reward", "done"]
COVID_OUTPUTS = ["obs_agent_state", "obs_postsubsidy", "obs_lagged_stringency", "obs_policy_indicators", "obs_scalars",
                 "mask_agent", "mask_planner", "reward_agent", "reward_planner", "done"]
DUMP_BYTES = 60 * 10 ** 6   # under 64 MB with the .npy headers


def sample_outputs(bufs, names, E):
    """--dump-outputs: the step's output buffers for a fixed, seeded sample of env replicas (all of them when they fit in
    DUMP_BYTES), copied to the host as float32, or float64 where float32 would not hold every value (f64, i32), and the
    sampled replicas' indices as env_index."""
    import torch

    ts = {n: bufs[n] for n in names if n in bufs}
    wide = {n for n, t in ts.items() if t.dtype in (torch.float64, torch.int32, torch.int64)}
    per_env = 8 + sum(t[0].numel() * (8 if n in wide else 4) for n, t in ts.items())   # 8: env_index
    n_env = int(min(E, DUMP_BYTES // max(1, per_env)))
    rows = np.sort(np.random.RandomState(0).choice(E, n_env, replace=False))
    idx = torch.as_tensor(rows, device=next(iter(ts.values())).device)
    out = {n: t.index_select(0, idx).to("cpu", torch.float64 if n in wide else torch.float32).numpy() for n, t in ts.items()}
    out["env_index"] = rows.astype(np.float64)
    return out


def write_outputs(outdir, arrays):
    os.makedirs(outdir, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(outdir, n + ".npy"), a)


def workload_config(key, E):
    """The `config` object of the JSON line - identical for the GPU arm and the reference (CPU) arm."""
    w = WORKLOADS[key]
    return {"workload": w["desc"], "envs_per_gpu": E, "n_agents": w["agents"], "world": w["world"],
            "actions": "uniformly random unmasked actions, drawn on the device inside the timed region", "auto_reset": True,
            "episode_phase": "staggered: replica e starts at t = e*T/E, one untimed episode of steps before timing",
            "l2": w["l2"]}


def host_cores():
    """Host threads this process may actually use (cgroup / affinity aware)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_quota_cores():
    """CPU time the container may use per second of wall clock, in cores (cgroup v2 cpu.max / v1 cfs quota); None: unlimited.
    The CPU arm and the expansion threads of the e2e leg both run under it: a 128-thread host with a 16-core quota delivers
    16 cores' worth of sustained CPU time whatever the thread count."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def cpu_throttle_counters():
    """(nr_throttled, throttled seconds) of this container's cgroup so far; None where the kernel does not say."""
    for path in ("/sys/fs/cgroup/cpu.stat", "/sys/fs/cgroup/cpu/cpu.stat"):
        try:
            kv = dict(line.split()[:2] for line in open(path).read().splitlines() if line.strip())
            if "throttled_usec" in kv:
                return int(kv.get("nr_throttled", 0)), float(kv["throttled_usec"]) * 1e-6
            if "throttled_time" in kv:
                return int(kv.get("nr_throttled", 0)), float(kv["throttled_time"]) * 1e-9
        except Exception:
            pass
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def committed_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the newest committed `ncu --set full`
    capture of this workload (profiles/r*_ncu_full_<kernel>[_<workload>]_raw.csv); None when there is none."""
    import csv
    import glob
    pats = ["r*_ncu_full_%s_%s_raw.csv" % (kernel, workload)]
    if workload == "c2":
        pats.append("r*_ncu_full_%s_raw.csv" % kernel)
    found = sorted(sum((glob.glob(os.path.join(ROOT, "profiles", p)) for p in pats), []),
                   key=lambda p: os.path.basename(p)[:4])  # by round tag
    if not found:
        return None, None
    path = found[-1]
    try:
        rows = list(csv.reader(open(path)))
        d, u = dict(zip(rows[0], rows[2])), dict(zip(rows[0], rows[1]))
        scale = {"Mbyte": 1e6, "Kbyte": 1e3, "Gbyte": 1e9, "byte": 1.0}
        tot = sum(float(d[k].replace(",", "")) * scale.get(u[k], 1.0) for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
        return tot, os.path.relpath(path, ROOT)
    except Exception:
        return None, None


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the measured regions.

    Started before the warm-up steps (nvidia-smi takes a few hundred ms to come up) at a 20 ms period; mark_begin() /
    mark_end() bracket, on the host clock, the K-step timed region plus its `sustained` repeats (the same loop, back to
    back) and only samples time-stamped inside are reported."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t_start = self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            self.t_start = time.time()
            deadline = time.time() + 3.0
            while not self.rows and time.time() < deadline:  # wait for the first sample: nvidia-smi is up
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        import datetime
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        parsed = []
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                parsed.append((ts, float(f[1]), float(f[2]), f[4:8]))
            except ValueError:
                continue
        t0, t1 = self.t0 or 0.0, self.t1 or time.time()
        inside = [p for p in parsed if t0 <= p[0] <= t1 + 0.005]
        window = "timed region + sustained repeats"
        if not inside:
            inside = [p for p in parsed if (self.t_start or 0.0) <= p[0] <= t1 + 0.03]
            window = "warm-up + timed region (measured regions shorter than the 20 ms sampling period)"
        sm, mx, reasons = [p[1] for p in inside], [p[2] for p in inside], set()
        for p in inside:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], p[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (the oracle is test infrastructure; bench.py may execute it only here: cpu_baseline and --impl reference)
# ---------------------------------------------------------------------------------------------------------------------
def covid_oracle_rate(n_envs, steps, warmup=1):
    """agent-env-steps/s of the numpy COVID oracle (single host thread per env loop; numpy releases no parallelism)."""
    from ai_economist_b200.foundation.covid19 import build_covid_params
    from ai_economist_b200.workloads import COVID_KWARGS
    from oracle.covid_oracle import CovidOracleEnv
    p = build_covid_params(**COVID_KWARGS)
    envs = [CovidOracleEnv(p) for _ in range(n_envs)]
    rng = np.random.RandomState(0)
    total = 0.0
    for t in range(warmup + steps):
        acts = [(rng.randint(0, 11, size=51) * (envs[e].t >= envs[e].cooldown_until), 0) for e in range(n_envs)]
        t0 = time.perf_counter()
        for e in range(n_envs):
            envs[e].step(acts[e][0], acts[e][1])
        dt = time.perf_counter() - t0
        if t >= warmup:
            total += dt
    return n_envs * 51 * steps / total, total


class OracleRunner:
    """The C oracle (port of the reference step) over n_envs replicas of one workload, driven with a host-side random
    policy whose sampling is excluded from the timed region (as the device-side sampler is on the GPU side of `value`)."""

    def __init__(self, cfg_name, n_envs, threads, seed0=500000):
        from ai_economist_b200 import foundation, workloads as wl
        from oracle.oracle import OracleBatch

        name, kw = wl.product_kwargs(cfg_name)
        env = foundation.make_env_instance(name, n_envs=n_envs, seed=seed0,
                                           stepper_factory=lambda spec, n, auto_reset: None, **kw)
        self.spec, self.n_envs, self.threads = env.spec, n_envs, threads
        host = env.host_reset_arrays()
        self.orc = OracleBatch(env.spec, n_envs)
        for e in range(n_envs):
            self.orc.load_env(e, {k: v[e] for k, v in host.items()})
        self.seg_a, self.seg_p = wl.mask_segments(env.spec, "a"), wl.mask_segments(env.spec, "p")
        self.sample = wl.sample_from_masks
        self.rng = np.random.RandomState(1)
        self.A = env.spec["n_agents"]

    def run(self, steps, warmup=2):
        total = 0.0
        for t in range(warmup + steps):
            ma, mp = self.orc.masks()           # one C call for every env's masks
            aa = self.sample(ma, self.seg_a, self.rng)
            ap = self.sample(mp, self.seg_p, self.rng) if self.seg_p else None
            t0 = time.perf_counter()
            self.orc.step(aa, ap, n_threads=self.threads)
            dt = time.perf_counter() - t0
            if t >= warmup:
                total += dt
        return (self.n_envs * self.A * steps / total if total > 0 else 0.0), total


def cpu_baseline_for(key, min_seconds=6.0):
    """cpu_baseline object: the oracle on this box's host cores over a bounded sample of the workload (>= ~6 s timed)."""
    w = WORKLOADS[key]
    if key == "c4":
        rate, total = covid_oracle_rate(8, 40)
        return {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": "8 env replicas x 40 steps, numpy oracle (one thread), %.1f s" % total}
    threads = host_cores()
    per_thread = {"c2": 64, "c3": 32, "c5": 4}[key]
    n_cpu = max(threads * per_thread, 256)
    runner = OracleRunner(w["cfg"], n_cpu, threads)
    probe, _ = runner.run(5, warmup=2)
    steps_cpu = int(max(10, min(5000, min_seconds * probe / (n_cpu * runner.A))))
    rate, total = runner.run(steps_cpu, warmup=0)
    return {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "cpu_quota_cores": cpu_quota_cores(),
            "sample": "%d env replicas x %d steps of the same workload on %d pinned host threads "
                      "(C oracle of the reference step), %.1f s" % (n_cpu, steps_cpu, threads, total)}


def reference_numpy_note():
    """The reference's own NumPy step cannot run on the GPU box (/root/reference is not there and its sources may not be
    copied); its per-core rate measured in the build container is committed with the script that produced it."""
    p = os.path.join(ROOT, "profiles", "reference_numpy_step.json")
    try:
        return json.load(open(p))
    except Exception:
        return None


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    key = args.workload
    w = WORKLOADS[key]
    t0 = time.perf_counter()
    if key == "c4":
        threads, n_envs = 1, 8
        rate, total = covid_oracle_rate(n_envs, args.steps, warmup=args.warmup)
        steps_run = args.steps
    else:
        threads = host_cores()
        # every timed step is one pass over a bounded sample of the workload: for c2 at least the full per-GPU batch
        n_envs = max(threads * {"c2": 256, "c3": 64, "c5": 4}[key], {"c2": 8192, "c3": 2048, "c5": 256}[key])
        runner = OracleRunner(w["cfg"], n_envs, threads)
        runner.run(max(0, args.warmup - 2), warmup=2)   # W untimed warm-up steps
        rate, total = runner.run(args.steps, warmup=0)  # exactly K timed steps, each a bounded sample of the workload
        steps_run = args.steps
    line = {
        "impl": "reference", "metric": METRIC if key != "c4" else METRIC.replace("gather-trade-build", "covid19"),
        "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / steps_run, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "i32+f64" if key != "c4" else "f32+f64", "data": "synthetic",
        "config": workload_config(key, w["envs_per_gpu"]),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": threads, "kind": "port", "cpu_quota_cores": cpu_quota_cores(),
                         "sample": "%d env replicas x %d steps per step-sample (C oracle, %d pinned pthreads), %.1f s"
                                   % (n_envs, steps_run, threads, total)},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "reference_numpy_step": reference_numpy_note(),
        "note": "the reference is pure Python and does not exist on the GPU box; this arm times oracle/ (a C "
                "restatement pinned to the reference by golden traces) on every host core it may use, which is far "
                "faster than the reference's own NumPy step (see reference_numpy_step: measured in the build container)",
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# GPU legs
# ---------------------------------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args, rank, world, dev):
        import torch
        import torch.distributed as dist
        self.args, self.rank, self.world, self.dev, self.torch, self.dist = args, rank, world, dev, torch, dist

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        t = self.torch.tensor([float(v)], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def time_steps(self, one_step, k):
        """K steps bracketed by barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks."""
        torch = self.torch
        self.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(k):
            one_step(i)
        ev1.record()
        self.barrier()
        return self.max_over_ranks(ev0.elapsed_time(ev1))

    def sustained(self, one_step, k, first_ms, target_ms=1000.0, max_repeats=200):
        """Repeat the K-step region until ~target_ms of device time is covered; median ms per step over the repeats."""
        reps = int(min(max_repeats, max(2, np.ceil(target_ms / max(first_ms, 1e-3)))))
        per = [first_ms / k]
        for _ in range(reps - 1):
            per.append(self.time_steps(one_step, k) / k)
        return float(np.median(per)), len(per), float(min(per)), float(max(per))


def measure_gtb(ctx, key, K, W, with_cpu, clocks=None, e2e_steps=20, e2e_mode="compact", e2e_threads=0, dump=False):
    """One gather-trade-build workload on this rank's GPU: value / sustained / per-kernel roofline / e2e."""
    import ctypes as C

    torch, args, rank, world, dev = ctx.torch, ctx.args, ctx.rank, ctx.world, ctx.dev
    from ai_economist_b200 import foundation, hostmem, workloads as wl
    from ai_economist_b200.sharding import shard_seeds

    w = WORKLOADS[key]
    E = args.envs_per_gpu or w["envs_per_gpu"]
    name, kw = wl.product_kwargs(w["cfg"])
    t_setup = time.perf_counter()
    # auto-reset semantics.  Default: the product's default for the scenario (reference-exact where a device-side reset
    # exists).  c5's uniform/... scenario regenerates a clumped 64x64 layout at every reset (tens of thousands of Gaussian
    # draws and 7x7 convolutions per env, one warp): with 150-step episodes ~14 of the 2 048 replicas reset in every step and
    # each holds its CTA for milliseconds, so the throughput line uses the snapshot restore - which is what the reference's
    # own GPU wrapper does at reset (WarpDrive save_copy_and_apply_at_reset, env_wrapper.py:299-337) - and the cost of the
    # reference-exact mode is measured next to it (`reset_reference_exact`).
    reset_mode = args.device_reset or w.get("device_reset")
    if reset_mode:
        kw["device_reset"] = reset_mode
    env = foundation.make_env_instance(name, n_envs=E, device=str(dev), seeds=shard_seeds(1000, rank, world, E),
                                       auto_reset=True, **kw)
    env.reset()
    st = env.stepper
    A, d, T = env.n_agents, st.dims, int(env.episode_length)
    # stagger the episode phase: replica e starts its first episode at t = e*T/E, then one episode of untimed steps
    st.state_view("t").copy_((torch.arange(E, device=dev, dtype=torch.int64) * T // E).to(torch.int32))

    # random policy fused into the step: the observation pass draws the next step's unmasked actions (aie_set_fused_policy)
    st.set_fused_policy(1234 + rank)

    def one_step(i):
        st.step()  # ONE launch: dynamics + observations/masks + next actions

    for i in range(T if args.preroll is None else args.preroll):
        one_step(i)
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t_setup

    for i in range(W):
        one_step(i)
    launches0 = st.launch_count()
    if clocks:
        clocks.mark_begin()
    ms_total = ctx.time_steps(one_step, K)
    launches = st.launch_count() - launches0
    outputs = sample_outputs(st.buf, GTB_OUTPUTS, E) if dump else None
    sus_ms, sus_n, sus_min, sus_max = ctx.sustained(one_step, K, ms_total)
    if clocks:
        clocks.mark_end()
    value = world * E * A * K / (ms_total * 1e-3)

    # ---- per-kernel durations (separate pass, CUDA events between the kernels, same stream) ----
    n_prof = 50
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(n_prof)]
    for i in range(n_prof):
        evs[i][0].record(); st.step()
        evs[i][1].record()
    torch.cuda.synchronize()
    k_ms = [None, float(np.mean([evs[i][0].elapsed_time(evs[i][1]) for i in range(n_prof)]))]
    # informational: the stand-alone sampler kernel (not launched in the timed loop) and the two halves of the fused step
    # kernel launched separately
    ev2 = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(10)]
    for i in range(10):
        ev2[i][0].record(); st.sample_random_actions(seed=98)
        ev2[i][1].record(); st.step_dynamics()
        ev2[i][2].record(); st.observe()
        ev2[i][3].record()
    torch.cuda.synchronize()
    k_ms[0] = float(np.mean([ev2[i][0].elapsed_time(ev2[i][1]) for i in range(10)]))
    half_ms = [float(np.mean([ev2[i][j + 1].elapsed_time(ev2[i][j + 2]) for i in range(10)])) for j in range(2)]
    peak, peak_src = peaks()
    ww = d.window * d.window
    obs_bytes = (A * ((d.n_map_channels + 1) * ww * 4 + 2 * ww * 2 + d.flat_agent * 4 + d.mask_agent * 4)
                 + d.flat_planner * 4 + A * d.flat_planner_agent * 4 + d.mask_planner * 4 + 4
                 + (d.n_map_channels * d.height * d.width * 4 + 2 * d.height * d.width * 2
                    if env.spec["planner_gets_spatial_info"] else 0))
    step_bytes = 2 * d.state_bytes + 4 * (A * d.n_act_agent + d.n_act_planner) + 8 * (A + 1) + 4
    # SURVEY §8(d)'s own figure counts a leaner record (no MT19937 key / episode statistics inside it)
    lean_state = d.state_bytes - 4 * 624 - 8 * d.n_stats
    kernels = {
        "aie_step_kernel": {"ms": k_ms[1], "alg_bytes_per_launch": E * (step_bytes + obs_bytes),
                            "what": "fused: TMA record in -> dynamics -> rewards -> observations/masks out -> record out",
                            "unfused_ms": {"dynamics_only": half_ms[0], "observe_only": half_ms[1]}},
        "aie_sample_kernel": {"ms": k_ms[0], "alg_bytes_per_launch": E * (A * d.mask_agent * 4 + A * d.n_act_agent * 4),
                              "what": "stand-alone random policy (aie_sample_random_actions); NOT launched in the timed loop, "
                                      "where the step kernel draws the actions itself"},
    }
    for k in kernels.values():
        k["achieved_gbs"] = k["alg_bytes_per_launch"] / (k["ms"] * 1e-3) / 1e9
        k["frac"] = k["achieved_gbs"] / peak
    dom = "aie_step_kernel"
    traffic, traffic_src = committed_traffic(key, dom)
    survey_bytes = step_bytes - 2 * d.state_bytes + 2 * lean_state + obs_bytes
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["frac"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "alg_bytes_per_env_step": step_bytes + obs_bytes,
                "frac_on_survey_8d_bytes": {"alg_bytes_per_env_step": survey_bytes,
                                            "frac": E * survey_bytes / (kernels[dom]["ms"] * 1e-3) / 1e9 / peak,
                                            "what": "SURVEY §8(d)'s accounting: record without the 2.5 KB MT19937 key and the "
                                                    "episode statistics (both travel in and out with the record here)"},
                "whole_step": {"alg_bytes_per_env_step": d.algorithmic_bytes_per_env_step,
                               "achieved": d.algorithmic_bytes_per_env_step * E / (sus_ms * 1e-3) / 1e9,
                               "frac": d.algorithmic_bytes_per_env_step * E / (sus_ms * 1e-3) / 1e9 / peak},
                "kernels": kernels}

    # ---- e2e through the host entry point with pinned HOST buffers ----
    out_host, out_ptrs, d2h = {}, {}, 0
    for nm in GTB_OUTPUTS:
        if nm in st.buf:
            # pinned host tensors from the package's allocator: blocks of replicas (one transfer slice each) on alternating
            # NUMA nodes, which is what the node-pinned expansion threads of aie_step_host_compact are matched to: every
            # socket has work from the first slice on (ai_economist_b200/hostmem.py)
            try:
                t = hostmem.pinned_empty(st.buf[nm].shape, st.buf[nm].dtype,
                                         numa=os.environ.get("AIE_BENCH_E2E_ALLOC", "blocks") if e2e_mode == "compact" else None)
            except Exception as ex:   # placement is an optimisation: never lose the line over it
                sys.stderr.write("hostmem.pinned_empty failed (%s: %s): plain pinned tensor for %s\n" % (type(ex).__name__, ex, nm))
                t = torch.empty(tuple(st.buf[nm].shape), dtype=st.buf[nm].dtype, pin_memory=True)
            out_host[nm] = t
            out_ptrs[nm] = C.c_void_p(t.data_ptr())
            d2h += t.numel() * t.element_size()
    act_a = torch.zeros(st.buf["actions_agent"].shape, dtype=torch.int32, pin_memory=True)
    act_p = torch.zeros(st.buf["actions_planner"].shape, dtype=torch.int32, pin_memory=True)
    h2d = act_a.numel() * 4 + (act_p.numel() * 4 if d.n_act_planner else 0)
    seg_a, seg_p = wl.mask_segments(env.spec, "a"), wl.mask_segments(env.spec, "p")
    rng = np.random.RandomState(rank)
    st.set_fused_policy(0)   # the e2e leg takes its actions from the host
    out_host["mask_agent"].copy_(st.buf["mask_agent"])
    out_host["mask_planner"].copy_(st.buf["mask_planner"])
    e2e_s, n_e2e, e2e_each = 0.0, max(3, e2e_steps), []
    thr0 = cpu_throttle_counters()
    E2E_WARM = 5   # untimed calls: thread pool start, first touch of the staging buffers, page-table warm-up
    for i in range(n_e2e + E2E_WARM):
        act_a.copy_(torch.from_numpy(wl.sample_from_masks(out_host["mask_agent"].numpy(), seg_a, rng)))
        if seg_p:
            act_p.copy_(torch.from_numpy(wl.sample_from_masks(out_host["mask_planner"].numpy(), seg_p, rng)))
        ctx.barrier() if i == E2E_WARM else torch.cuda.synchronize()
        t0 = time.perf_counter()
        st.step_host(C.c_void_p(act_a.data_ptr()), C.c_void_p(act_p.data_ptr()) if d.n_act_planner else None, out_ptrs,
                     compact=(e2e_mode == "compact"), n_threads=e2e_threads)
        dt = time.perf_counter() - t0  # the host entry points synchronise the stream before returning
        if i >= E2E_WARM:
            e2e_s += dt
            e2e_each.append(dt)
    thr1 = cpu_throttle_counters()
    e2e_value = world * E * A * n_e2e / ctx.max_over_ranks(e2e_s)
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "steps": n_e2e, "warmup_calls": E2E_WARM, "mode": e2e_mode,
           "value_at_median_step": world * E * A / float(np.median(e2e_each)),   # this rank's median call (robust to a stalled step)
           "ms_per_step": {"mean": 1e3 * e2e_s / n_e2e, "median": 1e3 * float(np.median(e2e_each)), "min": 1e3 * min(e2e_each),
                           "max": 1e3 * max(e2e_each)}}
    if e2e_mode == "plain":
        e2e.update(d2h_bytes_per_step=d2h,
                   what="aie_step_host: pinned host actions in, every observation/mask/reward/done tensor copied back "
                        "to pinned host memory each step (PCIe-bound)")
    else:
        e2e.update(d2h_bytes_per_step=E * st.compact_bytes_per_env(), host_tensor_bytes_per_step=d2h, host_threads=e2e_threads,
                   cpu_quota_cores=cpu_quota_cores(), ms_each=[round(1e3 * x, 3) for x in e2e_each],
                   cpu_quota_throttling=(None if thr0 is None or thr1 is None else
                                         {"periods_throttled": thr1[0] - thr0[0], "seconds_throttled": round(thr1[1] - thr0[1], 4),
                                          "what": "cgroup cpu.stat deltas over this leg: the container's CPU quota stopping "
                                                  "the process (all threads) until the next 100 ms period"}),
                   last_call_timing_ms={k: (round(v, 3) if isinstance(v, float) else v) for k, v in st.host_timing().items()},
                   what="aie_step_host_compact: pinned host actions in; every observation/mask/reward/done tensor lands "
                        "in pinned host memory each step, bit-/byte-packed over PCIe and expanded by host threads "
                        "(same bytes in the host tensors as the plain path)")
    res = {
        "value": value, "ms_per_step": ms_total / K, "steps": K, "warmup": W,
        "sustained": {"ms_per_step": sus_ms, "value": world * E * A / (sus_ms * 1e-3), "repeats": sus_n,
                      "min_ms_per_step": sus_min, "max_ms_per_step": sus_max,
                      "what": "median over repeats of the K-step timed region (same loop, same synchronisation)"},
        "config": dict(workload_config(key, E), parallelism="env replicas sharded over %d GPU(s), no collective on "
                       "the step path" % world, setup_s=t_setup, device_reset=("reference-exact (reset_mode 1)"
                       if env.spec.get("reset_mode", 0) == 1 else "snapshot restore (reset_mode 0)")),
        "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "dtype": "i32+f64", "n_agents": A, "outputs": outputs,
    }
    if with_cpu:
        res["cpu_baseline"] = cpu_baseline_for(key)
    del env, st, out_host, act_a, act_p
    torch.cuda.empty_cache()
    if reset_mode == "snapshot" and w.get("device_reset") == "snapshot" and not args.device_reset:
        try:   # the same workload with the reference-exact device reset (layout regenerated on the device at every reset)
            kw2 = dict(kw, device_reset="reference")
            env2 = foundation.make_env_instance(name, n_envs=E, device=str(dev), seeds=shard_seeds(1000, rank, world, E),
                                                auto_reset=True, **kw2)
            env2.reset()
            st2 = env2.stepper
            st2.state_view("t").copy_((torch.arange(E, device=dev, dtype=torch.int64) * T // E).to(torch.int32))
            st2.set_fused_policy(1234 + rank)
            for i in range(30):
                st2.step()
            ms2 = ctx.time_steps(lambda i: st2.step(), 30)
            res["reset_reference_exact"] = {"ms_per_step": ms2 / 30, "value": world * E * A * 30 / (ms2 * 1e-3), "steps": 30,
                                            "resets_per_step": E / float(T),
                                            "what": "same workload, device_reset='reference': every auto-reset regenerates the "
                                                    "clumped layout on the device from the env's own numpy stream (bit-exact with "
                                                    "the reference's reset())"}
            del env2, st2
            torch.cuda.empty_cache()
        except Exception as ex:
            res["reset_reference_exact"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
    return res


def measure_covid(ctx, key, K, W, with_cpu, clocks=None, e2e_steps=20, dump=False):
    """BASELINE config 4: one fused kernel per step (+ the random-policy sampler)."""
    torch, args, rank, world, dev = ctx.torch, ctx.args, ctx.rank, ctx.world, ctx.dev
    from ai_economist_b200 import foundation
    from ai_economist_b200.workloads import covid_reference_config

    w = WORKLOADS[key]
    E = args.envs_per_gpu or w["envs_per_gpu"]
    cfg = covid_reference_config()
    name = cfg.pop("scenario_name")
    env = foundation.make_env_instance(name, n_envs=E, device=str(dev), auto_reset=True, **cfg)
    env.reset()
    st = env.stepper
    S = 51

    def one_step(i):
        st.sample_random_actions(seed=7 + rank)
        st.step()

    for i in range(W):
        one_step(i)
    l0 = st.launch_count()
    if clocks:
        clocks.mark_begin()
    ms_total = ctx.time_steps(one_step, K)
    launches = st.launch_count() - l0
    outputs = sample_outputs(st.buf, COVID_OUTPUTS, E) if dump else None
    sus_ms, sus_n, sus_min, sus_max = ctx.sustained(one_step, K, ms_total, max_repeats=20)
    if clocks:
        clocks.mark_end()
    value = world * E * S * K / (ms_total * 1e-3)
    # per-kernel durations: the cost of the history scan depends on how many stringency changes the window holds, so
    # the event-separated pass replays the SAME stretch of the episode as the timed region (reset, same warm-up)
    env.reset()
    for i in range(W):
        one_step(i)
    n_prof = min(K, 300)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_prof)]
    for i in range(n_prof):
        evs[i][0].record(); st.sample_random_actions(seed=7 + rank)
        evs[i][1].record(); st.step()
        evs[i][2].record()
    torch.cuda.synchronize()
    k_ms = [float(np.mean([evs[i][j].elapsed_time(evs[i][j + 1]) for i in range(n_prof)])) for j in range(2)]
    peak, peak_src = peaks()
    L = env.params["filter_len"]
    out_bytes = 4 * (6 * S + 3 * S + 4 + 11 * S + 21 + S) + 8 + 4
    step_bytes = out_bytes + 2 * (9 * S * 4 + 2 * S * 4 + 16) + (L + 1) * S + S + 4 * S + 4   # + ring read/1-row write + actions
    kernels = {"aie_covid_step_kernel": {"ms": k_ms[1], "alg_bytes_per_launch": E * step_bytes},
               "aie_covid_sample_kernel": {"ms": k_ms[0], "alg_bytes_per_launch": E * (11 * S * 4 + 21 * 4 + 4 * S)}}
    for k in kernels.values():
        k["achieved_gbs"] = k["alg_bytes_per_launch"] / (k["ms"] * 1e-3) / 1e9
        k["frac"] = k["achieved_gbs"] / peak
    dom = "aie_covid_step_kernel"
    traffic, traffic_src = committed_traffic(key, dom)
    # e2e: pinned host actions in, all outputs back
    names = COVID_OUTPUTS
    host = {n: torch.empty(st.buf[n].shape, dtype=st.buf[n].dtype, pin_memory=True) for n in names}
    act_a = torch.zeros((E, S), dtype=torch.int32, pin_memory=True)
    act_p = torch.zeros((E,), dtype=torch.int32, pin_memory=True)
    d2h = sum(t.numel() * t.element_size() for t in host.values())
    rng = np.random.RandomState(rank)
    host["mask_agent"].copy_(st.buf["mask_agent"]); host["mask_planner"].copy_(st.buf["mask_planner"])
    e2e_s, n_e2e = 0.0, max(3, e2e_steps)
    for i in range(n_e2e + 2):
        ma, mp = host["mask_agent"].numpy(), host["mask_planner"].numpy()
        act_a.copy_(torch.from_numpy(np.argmax(ma * (rng.random_sample(ma.shape) + 1e-3), axis=1).astype(np.int32)))
        act_p.copy_(torch.from_numpy(np.argmax(mp * (rng.random_sample(mp.shape) + 1e-3), axis=1).astype(np.int32)))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        st.buf["actions_agent"].copy_(act_a, non_blocking=True); st.buf["actions_planner"].copy_(act_p, non_blocking=True)
        st.step()
        for n in names:
            host[n].copy_(st.buf[n], non_blocking=True)
        torch.cuda.synchronize()
        if i >= 2:
            e2e_s += time.perf_counter() - t0
    e2e_value = world * E * S * n_e2e / ctx.max_over_ranks(e2e_s)
    res = {
        "value": value, "ms_per_step": ms_total / K, "steps": K, "warmup": W,
        "sustained": {"ms_per_step": sus_ms, "value": world * E * S / (sus_ms * 1e-3), "repeats": sus_n,
                      "min_ms_per_step": sus_min, "max_ms_per_step": sus_max,
                      "what": "median over repeats of the K-step timed region"},
        "config": dict(workload_config(key, E), parallelism="env replicas sharded over %d GPU(s), no collective on the "
                       "step path" % world, episode_phase="lock-step (deterministic scenario); the timed region covers "
                       "the episode from the warm-up on, K = 540 is one whole episode"),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": E * (S + 1) * 4, "d2h_bytes_per_step": d2h,
                "steps": n_e2e, "what": "pinned host actions -> device, step, every observation/mask/reward/done tensor "
                                        "back to pinned host"},
        "gpu_launches": launches, "dtype": "f32+f64", "n_agents": S, "outputs": outputs,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                     "frac": kernels[dom]["frac"], "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src, "alg_bytes_per_env_step": step_bytes, "kernels": kernels},
    }
    if with_cpu:
        res["cpu_baseline"] = cpu_baseline_for(key)
    ref = reference_cuda_leg(ctx, env.params, E, min(K, 540), ms_total / K, k_ms[1])
    if ref:
        res["vs_reference_cuda"] = ref
    del env, st, host
    torch.cuda.empty_cache()
    return res


def reference_cuda_leg(ctx, params, E, K, ours_ms_per_step, ours_step_kernel_ms):
    """Baseline leg for config 4: the reference's OWN CUDA kernels (covid19_env_step.cu / covid19_components_step.cu,
    compiled for sm_100a from /root/reference into oracle/_ref/ by oracle/build_ref_covid.py) on the same GPU, same
    number of replicas, launched the way the reference's wrapper launches them (grid = envs, block = 52, five launches
    per step).  Like cpu_baseline this is a reported baseline, never the thing shipped; None when the library was not
    built (no /root/reference at build time).  Its kernels' cost does not depend on the actions (they rewrite the whole
    convolution signal every step), so a fixed action tensor is stepped and its reset copy is left out (in its favour)."""
    try:
        from oracle import build_ref_covid
        if not build_ref_covid.available():
            return None
        from oracle.ref_covid_cuda import RefCovidCuda
    except Exception:
        return None
    torch = ctx.torch
    try:
        ref = RefCovidCuda(params, E, device=str(ctx.dev))
        g = torch.Generator(device=ctx.dev); g.manual_seed(5)
        ref.t["actions_a"].copy_(torch.randint(0, 11, ref.t["actions_a"].shape, device=ctx.dev, generator=g, dtype=torch.int32))
        for i in range(5):
            ref.step()
        ms = ctx.time_steps(lambda i: ref.step(), K)
        out = {"ms_per_step": ms / K, "value": ctx.world * E * 51 * K / (ms * 1e-3), "unit": UNIT, "steps": K, "envs_per_gpu": E,
               "launches_per_step": ref.launches_per_step(), "speedup_whole_step": (ms / K) / ours_ms_per_step,
               "speedup_step_kernel_only": (ms / K) / ours_step_kernel_ms,
               "what": "reference CUDA kernels (sm_100a build of the unmodified sources, nvcc -O3) on this GPU: "
                       "CudaControlUSStateOpenCloseStatusStep, CudaFederalGovernmentSubsidyStep, CudaVaccinationCampaignStep, "
                       "CudaCovidAndEconomySimulationStep, CudaComputeReward; speedup = its ms/step over ours (sampler + step)"}
        del ref
        torch.cuda.empty_cache()
        return out
    except Exception as ex:
        return {"error": "%s: %s" % (type(ex).__name__, ex)}


def compact(res):
    """What a sub-workload contributes to the headline line's `workloads` object."""
    r = res["roofline"]
    return {"value": res["value"], "ms_per_step": res["ms_per_step"], "steps": res["steps"],
            "sustained": {k: res["sustained"][k] for k in ("ms_per_step", "value", "repeats")},
            "roofline": {"kernel": r["kernel"], "frac": r["frac"], "achieved": r["achieved"], "traffic": r["traffic"],
                         "traffic_source": r.get("traffic_source"), "alg_bytes_per_env_step": r["alg_bytes_per_env_step"],
                         "kernel_ms": {k: v["ms"] for k, v in r["kernels"].items()}},
            "e2e": res["e2e"], "gpu_launches": res["gpu_launches"], "n_agents": res["n_agents"],
            "envs_per_gpu": res["config"]["envs_per_gpu"], "device_reset": res["config"].get("device_reset"),
            **({"reset_reference_exact": res["reset_reference_exact"]} if "reset_reference_exact" in res else {}),
            **({"vs_reference_cuda": res["vs_reference_cuda"]} if "vs_reference_cuda" in res else {}),
            **({"cpu_baseline": res["cpu_baseline"]} if "cpu_baseline" in res else {})}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--envs-per-gpu", type=int, default=None)
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--e2e-mode", choices=["plain", "compact"], default="compact",
                    help="transfer format of the e2e leg: plain D2H copies, or the compacted transfer (aie_step_host_compact)")
    ap.add_argument("--e2e-threads", type=int, default=0, help="host threads expanding the compacted transfer (0: auto)")
    ap.add_argument("--device-reset", choices=["reference", "snapshot"], default=None,
                    help="auto-reset semantics (default: per workload; see measure_gtb)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--preroll", type=int, default=None, help="untimed steps after staggering the episode phases (default: one episode)")
    ap.add_argument("--no-extra-workloads", action="store_true",
                    help="headline workload only (skip the c3/c4/c5 entries of `workloads`)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (a fixed, seeded sample of env replicas "
                         "when the whole batch exceeds 64 MB; rank 0's replicas)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)

    import torch
    import torch.distributed as dist

    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    torch.cuda.set_device(local_rank)
    torch.set_num_threads(1)   # no OpenMP team for the small host-side tensor ops of the e2e loop (its idle threads would spin
    #                            on the container's CPU quota); the expansion threads are the library's own
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ctx = Ctx(args, rank, world, dev)
    key = args.workload
    with_cpu = world == 1 and not args.no_cpu_baseline
    clocks = ClockSampler(local_rank) if rank == 0 else None
    if clocks:
        clocks.start()
    fn = measure_covid if key == "c4" else measure_gtb
    if args.e2e_threads == 0:   # expansion threads of the e2e leg: this rank's share of half the host's hardware threads
        # (one per physical core: the expansion is bound by the memory controllers, 48 - 64 threads are as fast as 96 on the
        # 2 x 32-core B200 host and burn half the CPU time, profiles/r02z_e2e_transfer_knobs.txt section 7)
        args.e2e_threads = max(8, host_cores() // (2 * max(1, world)))
    kw = {} if key == "c4" else dict(e2e_mode=args.e2e_mode, e2e_threads=args.e2e_threads)
    res = fn(ctx, key, args.steps, args.warmup, with_cpu, clocks=clocks, e2e_steps=args.e2e_steps,
             dump=bool(args.dump_outputs) and rank == 0, **kw)
    outputs = res.pop("outputs")
    clk = clocks.stop() if clocks else None
    extra = {}
    if key == "c2" and not args.no_extra_workloads and not args.envs_per_gpu:
        for k2 in ("c3", "c4", "c5"):
            f2 = measure_covid if k2 == "c4" else measure_gtb
            kw2 = {} if k2 == "c4" else dict(e2e_mode=args.e2e_mode, e2e_threads=args.e2e_threads)
            try:
                extra[k2] = compact(f2(ctx, k2, WORKLOADS[k2]["steps"], max(3, min(args.warmup, 20)), False, e2e_steps=10, **kw2))
            except Exception as ex:   # the headline line must survive a failing extra workload (all ranks fail alike)
                extra[k2] = {"error": "%s: %s" % (type(ex).__name__, ex)}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        "metric": METRIC if key != "c4" else METRIC.replace("gather-trade-build", "covid19"),
        "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": res["dtype"], "data": "synthetic", "config": res["config"], "clocks": clk, "sustained": res["sustained"],
        "e2e": res["e2e"], "gpu_launches": res["gpu_launches"], "roofline": res["roofline"],
    }
    if "cpu_baseline" in res:
        line["cpu_baseline"] = res["cpu_baseline"]
        line["reference_numpy_step"] = reference_numpy_note()
    if "vs_reference_cuda" in res:
        line["vs_reference_cuda"] = res["vs_reference_cuda"]
    if extra:
        line["workloads"] = extra
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
