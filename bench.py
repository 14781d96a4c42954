#!/usr/bin/env python
"""bench.py -- env steps/sec of the batched job-shop environment on B200.

One "step" = one pass of the hot path over the whole batch: ONE fused launch applies every env's
action (time advance, legal-action heuristics, observation, mask, reward, done all written to HBM)
and samples the next action with the device masked-uniform policy.  Headline workload =
BASELINE.json configs[2]: N = 65 536 concurrent ta80 (100x20) envs per GPU, auto-reset, weak scaling
across GPUs (no per-step communication; one NCCL all-gather of the per-shard episode statistics).

The same JSON line carries, under "configs", the other BASELINE.json configurations measured in the
same run (cfg2 ta01 N=4096, cfg4 ta80 N=262144 in total over the ranks, cfg5 mixed ta01..ta80 with
the on-device FIFO / MWR rules), each with its algorithmic bytes and HBM-roofline fraction, and under
"cpu_baseline" the reference's CPU path timed on this box's host cores: the C oracle port AND the
unmodified Python reference (oracle/_ref, installed by oracle/install_ref.py).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--configs all|none] [--dump-outputs DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

METRIC = "env steps/sec (N=65536 ta80)"
UNIT = "env_steps/s"
TA80_EPISODE = 2236          # masked-random episode length on ta80 (BASELINE.md section 2): pre-roll period


def b_alg(J, M):
    """Algorithmic bytes per env-step (SURVEY.md section 8(d))."""
    return 72 * J + 8 * M + 27


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def usable_cpus():
    """Host parallelism actually available to this process: min(online CPUs, affinity mask, cgroup quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, int(q / per + 0.5)))
        except Exception:
            pass
    return n


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU legs
def cpu_port_leg(instance, budget_s, threads=None):
    """The reference's CPU path restated in C (oracle/jss_oracle.c, kind "port"), masked-uniform policy,
    auto-reset, one env per host thread, all usable host threads.  Returns (steps/s, threads, sample)."""
    from jssenv_b200.instances import load_instance
    from oracle.jss_oracle import OracleEnv
    P = threads or usable_cpus()
    m, d = load_instance(instance)
    envs = [OracleEnv(m, d) for _ in range(P)]
    envs[0].run_random(1, 0, 20000)                   # warm-up
    res = [None] * P

    def work(i):
        res[i] = envs[i].run_random_timed(1, i, budget_s)   # ctypes releases the GIL; bounded by wall time

    ths = [threading.Thread(target=work, args=(i,)) for i in range(P)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    steps = sum(r[0] for r in res)
    return steps / dt, P, (f"{P} host threads (os.cpu_count()={os.cpu_count()}, usable={usable_cpus()}) x {budget_s:.0f} s of "
                           f"{instance} steps (masked-random, auto-reset): {steps} steps")


def py_ref_worker(instance, seconds, seed):
    """ONE worker process of the Python-reference leg: the UNMODIFIED reference JssEnv (oracle/_ref or
    /root/reference through oracle/ref_shim.py), masked-uniform policy (np.flatnonzero + Generator.integers,
    BASELINE.md section 3), auto-reset; 1 s warm-up, then `seconds` of wall time.  Prints one JSON line."""
    import numpy as np
    from oracle.ref_shim import load_reference, reference_instance_path
    JssEnv, _ = load_reference()
    env = JssEnv({"instance_path": reference_instance_path(instance)})
    rng = np.random.default_rng(seed)
    obs = env.reset()
    steps = resets = 0
    t_step = 0.0
    clock = time.perf_counter
    t_warm = clock() + 1.0
    t_end = None
    while True:
        now = clock()
        if t_end is None:
            if now >= t_warm:
                t_end, t_begin, steps, resets, t_step = now + seconds, now, 0, 0, 0.0
        elif now >= t_end:
            break
        legal = np.flatnonzero(obs["action_mask"])
        a = int(legal[rng.integers(len(legal))])
        t0 = clock()
        obs, _, done, _, _ = env.step(a)
        t_step += clock() - t0
        steps += 1
        if done:
            obs = env.reset()
            resets += 1
    print(json.dumps({"steps": steps, "resets": resets, "elapsed": clock() - t_begin, "step_only_s": t_step}))


def python_reference_leg(instance, seconds, procs=None):
    """P worker PROCESSES (the reference is single-threaded Python; the GIL rules out threads), each owning one
    unmodified reference env.  Returns a dict, or {"unavailable": why}."""
    from oracle.ref_shim import reference_available, REFERENCE_ROOT
    if not reference_available():
        return {"unavailable": "unmodified reference not installed (oracle/install_ref.py needs /root/reference)"}
    P = procs or usable_cpus()
    cmd = [sys.executable, os.path.abspath(__file__), "--py-ref-worker", instance, str(seconds)]
    t0 = time.perf_counter()
    ps = [subprocess.Popen(cmd + [str(i)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for i in range(P)]
    outs = []
    for pr in ps:
        so, se = pr.communicate(timeout=seconds * 6 + 120)
        if pr.returncode != 0:
            return {"unavailable": "reference worker failed: " + se.strip().splitlines()[-1][:200]}
        outs.append(json.loads(so.strip().splitlines()[-1]))
    wall = time.perf_counter() - t0
    total = sum(o["steps"] / o["elapsed"] for o in outs)
    step_only = sum(o["step_only_s"] for o in outs) / max(1, sum(o["steps"] for o in outs))
    return {"value": total, "unit": UNIT, "cores": P, "per_core": total / P, "step_only_us": step_only * 1e6,
            "kind": "reference", "cpu": cpu_model(), "source": os.path.relpath(REFERENCE_ROOT, ROOT) if REFERENCE_ROOT.startswith(ROOT) else REFERENCE_ROOT,
            "sample": f"{P} worker processes x {seconds:.0f} s (after 1 s warm-up) of the UNMODIFIED Python reference JssEnv.step() on "
                      f"{instance}, masked-random policy, resets included: {sum(o['steps'] for o in outs)} steps, wall {wall:.1f} s"}


def facade_latency(instance, seconds, device):
    """us per JssEnv.step() through the single-env drop-in facade (one launch + one sync per transition; the
    attributes are numpy reads of a pinned host block), README.md:43-65 loop with the masked-random policy."""
    import numpy as np
    from jssenv_b200 import JssEnv
    env = JssEnv({"instance_path": instance}, device=device)
    rng = np.random.default_rng(0)
    obs = env.reset()
    clock = time.perf_counter
    steps, t_step = 0, 0.0
    t_end = clock() + seconds
    warm = 200
    while clock() < t_end:
        legal = np.flatnonzero(obs["action_mask"])
        a = int(legal[rng.integers(len(legal))])
        t0 = clock()
        obs, _, done, _, _ = env.step(a)
        dt = clock() - t0
        if warm > 0:
            warm -= 1
        else:
            t_step += dt; steps += 1
        if done:
            obs = env.reset()
    env.close()
    return t_step / max(1, steps) * 1e6, steps


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path on all usable host threads.  value = the C oracle port (the
    stronger baseline: ~75x faster per core than the Python original); the unmodified Python reference timed on the
    same box is reported beside it.  Each "step" is one bounded wall-time window of the workload."""
    if rank != 0:
        return
    J, M = 100, 20
    windows = max(1, min(args.steps, 3))
    warm = 1 if args.warmup > 0 else 0
    vals, sample, P = [], "", 1
    for k in range(warm + windows):
        v, P, sample = cpu_port_leg("ta80", 2.0 if k < warm else args.cpu_seconds)
        if k >= warm:
            vals.append(v)
    value = sum(vals) / len(vals)
    pyref = python_reference_leg("ta80", args.cpu_seconds)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": "ta80 (100x20) masked-random, auto-reset, CPU oracle port of the reference step()",
                   "envs": P, "bytes_per_env_step": b_alg(J, M), "timed_windows": windows,
                   "window_seconds": args.cpu_seconds},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": P, "kind": "port", "sample": sample, "cpu": cpu_model(),
                         "python_reference": pyref},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------ GPU legs
def preroll(env, rule, period, torch):
    """Stagger the envs' episode phases deterministically before timing: env i executes (i * 7919) mod `period`
    transitions (auto-reset keeps short episodes cycling), the others are skipped (JSS_ACTION_SKIP), so that a
    short timed window samples the stationary mix of episode phases instead of `period` envs in lock-step."""
    n = env.num_envs
    ids = torch.arange(n, device=env.device, dtype=torch.int64) + int(env.env_id_base)
    quota = ((ids * 7919) % period).to(torch.int32)
    skip = torch.full((n,), -1, dtype=torch.int32, device=env.device)
    for k in range(period):
        a = env.policy(rule)
        env.step(torch.where(quota > k, a, skip))
    return env.policy(rule).clone()


def time_fused_steps(env, rule, acts, warm, steps, torch, dist=None, world=1):
    """`steps` fused launches (apply actions + choose the next ones) between CUDA events on the launching stream."""
    for _ in range(warm):
        *_, acts = env.step_sample(acts, rule)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    l0 = env.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        *_, acts = env.step_sample(acts, rule)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    launches = env.launch_count - l0
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, launches, acts


def config_entry(workload, n_total, ms, steps, mean_balg, peak, launches, world=1, extra=None):
    per_step = ms / steps
    d = {"workload": workload, "envs_total": n_total, "steps": steps, "ms_per_step": per_step,
         "env_steps_per_s": n_total * steps / (ms * 1e-3), "bytes_per_env_step": mean_balg,
         "achieved_GBps_per_gpu": mean_balg * (n_total / world) / (per_step * 1e-3) / 1e9,
         "launches_per_step": launches / steps}
    d["frac_of_hbm_peak"] = d["achieved_GBps_per_gpu"] / peak
    if extra:
        d.update(extra)
    return d


def dump_outputs(directory, env, acts, torch, budget=60_000_000):
    """Write what the last timed step_sample() returned to its caller as float32 .npy files (exact: every value is
    float32 already or an integer below 2**24), so that two builds can be compared output for output.  When the batch
    exceeds `budget` bytes, a fixed seeded sample of the envs is written; env_index.npy holds their indices."""
    import numpy as np
    arrays = {"real_obs": env.real_obs, "action_mask": env.action_mask, "reward": env.reward, "done": env.done,
              "truncated": env._truncated, "next_actions": acts}
    n = env.num_envs
    row_bytes = 4 * (1 + sum(int(np.prod(a.shape[1:])) for a in arrays.values()))
    rows = min(n, budget // row_bytes)
    idx = np.arange(n) if rows == n else np.sort(np.random.default_rng(0).choice(n, rows, replace=False))
    sel = torch.as_tensor(idx, device=env.device)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "env_index.npy"), idx.astype(np.float32))
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a.index_select(0, sel).float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=65536, help="envs per GPU")
    ap.add_argument("--instance", default="ta80")
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--configs", default="all", choices=["all", "none"], help="also measure cfg2 / cfg4 / cfg5")
    ap.add_argument("--config-steps", type=int, default=0, help="timed steps of the secondary configs (default max(K, 300))")
    ap.add_argument("--no-preroll", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    ap.add_argument("--py-ref-worker", nargs=3, metavar=("INSTANCE", "SECONDS", "SEED"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.py_ref_worker:
        py_ref_worker(args.py_ref_worker[0], float(args.py_ref_worker[1]), int(args.py_ref_worker[2]))
        return
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # CPU baselines first (N = 1 only, before any CUDA context exists in this process)
    cpu_baseline = None
    if not args.no_cpu and world == 1:
        v, P, sample = cpu_port_leg(args.instance, args.cpu_seconds)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": P, "kind": "port", "sample": sample, "cpu": cpu_model(),
                        "python_reference": python_reference_leg(args.instance, args.cpu_seconds)}

    import numpy as np
    import torch
    import torch.distributed as dist
    from jssenv_b200 import JssVecEnv
    from jssenv_b200.distributed import all_gather_stats

    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL prints its version banner on stdout at the first collective; keep stdout = ONE JSON line
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    peak, peak_src = load_peaks()
    N = args.envs
    K, W = args.steps, max(3, args.warmup)
    env = JssVecEnv(N, {"instance_path": args.instance}, device=local_rank, auto_reset=True,
                    env_id_base=rank * N, seed=1234)
    J, M = env.jobs, env.machines
    env.reset()
    # clocks are sampled from the pre-roll (the same kernels, ~0.5 s of load) through the timed region: the timed
    # region alone (K launches of ~0.1 ms) is shorter than one nvidia-smi sampling period
    sampler = ClockSampler(local_rank)
    sampler.start()
    if args.no_preroll:
        acts = env.policy("RANDOM").clone()
        for _ in range(3000):
            *_, acts = env.step_sample(acts, "RANDOM")
    else:
        acts = preroll(env, "RANDOM", TA80_EPISODE if J * M >= 2000 else int(1.13 * J * M), torch)
    elapsed_ms, launches, acts = time_fused_steps(env, "RANDOM", acts, W, K, torch, dist, world)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env, acts, torch)
    # the timed region is K launches of ONE kernel (the fused step), bracketed by CUDA events on the
    # launching stream: its average launch duration is elapsed / K (launch gaps, if any, count against us)
    step_kernel_ms = elapsed_ms / K
    stats = all_gather_stats(env.stats())
    value = world * N * K / (elapsed_ms * 1e-3)

    # ---- e2e: the same transitions through the host-buffer API (H2D actions, D2H obs/mask/reward/done)
    e2e = None
    if not args.no_e2e:
        # pipelined host-buffer API: begin(step k) -> wait mask k -> host policy -> begin(step k+1) while the
        # observation of step k is still crossing PCIe into its own pinned buffer -> consume obs k.
        # packed: the observation crosses PCIe as 10-byte integer records per job and is expanded to the exact
        # fp32 (N, J, 7) array by the host pool inside the timed region; plain: 28 bytes of fp32 per job by DMA.
        bound = JssVecEnv.host_configure(0, local_rank)   # pool = usable CPUs / local ranks, on the GPU's NUMA node
        threads = int(env._L.jss_host_threads())

        phase = {}

        def run_e2e(packed, steps, dma_fraction=0.0):
            mask = np.ascontiguousarray(env.action_mask.cpu().numpy())
            env.host_step_begin(env.host_masked_random(mask, 0), packed=packed, dma_fraction=dma_fraction)
            checksum = 0.0
            ph = [0.0, 0.0, 0.0, 0.0]
            clock = time.perf_counter

            def e2e_step(k):
                t0 = clock()
                m, rew, dn = env.host_wait_mask()
                t1 = clock()
                a_next = env.host_masked_random(m, k)
                t2 = clock()
                env.host_step_begin(a_next, packed=packed, dma_fraction=dma_fraction)
                t3 = clock()
                o = env.host_wait_obs(previous=True)         # the step's observation, fp32 on the host
                t4 = clock()
                ph[0] += t1 - t0; ph[1] += t2 - t1; ph[2] += t3 - t2; ph[3] += t4 - t3
                return o

            for k in range(1, 4):
                e2e_step(k)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for k in range(steps):
                obs_host = e2e_step(10 + k)
                checksum += float(obs_host[k % N, 0, 1])      # touch the result
            env.host_wait_obs()
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            n_calls = steps + 3
            phase[("hybrid %.2f" % dma_fraction if dma_fraction > 0 else "packed") if packed else "fp32_dma"] = {
                "wait_mask_ms": ph[0] / n_calls * 1e3, "host_policy_ms": ph[1] / n_calls * 1e3,
                "begin_ms": ph[2] / n_calls * 1e3, "wait_obs_and_expand_ms": ph[3] / n_calls * 1e3}
            return world * N * steps / float(dt.item())

        ms_b, ws_b = int(env._b.mask_stride), int(env._L.jss_host_wire_stride(env._h))
        run_e2e(True, 8)                                  # first touches: pinned buffers are allocated here, not in a timed run
        run_e2e(False, 4)
        # the split between "packed rows + host expansion" and "final fp32 rows by DMA" that balances this box's host
        # cores against its PCIe link, and the worker layout (one CPU per worker vs. confined to the GPU's NUMA node:
        # pinning wins on a quiet host, loses when a neighbour keeps one of the CPUs busy): short calibration runs,
        # then the timed run with the best pair
        # (share 1.0 = everything by DMA: the least host-DRAM traffic, which wins when 8 ranks share one host's memory system)
        calib = {}
        for pin in (1, 0):
            os.environ["JSS_HOST_PIN"] = str(pin)
            JssVecEnv.host_configure(0, local_rank)
            for f in (0.0, 0.1, 0.2, 0.3, 0.45, 0.7, 1.0):
                calib[(pin, f)] = run_e2e(True, 16, f)
        keys = sorted(calib)
        if world > 1:                                     # every rank must pick the same pair
            t = torch.tensor([calib[k] for k in keys], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            calib = dict(zip(keys, t.tolist()))
        pin_best, f_best = max(calib, key=calib.get)
        os.environ["JSS_HOST_PIN"] = str(pin_best)
        bound = JssVecEnv.host_configure(0, local_rank)
        phase.clear()
        v_packed = run_e2e(True, args.e2e_steps, f_best)
        v_plain = run_e2e(False, max(10, args.e2e_steps // 4))
        n_dma = min(N, int(f_best * N) // 256 * 256) if f_best > 0 else 0
        e2e = {"value": v_packed, "unit": UNIT,
               "h2d_bytes_per_step": 4 * N,
               "d2h_bytes_per_step": N * ms_b + (N - n_dma) * ws_b + n_dma * J * 7 * 4 + 16 * N,
               "dma_fraction": f_best, "workers_pinned": bool(pin_best),
               "calibration": {f"pin={k[0]} dma={k[1]}": v for k, v in calib.items()},
               "steps": args.e2e_steps, "host_threads": threads, "numa_bound_cpus": bound,
               "fp32_dma_variant": {"value": v_plain, "d2h_bytes_per_step": N * ms_b + N * J * 7 * 4 + 16 * N},
               "host_ms_per_step": phase,
               "note": "jss_host_step_begin_hybrid / jss_host_wait / jss_host_expand_obs_range (pinned host buffers): H2D actions, "
                       "step kernel, D2H mask + scalar records every step; the observation of a share `dma_fraction` of the envs "
                       "crosses PCIe as final fp32 rows, the rest as packed integer rows (10 B per job) that the host pool expands "
                       "to the exact fp32 (N, J, 7) observation; expansion and the host masked-random policy are inside the timed "
                       "region; fp32_dma_variant = everything as 28 B per job of fp32 real_obs over PCIe (the round-1 path)"}
    env.close()
    del env

    # ---- the other BASELINE.json configurations, same run, same timing method
    configs = {}
    if args.configs == "all":
        KC = args.config_steps or max(K, 300)
        if world == 1:
            # cfg2: ta01 N = 4096, masked-random
            e2 = JssVecEnv(4096, {"instance_path": "ta01"}, device=local_rank, auto_reset=True, seed=1)
            e2.reset()
            e2.rollout("RANDOM", 20000, write_obs=True)     # ~80 ms of load: the small-batch timings below are a few ms long
            torch.cuda.synchronize()                         # and must not start on a GPU that idled down its clocks
            e2.reset()
            a2 = e2.policy("RANDOM").clone() if args.no_preroll else preroll(e2, "RANDOM", 253, torch)
            ms, ln, a2 = time_fused_steps(e2, "RANDOM", a2, W, KC, torch)
            configs["cfg2_ta01_N4096_random"] = config_entry(
                "ta01 (15x15) N=4096, masked-random, one fused launch per step, obs/mask/reward/done written every step",
                4096, ms, KC, b_alg(15, 15), peak, ln,
                extra={"note": "5 MB per step: L2-resident and < 1 wave (4096 warps) -> launch/latency-bound by construction"})
            # the same workload as a K-step fused device loop that RECORDS the trajectory: every transition's
            # observation / mask / reward / done / action is kept in [K][N][...] buffers (jss_rollout_traj)
            KR, reps = 256, 8
            tr = e2.rollout_record("RANDOM", KR)
            tr = e2.rollout_record("RANDOM", KR, out=tr)
            torch.cuda.synchronize()
            l0 = e2.launch_count
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(reps):
                tr = e2.rollout_record("RANDOM", KR, out=tr)
            ev1.record()
            torch.cuda.synchronize()
            configs["cfg2_ta01_N4096_random_rollout_record"] = config_entry(
                f"ta01 (15x15) N=4096, masked-random, {KR} transitions per launch in one fused device loop, EVERY transition's "
                "obs/mask/reward/done/action recorded into [K][N][...] trajectory buffers",
                4096, ev0.elapsed_time(ev1), KR * reps, b_alg(15, 15), peak, e2.launch_count - l0,
                extra={"trajectory_bytes_per_env_step": 15 * 7 * 4 + int(e2._b.mask_stride) + 16 + 4})
            del tr
            e2.close()
            del e2
            # cfg5: mixed ta01..ta80 N = 65536, on-device FIFO / MWR (+ masked-random for comparison)
            names = ["ta%02d" % (k + 1) for k in range(80)]
            n5 = 65536
            e5 = JssVecEnv(n5, {"instance_paths": names, "env_to_instance": np.arange(n5) % 80}, device=local_rank,
                           auto_reset=True, seed=2)
            balg5 = float(np.mean([b_alg(int(j), int(m)) for j, m in zip(e5.env_jobs, e5.env_machines)]))
            for rule in ("FIFO", "MWR", "RANDOM"):
                e5.reset()
                a5 = e5.policy(rule).clone() if args.no_preroll else preroll(e5, rule, TA80_EPISODE, torch)
                ms, ln, a5 = time_fused_steps(e5, rule, a5, W, KC, torch)
                configs[f"cfg5_mixed_ta01-80_N65536_{rule}"] = config_entry(
                    f"env i runs ta((i mod 80)+1), N=65536, on-device {rule} rule (10 % no-op coin from the counter RNG), "
                    "fused step + rule per step, obs written every step", n5, ms, KC, balg5, peak, ln)
            e5.close()
            del e5
            # cfg1: ta01 single env through the drop-in facade (the GPU path; there is no CPU product path): latency per
            # step() next to the unmodified Python reference's step() on the same box
            fac = {}
            for inst in ("ta01", "ta80"):
                us, n_st = facade_latency(inst, 1.5, local_rank)
                ref = python_reference_leg(inst, 2.0, procs=1) if not args.no_cpu else {"unavailable": "--no-cpu"}
                fac[inst] = {"facade_us_per_step": us, "steps": n_st,
                             "python_reference_us_per_step": ref.get("step_only_us"), "python_reference": ref.get("unavailable")}
            configs["cfg1_single_env_facade"] = {
                "workload": "JssEnv(env_config).step(a) one env at a time (gym.make('jss-v1') drop-in), masked-random policy: one fused "
                            "step+decode launch and one stream sync per transition, outputs written by the GPU straight into pinned host memory",
                **fac}
        # cfg4 as stated: ta80 N = 262144 IN TOTAL, sharded over the ranks (8 x 32768 at --gpus 8)
        n4 = 262144 // world
        e4 = JssVecEnv(n4, {"instance_path": "ta80"}, device=local_rank, auto_reset=True, env_id_base=rank * n4, seed=4)
        e4.reset()
        a4 = e4.policy("RANDOM").clone() if args.no_preroll else preroll(e4, "RANDOM", TA80_EPISODE, torch)
        ms, ln, a4 = time_fused_steps(e4, "RANDOM", a4, W, KC, torch, dist, world)
        st4 = all_gather_stats(e4.stats())
        configs["cfg4_ta80_N262144_total"] = config_entry(
            f"ta80 N=262144 in total = {world} x {n4} (contiguous shards, no per-step communication, NCCL all-gather of the "
            "per-shard statistics)", 262144, ms, KC, b_alg(100, 20), peak, ln, world=world,
            extra={"scaling": "strong", "episodes_gathered": st4["episodes"]})
        e4.close()
        del e4

    if rank == 0:
        balg = b_alg(J, M)
        achieved = balg * N / (step_kernel_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None               # dram__bytes_read+write per launch: OFFLINE data from the committed ncu capture
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tj["n_envs"] == N and tj["instance"] == args.instance:
                traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
                traffic_src = "offline: ncu --set full capture committed under profiles/ (" + tj.get("source", "traffic.json") + ")"
        except Exception:
            pass
        kj = 1 if J <= 32 else (2 if J <= 64 else (4 if J <= 128 else 8))
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": elapsed_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": {"workload": f"{args.instance} ({J}x{M}) N={N} per GPU, one fused launch per step (apply actions + masked-random "
                                   "sampling of the next ones), auto-reset", "envs_per_gpu": N, "parallelism": f"env-shard x{world}",
                       "l2": "per-step working set (state 140 MB + obs 190 MB at N=65536) exceeds the 126 MB L2",
                       "preroll": "none" if args.no_preroll else "env i pre-stepped (i*7919 mod 2236) transitions: the timed window sees the stationary mix of episode phases",
                       "bytes_per_env_step": balg},
            "clocks": clocks, "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes_per_launch": balg * N,
                         "kernel": f"jss_step_kernel<KJ={kj}, fused sampler, uniform batch>", "kernel_ms": step_kernel_ms,
                         "peak_source": peak_src},
            "episode_stats": stats,
        }
        if e2e:
            out["e2e"] = e2e
        if configs:
            out["configs"] = configs
        if cpu_baseline:
            out["cpu_baseline"] = cpu_baseline
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
