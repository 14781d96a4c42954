"""Throughput of generator mode (a fresh random instance per env and episode) against one fixed instance of the same
shape, in the same process: env-steps/s of the fused RANDOM step_sample at N envs, the achieved share of HBM
bandwidth of the algorithmic bytes, and the time of a full-batch reset() (which regenerates every instance).

    python tools/bench_generated.py [--envs 65536] [--steps 300] [--warmup 5] [--rounds 3]

Prints one JSON line (with the GPU's name and power limit).  Timing: CUDA events around `steps` back-to-back launches
(one launch per step), after `warmup` launches; the generated and the fixed-instance runs of a shape alternate, and
each round's rate is reported with the median.  Every env is pre-stepped a different number of transitions first (as
bench.py does), so the timed window sees the stationary mix of episode phases, auto-resets included."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def b_alg(J, M):
    """Algorithmic bytes per env-step of a fixed instance (bench.py, SURVEY.md section 8(d))."""
    return 72 * J + 8 * M + 27


def b_alg_gen(J, M):
    """... plus the env's own tables read every env-step in generator mode: ops (2 B per op), jobs_length (4 B per job)
    and the 64-byte descriptor."""
    return b_alg(J, M) + 2 * J * M + 4 * J + 64


def hbm_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (as bench.py)"


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except Exception:
        pass
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    assert args.warmup >= 3 and args.rounds >= 1
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_generated.py measures on a CUDA device; none is available")
    from jssenv_b200 import JssVecEnv
    from jssenv_b200.instances import generate_instance

    n = args.envs
    peak, peak_src = hbm_peak_gbs()
    shapes = [(100, 20, 2236), (20, 20, 450)]   # (J, M, pre-roll period ~ one masked-random episode)
    result = {"gpu": gpu_info(), "envs": n, "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
              "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "shapes": {}}
    for J, M, period in shapes:
        gen = JssVecEnv(n, {"generator": {"jobs": J, "machines": M, "duration": (1, 99), "seed": 1}}, seed=1, auto_reset=True)
        fixed = JssVecEnv(n, {"instance_path": generate_instance(J, M, (1, 99), 1, 0, 0)}, seed=1, auto_reset=True)
        envs = {"generated": gen, "fixed": fixed}
        acts = {}
        quota = torch.as_tensor((np.arange(n, dtype=np.int64) * 7919) % period, device="cuda")
        for name, env in envs.items():                 # pre-roll: env i takes quota[i] transitions
            env.reset()
            a = env.policy("RANDOM")
            skip = torch.full_like(a, -1)
            for k in range(period):
                env.step_sample(torch.where(quota > k, a, skip), "RANDOM", out=a)
            acts[name] = a
        torch.cuda.synchronize()
        rates = {name: [] for name in envs}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for r in range(args.rounds):
            for name, env in envs.items():             # alternated within each round
                a = acts[name]
                for _ in range(args.warmup):
                    env.step_sample(a, "RANDOM")
                ev0.record()
                for _ in range(args.steps):
                    env.step_sample(a, "RANDOM")
                ev1.record()
                ev1.synchronize()
                rates[name].append(n * args.steps / (ev0.elapsed_time(ev1) * 1e-3))
        st = gen.stats()
        assert st["envs_error"] == 0 and st["episodes"] > 0
        res = {}
        for name, bpe in (("generated", b_alg_gen(J, M)), ("fixed", b_alg(J, M))):
            med = float(np.median(rates[name]))
            res[name] = {"env_steps_per_s": med, "rounds": [float(v) for v in rates[name]],
                         "us_per_step": n / med * 1e6, "bytes_per_env_step": bpe,
                         "achieved_GBps": med * bpe / 1e9, "frac_of_hbm_peak": med * bpe / 1e9 / peak}
        res["generated_over_fixed"] = res["generated"]["env_steps_per_s"] / res["fixed"]["env_steps_per_s"]
        # full-batch reset: regenerates all N instances
        for _ in range(3):
            gen.reset()
        times = []
        for _ in range(10):
            ev0.record()
            gen.reset()
            ev1.record()
            ev1.synchronize()
            times.append(ev0.elapsed_time(ev1) * 1e3)
        res["reset_all_us"] = float(np.median(times))
        result["shapes"][f"{J}x{M}"] = res
        for env in envs.values():
            env.close()
        del gen, fixed, envs
        torch.cuda.synchronize()
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
