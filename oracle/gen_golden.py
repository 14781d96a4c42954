"""Generate the committed golden fixtures under tests/golden/ from the UNMODIFIED
Python reference.  Run in the build container only (needs /root/reference):

    python oracle/gen_golden.py

Outputs
  tests/golden/optimal_sequences.json   the 12 per-machine optimal job orders and
                                        makespans held by the reference's own
                                        tests/test_solutions.py (known-answer tests)
  tests/golden/trace_<inst>_<policy>.npz  step-by-step traces of the reference env:
        actions[T], mask[T+1, J+1] (row 0 = after reset), obs[T+1, J, 7] float64,
        reward[T] float64, done[T], t[T+1], nb_legal[T+1], nb_machine_legal[T+1],
        plus the integer state arrays after every step, stored in the lossless compact
        form of compact_trace() (tests/helpers.py load_trace() reads both forms)
  tests/golden/known_answers.json       steps / makespan / sum(reward) of whole episodes under the
                                        deterministic "lowest/highest legal index" policies
  tests/golden/cr_factor_makespans.json CriticalRatio(due_date_factor=1.0 / 2.25 / 4.0), np.random.seed(0)
  tests/golden/rule_makespans.json      makespans of every dispatching rule with
                                        np.random.seed(0) before run_episode
"""
import ast
import json
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from oracle.ref_shim import REFERENCE_ROOT, load_reference, reference_instance_path  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def extract_optimal_sequences():
    """Pull `solution_sequence` and the asserted makespan out of each
    test_optimum_* method of the reference's tests/test_solutions.py."""
    path = os.path.join(REFERENCE_ROOT, "tests", "test_solutions.py")
    tree = ast.parse(open(path).read())
    out = {}
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name.startswith("test_optimum_"):
            inst = node.name[len("test_optimum_"):]
            seq, makespan, wait = None, None, None
            for sub in ast.walk(node):
                if isinstance(sub, ast.Assign) and getattr(sub.targets[0], "id", None) == "solution_sequence":
                    seq = ast.literal_eval(sub.value)
                if isinstance(sub, ast.Call) and getattr(sub.func, "attr", None) == "assertEqual":
                    a0, a1 = sub.args[0], sub.args[1]
                    if (isinstance(a0, ast.Attribute) and a0.attr == "current_time_step"
                            and isinstance(a1, ast.Constant) and a1.value != 0):
                        makespan = a1.value
                if isinstance(sub, ast.Call) and getattr(sub.func, "attr", None) == "increase_time_step":
                    wait = "increase_time_step"   # ta01 waits with the raw hook (test_solutions.py:66)
                if (isinstance(sub, ast.Call) and getattr(sub.func, "attr", None) == "step" and sub.args
                        and isinstance(sub.args[0], ast.Attribute) and sub.args[0].attr == "jobs"):
                    wait = "step_noop"            # ta41.. wait with env.step(env.jobs) (e.g. :762)
            out[inst] = {"makespan": makespan, "wait": wait, "solution_sequence": seq}
    return out


def record_trace(JssEnv, inst, policy, seed, max_steps=None):
    env = JssEnv({"instance_path": reference_instance_path(inst)})
    rng = np.random.default_rng(seed)
    obs = env.reset()
    J = env.jobs
    rec = {k: [] for k in ("actions", "mask", "obs", "reward", "done", "t", "nb_legal", "nb_machine_legal",
                           "todo", "tufco", "tuam", "idle_last", "total_idle", "total_perform", "needed",
                           "blocked", "machine_legal")}

    def snap():
        rec["mask"].append(obs["action_mask"].copy())
        rec["obs"].append(obs["real_obs"].copy())
        rec["t"].append(env.current_time_step)
        rec["nb_legal"].append(env.nb_legal_actions)
        rec["nb_machine_legal"].append(env.nb_machine_legal)
        rec["todo"].append(env.todo_time_step_job.copy())
        rec["tufco"].append(env.time_until_finish_current_op_jobs.copy())
        rec["tuam"].append(env.time_until_available_machine.copy())
        rec["idle_last"].append(env.idle_time_jobs_last_op.copy())
        rec["total_idle"].append(env.total_idle_time_jobs.copy())
        rec["total_perform"].append(env.total_perform_op_time_jobs.copy())
        rec["needed"].append(env.needed_machine_jobs.copy())
        rec["blocked"].append(env.action_illegal_no_op.copy())
        rec["machine_legal"].append(env.machine_legal.copy())

    snap()
    done, steps = False, 0
    while not done and (max_steps is None or steps < max_steps):
        mask = obs["action_mask"]
        legal = np.flatnonzero(mask)
        if policy == "random":
            a = int(legal[rng.integers(len(legal))])
        elif policy == "lowest":
            a = int(legal[0])
        elif policy == "highest":
            a = int(legal[-1])
        elif policy == "forcednoop":
            # like the reference's ta41.. replays: every 5th decision waits with
            # step(J) even if the mask says no, whenever an event is pending
            if steps % 5 == 4 and len(env.next_time_step) > 0:
                a = J
            else:
                jl = np.flatnonzero(mask[:J])
                a = int(jl[rng.integers(len(jl))]) if len(jl) else J
        else:
            raise ValueError(policy)
        obs, r, done, _, _ = env.step(a)
        rec["actions"].append(a)
        rec["reward"].append(r)
        rec["done"].append(done)
        snap()
        steps += 1
    arrays = {
        "actions": np.array(rec["actions"], np.int32),
        "mask": np.packbits(np.array(rec["mask"], np.uint8), axis=1),
        "obs": np.array(rec["obs"], np.float64),
        "reward": np.array(rec["reward"], np.float64),
        "done": np.array(rec["done"], np.uint8),
        "t": np.array(rec["t"], np.int32),
        "nb_legal": np.array(rec["nb_legal"], np.int32),
        "nb_machine_legal": np.array(rec["nb_machine_legal"], np.int32),
        "shape": np.array([env.jobs, env.machines], np.int32),
    }
    for k in ("todo", "tufco", "tuam", "idle_last", "total_idle", "total_perform", "needed"):
        arrays[k] = np.array(rec[k], np.int16 if k != "needed" else np.int8)
    for k in ("blocked", "machine_legal"):
        arrays[k] = np.packbits(np.array(rec[k], np.uint8), axis=1)
    return arrays


DELTA_CODED = ("t", "todo", "tufco", "tuam", "idle_last", "total_idle", "total_perform", "needed", "obs_index")


def compact_trace(arrays):
    """Lossless smaller form of a trace, so that a whole ta80 episode stays a small fixture: obs as int16 indices
    into its distinct float64 values, and the slowly changing per-step integer arrays as differences between
    consecutive steps (wrapping in their own dtype, which the running sum in load_trace() undoes exactly)."""
    out = dict(arrays)
    values, index = np.unique(out.pop("obs"), return_inverse=True)
    assert len(values) <= np.iinfo(np.int16).max + 1
    out["obs_values"], out["obs_index"] = values, index.reshape(arrays["obs"].shape).astype(np.int16)
    for k in DELTA_CODED:
        out[k] = np.diff(out[k], axis=0, prepend=np.zeros_like(out[k][:1]))
    out["delta"] = np.array(DELTA_CODED)
    return out


def main():
    os.makedirs(GOLD, exist_ok=True)
    JssEnv, dispatching = load_reference()
    seqs = extract_optimal_sequences()
    assert len(seqs) == 12 and all(v["makespan"] and v["solution_sequence"] for v in seqs.values()), seqs.keys()
    json.dump(seqs, open(os.path.join(GOLD, "optimal_sequences.json"), "w"), separators=(",", ":"))
    print("optimal sequences:", {k: (v["makespan"], v["wait"]) for k, v in seqs.items()})

    plan = [("ta01", "random", 0), ("ta01", "random", 1), ("ta01", "lowest", 0), ("ta01", "highest", 0),
            ("ta01", "forcednoop", 3), ("ta15", "random", 2), ("ta31", "random", 3), ("ta41", "random", 4),
            ("ta41", "lowest", 0), ("ta45", "forcednoop", 5), ("ta62", "random", 6), ("dmu16", "random", 7),
            ("dmu16", "lowest", 0), ("ta80", "random", 8), ("ta80", "lowest", 0, 400), ("ta80", "highest", 0, 400)]
    for inst, policy, seed, *cap in plan:
        arrays = record_trace(JssEnv, inst, policy, seed, cap[0] if cap else None)
        fn = os.path.join(GOLD, f"trace_{inst}_{policy}{seed}.npz")
        np.savez_compressed(fn, **compact_trace(arrays))
        print(f"{fn}: steps={len(arrays['actions'])} makespan={arrays['t'][-1]} "
              f"sum_reward={arrays['reward'].sum()!r} size={os.path.getsize(fn)}")

    # whole-episode known answers for deterministic policies (no per-step data)
    known = {}
    for inst in ("ta01", "ta21", "ta41", "ta51", "ta71", "ta80", "dmu16", "dmu20"):
        for policy in ("lowest", "highest"):
            a = record_trace(JssEnv, inst, policy, 0)
            known[f"{inst}_{policy}"] = {"steps": int(len(a["actions"])), "makespan": int(a["t"][-1]),
                                         "sum_reward": float(a["reward"].sum()),
                                         "action_crc": int(np.bitwise_xor.reduce(
                                             (a["actions"].astype(np.int64) + 1) * (np.arange(len(a["actions"])) + 1)))}
    json.dump(known, open(os.path.join(GOLD, "known_answers.json"), "w"), indent=1)
    print("known answers:", {k: (v["steps"], v["makespan"]) for k, v in known.items()})

    rules = {}
    for inst in ("ta01", "ta41", "ta80", "dmu16"):
        rules[inst] = {}
        for name, rule in dispatching.DISPATCHING_RULES.items():
            env = JssEnv({"instance_path": reference_instance_path(inst)})
            np.random.seed(0)
            total_reward, makespan = rule.run_episode(env)
            rules[inst][name] = {"makespan": int(makespan), "total_reward": float(total_reward)}
        print(inst, {k: v["makespan"] for k, v in rules[inst].items()})
    json.dump(rules, open(os.path.join(GOLD, "rule_makespans.json"), "w"), indent=1)

    # CriticalRatio with non-default due_date_factor (dispatching.py:337-349)
    crf = {}
    for inst in ("ta01", "ta41", "ta80"):
        crf[inst] = {}
        for f in (1.0, 2.25, 4.0):
            env = JssEnv({"instance_path": reference_instance_path(inst)})
            np.random.seed(0)
            total_reward, makespan = dispatching.CriticalRatio(due_date_factor=f).run_episode(env)
            crf[inst][str(f)] = {"makespan": int(makespan), "total_reward": float(total_reward)}
    json.dump(crf, open(os.path.join(GOLD, "cr_factor_makespans.json"), "w"), indent=1)


if __name__ == "__main__":
    main()
