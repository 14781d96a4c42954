"""Shared helpers for the parity tests (oracle side)."""
import glob
import json
import os

import numpy as np

from jssenv_b200.instances import load_instance
from oracle.jss_oracle import OracleEnv

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def oracle_env(name):
    m, d = load_instance(name)
    return OracleEnv(m, d)


def golden_traces():
    return sorted(glob.glob(os.path.join(GOLDEN, "trace_*.npz")))


def load_trace(path):
    z = np.load(path)
    J, M = [int(x) for x in z["shape"]]
    tr = {k: z[k] for k in z.files}
    if "obs_index" in tr:                       # compact form (oracle/gen_golden.py compact_trace)
        for k in tr.pop("delta"):
            tr[k] = np.cumsum(tr[k], axis=0, dtype=tr[k].dtype)
        tr["obs"] = tr.pop("obs_values")[tr.pop("obs_index")]
    tr["mask"] = np.unpackbits(z["mask"], axis=1)[:, : J + 1].astype(bool)
    tr["blocked"] = np.unpackbits(z["blocked"], axis=1)[:, :J].astype(bool)
    tr["machine_legal"] = np.unpackbits(z["machine_legal"], axis=1)[:, :M].astype(bool)
    tr["inst"] = os.path.basename(path).split("_")[1]
    return tr


def load_json(name):
    with open(os.path.join(GOLDEN, name)) as f:
        return json.load(f)


def replay_optimal(env, spec, step_fn=None, wait_fn=None):
    """The replay loop of the reference's tests/test_solutions.py (e.g. :36-73):
    walk the machines, play the next job of a machine's optimal order when it is
    legal, otherwise wait (raw increase_time_step for ta01, step(J) for the rest).
    `env` needs machine_legal, needed_machine_jobs, legal_actions, step, jobs."""
    seq = spec["solution_sequence"]
    job_nb, machine_nb = len(seq[0]), len(seq)
    index_machine = [0] * machine_nb
    done = False
    env.reset()
    assert env.current_time_step == 0
    while not done:
        no_op = True
        for machine in range(machine_nb):
            if done:
                break
            if env.machine_legal[machine] and index_machine[machine] < job_nb:
                a = seq[machine][index_machine[machine]]
                if env.needed_machine_jobs[a] == machine and env.legal_actions[a]:
                    no_op = False
                    assert int(np.sum(env.legal_actions[:-1])) == env.nb_legal_actions
                    _, _, done, _, _ = env.step(a)
                    index_machine[machine] += 1
        if no_op and not done:
            assert len(env.next_time_step) > 0
            prev = env.current_time_step
            if spec["wait"] == "increase_time_step":
                env.increase_time_step()
            else:
                _, _, done, _, _ = env.step(env.jobs)
            assert env.current_time_step > prev
    assert sum(index_machine) == job_nb * machine_nb
    return env.current_time_step
