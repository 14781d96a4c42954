"""Generator mode (jss_assign_generated): a fresh random instance per env and episode, drawn on the device.

CPU: the generator contract restated in numpy (and pinned by a golden fixture), its statistics, the exactness of the
observation division for the divisors it produces, and the kernels under host emulation (tests/emu) against the
host generator, the fixed-instance kernels and the CPU oracle.  GPU (-m gpu): the same checks at user sizes, and a
long 65 536-env run of the 100x20 shape."""
import json
import os
import subprocess

import numpy as np
import pytest

from jssenv_b200 import _native as N
from jssenv_b200.instances import generate_instance
from oracle.jss_oracle import OracleEnv
from tests import parity_common as pc
from tests.emu.emu_backend import use_emulation
from tests.helpers import GOLDEN

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
M64 = (1 << 64) - 1


@pytest.fixture(scope="module", autouse=True)
def _library():
    from jssenv_b200.build import build
    build()


@pytest.fixture
def emu():
    with use_emulation():
        yield


def restated(J, M, duration, seed, g, k):
    """include/jss_b200.h, generator mode, restated with the tests' copy of jss_hash3."""
    dmin, dmax = duration
    s = (seed ^ 0x6A09E667F3BCC909) & M64

    def h(j, i, w):
        return pc._hash3(s, g, ((k << 20) | (((j * M + i) << 1) | w)) & M64)

    def pick(x, n):
        return (x * n) >> 32

    machine = np.zeros((J, M), np.int32)
    dur = np.zeros((J, M), np.int32)
    for j in range(J):
        perm = list(range(M))
        for i in range(M):
            dur[j, i] = dmin + pick(h(j, i, 0), dmax - dmin + 1)
        for i in range(M - 1):
            r = i + pick(h(j, i, 1), M - i)
            perm[i], perm[r] = perm[r], perm[i]
        machine[j] = perm
    return machine, dur


# ------------------------------------------------------------------ the contract (CPU)
@pytest.mark.parametrize("J,M,duration,seed", [(15, 15, (1, 99), 0), (3, 2, (1, 1), 7), (100, 20, (1, 99), 123456789),
                                               (128, 32, (1, 2047), 2**63 + 5), (33, 7, (5, 200), 42)])
def test_generate_instance_matches_restated_contract(J, M, duration, seed):
    for g in (0, 1, 5, 2**40 + 3):
        for k in (0, 1, 2, 4095, 4096, 123457, 2**31 - 1):
            m, d = generate_instance(J, M, duration, seed, g, k)
            m2, d2 = restated(J, M, duration, seed, g, k)
            assert np.array_equal(m, m2) and np.array_equal(d, d2), (g, k)
            assert all(sorted(r) == list(range(M)) for r in m.tolist())
            assert d.min() >= duration[0] and d.max() <= duration[1]


def test_env_and_index_pairs_give_different_instances():
    seen = set()
    for g in range(8):
        for k in range(8):
            m, d = generate_instance(10, 10, (1, 99), 3, g, k)
            seen.add(m.tobytes() + d.tobytes())
    assert len(seen) == 64


def test_generated_draws_are_uniform():
    from scipy.stats import chisquare
    J, M, lo, hi = 20, 20, 1, 99
    dur_counts = np.zeros(hi - lo + 1, np.int64)
    pos_counts = np.zeros((M, M), np.int64)            # [position][machine]
    for k in range(250):                               # 250 x 400 = 100 000 draws of each kind
        m, d = generate_instance(J, M, (lo, hi), 2024, k % 5, k)
        dur_counts += np.bincount((d - lo).ravel(), minlength=hi - lo + 1)
        for i in range(M):
            pos_counts[i] += np.bincount(m[:, i], minlength=M)
    assert dur_counts.sum() >= 10**5 and pos_counts.sum() >= 10**5
    assert chisquare(dur_counts).pvalue > 1e-3
    assert chisquare(pos_counts.ravel()).pvalue > 1e-3


def test_golden_generated_instances():
    with open(os.path.join(GOLDEN, "generated_instances.json")) as f:
        gold = json.load(f)
    J, M, dur, seed = gold["jobs"], gold["machines"], tuple(gold["duration"]), gold["seed"]
    assert len(gold["instances"]) == 4
    for rec in gold["instances"]:
        m, d = generate_instance(J, M, dur, seed, rec["env"], rec["index"])
        assert m.tolist() == rec["machine"] and d.tolist() == rec["duration"], (rec["env"], rec["index"])


def test_markstein_division_is_exact_for_generated_divisors(tmp_path):
    """The observation quotients (jss_div) stay IEEE-exact, so real_obs stays inside [0, 1], for the divisors that
    generated instances produce (tools/check_div.c, every numerator 0..y)."""
    exe = tmp_path / "check_div"
    subprocess.check_call(["gcc", "-O1", "-ffp-contract=off", "-o", str(exe), os.path.join(ROOT, "tools", "check_div.c"), "-lm"])
    args, seen = [], set()
    for J, M, dur in ((15, 15, (1, 99)), (20, 20, (1, 99)), (100, 20, (1, 99)), (50, 10, (1, 200)), (128, 32, (1, 2047))):
        for k in range(200):
            m, d = generate_instance(J, M, dur, 11, k % 7, k)
            for y in (int(d.max()), int(d.sum(1).max()), int(d.sum()), M):
                if y not in seen:
                    seen.add(y)
                    args += [str(y), str(y)]
    r = subprocess.run([str(exe)] + args, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "0 mismatches" in r.stdout, r.stdout[-400:]


def test_generator_kernels_compile_as_warp_convergent_code():
    """The generator-mode kernels keep the property the fixed-instance step kernels have (see
    test_step_kernels_compile_as_warp_convergent_code): no collective guarded by BRA.DIV."""
    import collections
    import re
    import shutil
    from jssenv_b200.build import build
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([tool, "-sass", build()], capture_output=True, text=True, check=True).stdout
    div, cur = collections.Counter(), None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            div[cur] += 0
        elif cur and "BRA.DIV" in line:
            div[cur] += 1
    gen = {k: v for k, v in div.items() if k.startswith(("_Z19jss_gen_step_kernel", "_Z18jss_gen_env_kernel"))}
    assert len(gen) == 9 + 9, sorted(gen)
    assert not any(gen.values()), gen


# ------------------------------------------------------------------ checks shared by the emulation and GPU tests
def gen_env(n, J, M, duration=(1, 99), inst_seed=5, **kw):
    from jssenv_b200 import JssVecEnv
    return JssVecEnv(n, {"generator": {"jobs": J, "machines": M, "duration": duration, "seed": inst_seed}}, **kw)


def gen_factory(J, M, duration=(1, 99), inst_seed=5):
    """make_env for the parity_common helpers: the instance config they pass is replaced by the generator."""
    return lambda n, cfg, **kw: gen_env(n, J, M, duration, inst_seed, **kw)


def assert_tables_match_host(env, envs=None):
    t = {k: pc._np(v) for k, v in env.env_instances().items()}
    g = env.generator
    for i in (range(env.num_envs) if envs is None else envs):
        m, d = generate_instance(g["jobs"], g["machines"], g["duration"], g["seed"], env.env_id_base + int(i), int(t["index"][i]))
        assert np.array_equal(t["machine"][i], m) and np.array_equal(t["duration"][i], d), (i, int(t["index"][i]))
    return t


def check_device_tables(n, J, M, n_steps, seed=1):
    env = gen_env(n, J, M, seed=seed, auto_reset=True)
    t = assert_tables_match_host(env)
    assert (t["index"] == 0).all()
    env.reset(np.arange(n) % 2 == 0)                   # explicit masked reset: instance 1 for the even envs
    t = assert_tables_match_host(env)
    assert np.array_equal(t["index"], (np.arange(n) % 2 == 0).astype(np.int32))
    env.reset()
    acts = env.policy("RANDOM")
    for k in range(n_steps):
        *_, acts = env.step_sample(acts, "RANDOM")
    t = assert_tables_match_host(env)
    ep = pc._np(env.episode_count)
    # instance after the explicit resets: 2 (even envs) or 1; then one more per auto-reset, and every finished episode
    # but (possibly) a last one ended in the final transition was followed by an auto-reset
    auto = t["index"] - (1 + (np.arange(n) % 2 == 0))
    assert ((auto == ep) | (auto == ep - 1)).all()
    assert (ep >= 3).all(), ep.min()
    return env


def check_differential_vs_fixed(n, J, M, seed=2, max_steps=100000):
    """Generator handle vs a normal handle loaded with the host-generated instance 0 of every env: bit-identical
    outputs and state on every step until the envs are done."""
    from jssenv_b200 import JssVecEnv
    a = gen_env(n, J, M, inst_seed=seed)
    insts = [generate_instance(J, M, (1, 99), seed, i, 0) for i in range(n)]
    b = JssVecEnv(n, {"instance_paths": insts, "env_to_instance": np.arange(n)})
    for k in range(max_steps):
        acts = a.policy("RANDOM", step_index=k).clone()   # masked-uniform over each env's legal actions
        a.step(acts); b.step(acts)
        for name in ("action_mask", "real_obs", "reward", "reward_raw", "done", "current_time_step", "flags"):
            assert np.array_equal(pc._np(getattr(a, name)), pc._np(getattr(b, name))), (k, name)
        if k % 10 == 0 or pc._np(a.done).all():
            xa, xb = a.export_state(), b.export_state()
            for key in xa:
                assert np.array_equal(pc._np(xa[key]), pc._np(xb[key])), (k, key)
        if pc._np(a.done).all():
            break
    assert pc._np(a.done).all()
    assert a.stats() == b.stats()
    assert np.array_equal(pc._np(a.last_makespan), pc._np(b.last_makespan))


def check_oracle_episodes(n, J, M, n_steps, spot=None, seed=3):
    """Masked-random episodes with auto-reset: the oracle of each spot env is rebuilt from the host-generated instance k
    at every reset; actions, outputs, episode statistics and stats() match."""
    env = gen_env(n, J, M, inst_seed=seed, seed=seed, auto_reset=True)
    spot = list(range(n)) if spot is None else list(spot)
    oracles = {i: OracleEnv(*generate_instance(J, M, (1, 99), seed, i, 0)) for i in spot}
    for o in oracles.values():
        o.reset()
    k_of = {i: 0 for i in spot}
    done = {i: False for i in spot}
    eps = {i: [] for i in spot}
    ret = {i: 0 for i in spot}
    for step in range(n_steps):
        acts = env.policy("RANDOM")
        a_host = pc._np(acts)
        env.step(acts)
        obs = env._obs()
        for i in spot:
            o = oracles[i]
            if done[i]:                                # this transition is the auto-reset: instance k + 1
                k_of[i] += 1
                o = oracles[i] = OracleEnv(*generate_instance(J, M, (1, 99), seed, i, k_of[i]))
                o.reset(); done[i] = False; ret[i] = 0
                pc.compare_env_to_oracle(env, i, o, obs, ctx=f"auto-reset step {step}")
                continue
            assert a_host[i] == o.masked_random_action(seed, i, step), (step, i)
            _, r, done[i], _, _ = o.step(int(a_host[i]))
            ret[i] += o.last_raw_reward
            pc.compare_env_to_oracle(env, i, o, obs, ctx=f"step {step}")
            if done[i]:
                eps[i].append((o.current_time_step, ret[i]))
                assert ret[i] == 2 * o.sum_op - M * o.current_time_step
    ec, lm, lr = pc._np(env.episode_count), pc._np(env.last_makespan), pc._np(env.last_return)
    for i in spot:
        assert len(eps[i]) >= 2, (i, len(eps[i]))
        assert ec[i] == len(eps[i]) and lm[i] == eps[i][-1][0] and lr[i] == eps[i][-1][1], i
    if len(spot) == n:
        st = env.stats()
        mk = [m for i in spot for m, _ in eps[i]]
        assert st["episodes"] == len(mk) and st["sum_makespan"] == sum(mk)
        assert st["min_makespan"] == min(mk) and st["max_makespan"] == max(mk)
        assert st["sum_return"] == sum(r for i in spot for _, r in eps[i]) and st["envs_error"] == 0
    return env


def check_shard_invariance(J, M, n_total, n_steps, seed=77):
    cuts = [0, n_total // 3, n_total]
    whole = gen_env(n_total, J, M, inst_seed=seed, seed=seed, auto_reset=True)
    shards = [gen_env(hi - lo, J, M, inst_seed=seed, seed=seed, auto_reset=True, env_id_base=lo)
              for lo, hi in zip(cuts[:-1], cuts[1:])]
    aw = whole.policy("RANDOM")
    a_s = [s.policy("RANDOM") for s in shards]
    for k in range(n_steps):
        *_, aw = whole.step_sample(aw, "RANDOM")
        for j, s in enumerate(shards):
            *_, a_s[j] = s.step_sample(a_s[j], "RANDOM")
    tw = {key: pc._np(v) for key, v in whole.env_instances().items()}
    for s, lo, hi in zip(shards, cuts[:-1], cuts[1:]):
        for name in ("action_mask", "real_obs", "reward", "reward_raw", "done", "current_time_step", "episode_count",
                     "last_makespan", "last_return"):
            assert np.array_equal(pc._np(getattr(s, name)), pc._np(getattr(whole, name))[lo:hi]), name
        ts = s.env_instances()
        for key in tw:
            assert np.array_equal(pc._np(ts[key]), tw[key][lo:hi]), key
    assert int(pc._np(whole.episode_count).min()) >= 1


# ------------------------------------------------------------------ emulation (CPU)
@pytest.mark.parametrize("J,M", [(6, 4), (40, 3), (70, 2)])   # lane classes KJ = 1, 2, 4
def test_emu_generated_device_tables(emu, J, M):
    check_device_tables(5, J, M, n_steps=4 * J * M + 20)


@pytest.mark.parametrize("J,M", [(7, 5), (36, 3)])
def test_emu_generated_differential_vs_fixed_instances(emu, J, M):
    check_differential_vs_fixed(6, J, M)


def test_emu_generated_oracle_episodes(emu):
    check_oracle_episodes(4, 6, 5, n_steps=120)


def test_emu_generated_fused_paths(emu):
    make = gen_factory(8, 4)
    for rule in ("RANDOM", "MWR", "CR"):
        pc.check_step_sample(make, ["g"] * 5, rule, n_steps=90, seed=12)
    pc.check_rollout_record(make, ["g"] * 5, "RANDOM", n_steps=90, seed=3)
    pc.check_rollout_record(make, ["g"] * 5, "CR", n_steps=90, seed=4)


def test_emu_generated_shard_invariance(emu):
    check_shard_invariance(6, 4, n_total=10, n_steps=80)


def check_error_codes():
    from jssenv_b200 import JssVecEnv
    from jssenv_b200._native import NativeError
    for J, M, dur, msg in ((129, 4, (1, 99), r"rc=-4"), (8, 33, (1, 99), r"rc=-4"), (8, 4, (1, 2048), r"rc=-4"),
                           (8, 4, (0, 9), r"rc=-4"), (8, 4, (9, 3), r"rc=-1"), (8, 1, (1, 9), r"rc=-1")):
        with pytest.raises(NativeError, match=msg):
            gen_env(2, J, M, dur)
        with pytest.raises(NativeError):
            generate_instance(J, M, dur, 0, 0, 0)
    with pytest.raises(NativeError, match="rc=-4"):
        gen_env(2, 8, 4, host_mirror=True)
    env = gen_env(3, 8, 4)
    snap = {k: v.clone() for k, v in env.export_state().items()}
    with pytest.raises(NativeError, match="rc=-4.*generator mode"):
        env.import_state(snap)
    with pytest.raises(NativeError, match="rc=-4"):
        env.host_step_begin(np.zeros(3, np.int32), packed=True)
    with pytest.raises(NativeError, match="rc=-4"):
        env.host_step_begin(np.zeros(3, np.int32), packed=True, dma_fraction=0.5)
    fixed = JssVecEnv(2, {"instance_path": "ta01"})
    assert fixed._L.jss_assign_generated(fixed._h, 8, 4, 1, 99, 0) == -5          # JSS_ERR_STATE
    # the plain host-buffer step works in generator mode
    ref = gen_env(3, 8, 4)
    acts = np.zeros(3, np.int32)
    obs, rew, done, _, _ = env.step_host(acts)
    ref.step(acts)
    assert np.array_equal(obs["real_obs"], pc._np(ref.real_obs)) and np.array_equal(obs["action_mask"], pc._np(ref.action_mask))


def test_emu_generated_error_codes(emu):
    check_error_codes()


# ------------------------------------------------------------------ GPU
gpu = pytest.mark.gpu


def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


@gpu
@pytest.mark.parametrize("n,J,M", [(4096, 20, 20), (1024, 100, 20)])
def test_gpu_generated_device_tables(n, J, M):
    _cuda()
    check_device_tables(n, J, M, n_steps=8 * J * M)


@gpu
@pytest.mark.parametrize("n,J,M", [(4096, 20, 20), (1024, 100, 20)])
def test_gpu_generated_differential_vs_fixed_instances(n, J, M):
    _cuda()
    check_differential_vs_fixed(n, J, M)


@gpu
@pytest.mark.parametrize("n,J,M", [(4096, 20, 20), (1024, 100, 20)])
def test_gpu_generated_oracle_episodes(n, J, M):
    _cuda()
    # about two masked-random episodes per env and a bit (~450 transitions for 20x20, ~2 240 for 100x20)
    check_oracle_episodes(n, J, M, n_steps=1200 if J == 20 else 5200, spot=range(0, n, n // 64))


@gpu
@pytest.mark.parametrize("n,J,M", [(4096, 20, 20), (1024, 100, 20)])
def test_gpu_generated_fused_paths(n, J, M):
    _cuda()
    make = gen_factory(J, M)
    for rule in N.RULES:
        pc.check_step_sample(make, ["g"] * n, rule, n_steps=600, seed=12)
    pc.check_rollout_record(make, ["g"] * n, "RANDOM", n_steps=300, seed=3)


@gpu
@pytest.mark.parametrize("n,J,M", [(4096, 20, 20), (1024, 100, 20)])
def test_gpu_generated_shard_invariance(n, J, M):
    _cuda()
    check_shard_invariance(J, M, n_total=n, n_steps=3 * J * M)


@gpu
def test_gpu_generated_error_codes():
    _cuda()
    check_error_codes()


@gpu
def test_gpu_generated_long_run_100x20():
    """65 536 envs of the 100x20 shape, RANDOM step_sample for 2 600 steps (about two episodes each)."""
    _cuda()
    import torch
    n, J, M = 65536, 100, 20
    env = gen_env(n, J, M, inst_seed=9, seed=9, auto_reset=True)
    acts = env.policy("RANDOM")
    checked = 0
    for k in range(2600):
        *_, acts = env.step_sample(acts, "RANDOM")
        ro = env.real_obs
        assert bool(torch.isfinite(ro).all()) and float(ro.min()) >= 0.0 and float(ro.max()) <= 1.0, k
        done = env.done
        assert torch.equal(~env.action_mask[:, :J].any(1), done), k
        if bool(done.any()):
            idx = torch.nonzero(done).squeeze(1)
            sum_op = env.env_instances()["duration"][idx].sum((1, 2))
            assert torch.equal(env.last_return[idx], 2 * sum_op - M * env.last_makespan[idx]), k
            checked += int(idx.numel())
    assert checked >= n // 2
    assert_tables_match_host(env, envs=np.random.default_rng(0).choice(n, 256, replace=False))
    st = env.stats()
    assert st["envs_error"] == 0 and st["episodes"] == int(env.episode_count.sum())
