"""CPU-only checks of the boundary: the built CUDA library loads and exports every
symbol include/jss_b200.h declares (no compute calls without a GPU), instance
ingestion, and the host-side sharding / statistics logic incl. a world_size-2 gloo run."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_header_symbols_exported_by_cuda_library():
    from jssenv_b200 import _native
    from jssenv_b200.build import build
    path = build()
    hdr = open(os.path.join(ROOT, "include", "jss_b200.h")).read()
    declared = set(re.findall(r"\b(jss_[a-z_]+)\s*\(", hdr))
    assert declared == set(_native.EXPORTED_SYMBOLS), declared ^ set(_native.EXPORTED_SYMBOLS)
    lib = ctypes.CDLL(path)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert lib.jss_abi_version() == _native.JSS_ABI_VERSION


_NO_DEVICE_WORKER = r"""
import sys
sys.path.insert(0, {root!r})
from jssenv_b200 import JssVecEnv
from jssenv_b200._native import NativeError
try:
    JssVecEnv(2, {{"instance_path": "ta01"}})
except NativeError as e:
    print("NativeError:", e)
"""


def test_no_cpu_fallback_without_gpu():
    """On a box without a CUDA device, constructing an env must fail loudly.  The devices are hidden from a fresh
    interpreter, so that this also holds where a GPU is present."""
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_WORKER.format(root=ROOT)], capture_output=True, text=True,
                       timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stdout + r.stderr
    assert re.search(r"^NativeError:.*(no CUDA device|no CPU fallback)", r.stdout, re.M), r.stdout + r.stderr


def test_buffers_struct_matches_header():
    from jssenv_b200 import _native
    hdr = open(os.path.join(ROOT, "include", "jss_b200.h")).read()
    body = hdr[hdr.index("typedef struct jss_buffers {"):hdr.index("} jss_buffers;")]
    fields = re.findall(r"\b(?:int32_t|uint8_t|uint32_t|float)\s*\*?\s*([a-z_0-9]+);", body)
    assert fields == [f[0] for f in _native.JssBuffers._fields_]


def test_instances_bundle_and_parser(tmp_path):
    from jssenv_b200.instances import bundled_names, load_instance, parse_taillard, write_taillard
    names = bundled_names()
    assert len(names) == 85 and "ta80" in names and "dmu16" in names
    m, d = load_instance("ta01")
    assert m.shape == (15, 15) and d.max() == 99 and d.sum() == 11671        # SURVEY section 8 sizes
    assert all(sorted(r) == list(range(15)) for r in m.tolist())
    p = write_taillard("ta01", tmp_path / "ta01.txt")
    m2, d2 = parse_taillard(p)
    assert np.array_equal(m, m2) and np.array_equal(d, d2)
    m3, d3 = load_instance(str(p))
    assert np.array_equal(m, m3)
    (tmp_path / "bad").write_text("2 1\n0 5\n0 6\n")
    with pytest.raises(ValueError, match="at least 2 machines"):            # jss_env.py:94
        parse_taillard(tmp_path / "bad")
    with pytest.raises(FileNotFoundError):
        load_instance("no_such_instance")


def test_shard_ranges_and_stats_combine():
    from jssenv_b200.distributed import combine_stats, shard_range
    for total, world in [(262144, 8), (65536, 4), (10, 3), (7, 8)]:
        spans = [shard_range(total, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == total
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1
    big = np.iinfo(np.int64).max
    c = combine_stats([[2, 100, 3000, 1400, 1600, -5, 1, 0], [0, 50, 0, big, 0, 0, 0, 1]])
    assert c == {"episodes": 2, "steps": 150, "sum_makespan": 3000, "min_makespan": 1400, "max_makespan": 1600,
                 "sum_return": -5, "envs_done": 1, "envs_error": 1}
    assert combine_stats([[0, 0, 0, big, 0, 0, 0, 0]])["min_makespan"] == -1


_GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import torch.distributed as dist
from jssenv_b200.distributed import all_gather_stats, shard_range
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
lo, hi = shard_range(1001, rank, world)
local = dict(episodes=hi - lo, steps=10 * (rank + 1), sum_makespan=1000 * (hi - lo), min_makespan=900 + rank,
             max_makespan=1100 + rank, sum_return=-rank, envs_done=rank, envs_error=0)
out = all_gather_stats(local)
assert out["episodes"] == 1001 and out["steps"] == 30 and out["min_makespan"] == 900 and out["max_makespan"] == 1101, out
assert out["sum_makespan"] == 1001000 and out["sum_return"] == -1 and out["envs_done"] == 1
dist.barrier(); dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_stats_all_gather_world_size_2_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_GLOO_WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29731", str(script)],
                       capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("ok") == 2


def test_markstein_division_is_exact_for_all_bundled_divisors(tmp_path):
    """jss_div() (3 instructions) == IEEE fp32 division for every numerator/divisor pair the bundled instances
    can produce (tools/check_div.c, exhaustive per divisor)."""
    from jssenv_b200.instances import bundled_names, load_instance
    exe = tmp_path / "check_div"
    subprocess.check_call(["gcc", "-O1", "-ffp-contract=off", "-o", str(exe), os.path.join(ROOT, "tools", "check_div.c"), "-lm"])
    args, seen = [], set()
    for n in bundled_names():
        m, d = load_instance(n)
        for y in (int(d.max()), int(d.sum(1).max()), int(d.sum()), m.shape[1]):
            if y not in seen:
                seen.add(y)
                args += [str(y), str(y)]
    for y in range(1, 257):
        args += [str(y), str(y)]
    r = subprocess.run([str(exe)] + args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "0 mismatches" in r.stdout, r.stdout[-400:]


def test_host_pool_regions_complete_after_reconfigure(tmp_path):
    """The host worker pool finishes every chunk of a parallel region before returning, also right after
    jss_host_configure() restarted its workers, as bench.py's e2e calibration does (tools/check_pool.cpp)."""
    exe = tmp_path / "check_pool"
    csrc = os.path.join(ROOT, "jssenv_b200", "csrc")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", csrc, "-o", str(exe), os.path.join(ROOT, "tools", "check_pool.cpp"),
                           os.path.join(csrc, "jss_host.cpp"), "-lpthread"])
    r = subprocess.run([str(exe), "2000"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and " 0 early returns" in r.stdout, r.stdout + r.stderr


def test_step_kernels_compile_as_warp_convergent_code():
    """SASS property of the built library: with the warp-uniformity hints (jss_uniform in csrc/jss_device.cuh) ptxas proves
    the step / rollout / policy kernels warp-convergent, i.e. no collective is guarded by BRA.DIV + a WARPSYNC stub.  The
    property is fragile (one branch on a value ptxas cannot classify brings all of them back), so it is pinned here.
    The uniform 4-jobs-per-lane step kernel is excluded on purpose (measured slower with the hint, see jss_hint_flags)."""
    import collections
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
    hot = {k: v for k, v in div.items()
           if k.startswith("_Z15jss_step_kernel") or k.startswith("_Z21jss_step_mixed_kernel") or k.startswith("_Z14jss_env_kernel")}
    assert len(hot) == 12 + 6 + 12, sorted(hot)
    excluded = {k for k in hot if k.startswith("_Z15jss_step_kernelILi4E")}
    assert len(excluded) == 3
    bad = {k: v for k, v in hot.items() if v and k not in excluded}
    assert not bad, bad
    assert all(hot[k] > 0 for k in excluded), "update jss_hint_flags / this test together"
