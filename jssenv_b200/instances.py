"""Instance ingestion (host side).

Mirrors the reference's parser (JSSEnv/envs/jss_env.py:72-95): a Taillard-format
text file has ``J M`` on line 1, then J lines of M ``machine duration`` pairs.
The bundled public benchmark set (ta01..ta80, dmu16..dmu20 -- the same 85
instances the reference ships under JSSEnv/envs/instances/) is stored in one
binary bundle, ``data/instances.npz`` (see tools/pack_instances.py).
"""
import os
from typing import Tuple, Union

import numpy as np

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "instances.npz")
_bundle = None

DEFAULT_INSTANCE = "ta80"  # the reference's default (jss_env.py:35-38)


def bundled_names():
    return sorted(_load_bundle().keys())


def _load_bundle():
    global _bundle
    if _bundle is None:
        with np.load(_DATA) as z:
            _bundle = {k: z[k].astype(np.int32) for k in z.files}
    return _bundle


def parse_taillard(path: Union[str, os.PathLike]) -> Tuple[np.ndarray, np.ndarray]:
    """Parse a Taillard-format file -> (machine[J, M], duration[J, M]) int32.

    Same acceptance rules as the reference: every job line must hold exactly M
    pairs (assert at jss_env.py:81); at least 2 machines (jss_env.py:94).
    """
    with open(path, "r") as f:
        lines = [ln.split() for ln in f]
    lines = [ln for ln in lines if ln]
    if not lines or len(lines[0]) != 2:
        raise ValueError(f"{path}: first line must be 'J M'")
    J, M = int(lines[0][0]), int(lines[0][1])
    if len(lines) - 1 != J:
        raise ValueError(f"{path}: expected {J} job lines, found {len(lines) - 1}")
    machine = np.zeros((J, M), dtype=np.int32)
    duration = np.zeros((J, M), dtype=np.int32)
    for j in range(J):
        row = list(map(int, lines[1 + j]))
        if len(row) % 2 != 0 or len(row) // 2 != M:
            raise ValueError(f"{path}: job {j} has {len(row)} numbers, expected {2 * M}")
        machine[j] = row[0::2]
        duration[j] = row[1::2]
    validate_instance(machine, duration)
    return machine, duration


def validate_instance(machine: np.ndarray, duration: np.ndarray) -> None:
    J, M = machine.shape
    if J <= 0:
        raise ValueError("need at least one job")
    if M <= 1:
        raise ValueError("We need at least 2 machines")  # jss_env.py:94
    if machine.min() < 0 or machine.max() >= M:
        raise ValueError("machine index out of range")
    if duration.max() <= 0:
        raise ValueError("max_time_op must be > 0")  # jss_env.py:91


def load_instance(spec: Union[str, os.PathLike, Tuple[np.ndarray, np.ndarray]]):
    """`spec` is a bundled name ('ta80'), a path to a Taillard-format file, or an
    already-parsed (machine, duration) pair."""
    if isinstance(spec, tuple):
        machine = np.ascontiguousarray(spec[0], dtype=np.int32)
        duration = np.ascontiguousarray(spec[1], dtype=np.int32)
        validate_instance(machine, duration)
        return machine, duration
    s = os.fspath(spec)
    if os.path.isfile(s):
        return parse_taillard(s)
    b = _load_bundle()
    key = os.path.basename(s)
    if key in b:
        arr = b[key]
        return np.ascontiguousarray(arr[:, :, 0]), np.ascontiguousarray(arr[:, :, 1])
    raise FileNotFoundError(f"instance '{spec}' is neither a file nor a bundled instance name")


def write_taillard(spec, path) -> str:
    """Emit an instance in the standard text format (for tools that want a file)."""
    machine, duration = load_instance(spec)
    J, M = machine.shape
    with open(path, "w") as f:
        f.write(f"{J} {M}\n")
        for j in range(J):
            f.write(" ".join(f"{int(machine[j, i])} {int(duration[j, i])}" for i in range(M)) + "\n")
    return os.fspath(path)


def generate_instance(jobs: int, machines: int, duration: Tuple[int, int], seed: int, env_id: int,
                      index: int) -> Tuple[np.ndarray, np.ndarray]:
    """Instance `index` of global env `env_id` in generator mode (``{"generator": ...}`` env configs), computed on the
    host by the library's own generator (jss_generate_instance) -> (machine[J, M], duration[J, M]) int32."""
    import ctypes
    from . import _native
    machine = np.empty((jobs, machines), np.int32)
    dur = np.empty((jobs, machines), np.int32)
    rc = _native.backend.library().jss_generate_instance(int(jobs), int(machines), int(duration[0]), int(duration[1]),
                                                         int(seed), int(env_id), int(index),
                                                         ctypes.c_void_p(machine.ctypes.data), ctypes.c_void_p(dur.ctypes.data))
    if rc != 0:
        msg = _native.backend.library().jss_last_error(None)
        raise _native.NativeError(f"jss_generate_instance failed (rc={rc}): {msg.decode() if msg else ''}")
    return machine, dur
