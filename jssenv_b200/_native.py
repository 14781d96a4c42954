"""ctypes binding of the C-ABI in include/jss_b200.h (the only native entry point).

The CUDA library ``libjss_b200.so`` is built in-tree by ``__graft_entry__.build()``
(nvcc, sm_100a).  There is no CPU implementation: if the library is missing, or no
B200-class device is present, construction fails loudly.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_uint8, c_uint32, c_uint64, c_void_p

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("JSS_B200_LIB") or os.path.join(_PKG_DIR, "libjss_b200.so")   # override: kernel-variant experiments only

JSS_ABI_VERSION = 3
ACTION_SKIP, ACTION_ADVANCE = -1, -2
CREATE_AUTO_RESET, CREATE_RECORD_SOLUTION, CREATE_HOST_MIRROR = 1, 2, 4
FLAG_DONE, FLAG_ERROR, FLAG_NOOP_LEGAL = 1, 2, 4
COIN_DEVICE, COIN_NEVER = 0, 1
WAIT_MASK, WAIT_OBS, WAIT_OBS_PREV = 1, 2, 3
RULES = {"RANDOM": 0, "SPT": 1, "FIFO": 2, "MWR": 3, "LWR": 4, "MOR": 5, "LOR": 6, "CR": 7}
STATS_KEYS = ("episodes", "steps", "sum_makespan", "min_makespan", "max_makespan", "sum_return",
              "envs_done", "envs_error")

EXPORTED_SYMBOLS = (
    "jss_abi_version", "jss_create", "jss_destroy", "jss_last_error", "jss_load_instances", "jss_assign",
    "jss_get_buffers", "jss_instance_scalars", "jss_reset", "jss_step", "jss_policy", "jss_rollout",
    "jss_step_host", "jss_host_step_begin", "jss_host_wait", "jss_step_sample", "jss_stats", "jss_export_state", "jss_import_state", "jss_host_masked_random",
    "jss_launch_count", "jss_set_cr_due_date_factor", "jss_host_step_begin_packed", "jss_host_wire_stride",
    "jss_host_expand_obs", "jss_host_configure", "jss_host_threads", "jss_host_set_simd", "jss_rollout_traj", "jss_step_export", "jss_host_step_begin_hybrid", "jss_host_expand_obs_range",
    "jss_assign_generated", "jss_get_env_instances", "jss_generate_instance",
)


class JssBuffers(ctypes.Structure):
    _fields_ = [
        ("n_envs", c_int32), ("jobs_max", c_int32), ("machines_max", c_int32), ("mask_stride", c_int32),
        ("action_mask", c_void_p), ("real_obs", c_void_p), ("scalar_stride", c_int32), ("host_mirror", c_int32),
        ("reward", c_void_p), ("reward_raw", c_void_p),
        ("done", c_void_p), ("time", c_void_p), ("flags_done", c_void_p), ("solution", c_void_p),
        ("episode_count", c_void_p), ("last_makespan", c_void_p), ("last_return", c_void_p),
        ("x_todo", c_void_p), ("x_tufco", c_void_p), ("x_idle_last", c_void_p), ("x_total_idle", c_void_p),
        ("x_col4", c_void_p), ("x_tuam", c_void_p), ("x_legal", c_void_p), ("x_blocked", c_void_p),
        ("mirror_actions", c_void_p),
    ]


class NativeError(RuntimeError):
    pass


def _declare(L):
    L.jss_abi_version.restype = c_int
    L.jss_create.argtypes = [POINTER(c_void_p), c_int, c_int, c_uint32, c_uint64]
    L.jss_destroy.argtypes = [c_void_p]
    L.jss_destroy.restype = None
    L.jss_last_error.argtypes = [c_void_p]
    L.jss_last_error.restype = c_char_p
    L.jss_load_instances.argtypes = [c_void_p, c_int, POINTER(c_int32), POINTER(c_int32), POINTER(c_int64),
                                     POINTER(c_int32), POINTER(c_int32)]
    L.jss_assign.argtypes = [c_void_p, POINTER(c_int32)]
    L.jss_get_buffers.argtypes = [c_void_p, POINTER(JssBuffers)]
    L.jss_instance_scalars.argtypes = [c_void_p, c_int, POINTER(c_int64)]
    L.jss_reset.argtypes = [c_void_p, c_void_p, c_void_p]
    L.jss_step.argtypes = [c_void_p, c_void_p, c_void_p]
    L.jss_policy.argtypes = [c_void_p, c_int, c_int, c_uint64, c_uint64, c_void_p, c_void_p]
    L.jss_step_sample.argtypes = [c_void_p, c_void_p, c_int, c_int, c_uint64, c_uint64, c_void_p, c_void_p]
    L.jss_rollout.argtypes = [c_void_p, c_int, c_uint64, c_uint64, c_int, c_int, c_void_p]
    L.jss_step_host.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.jss_host_step_begin.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.jss_host_wait.argtypes = [c_void_p, c_int]
    L.jss_host_step_begin_packed.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.jss_host_step_begin_packed.restype = c_int
    L.jss_host_step_begin_hybrid.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p]
    L.jss_host_step_begin_hybrid.restype = c_int
    L.jss_host_expand_obs_range.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int]
    L.jss_host_expand_obs_range.restype = c_int
    L.jss_host_wire_stride.argtypes = [c_void_p]
    L.jss_host_wire_stride.restype = c_int64
    L.jss_host_expand_obs.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p]
    L.jss_host_expand_obs.restype = c_int
    L.jss_host_configure.argtypes = [c_int, c_int]
    L.jss_host_configure.restype = c_int
    L.jss_rollout_traj.argtypes = [c_void_p, c_int, c_uint64, c_uint64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.jss_rollout_traj.restype = c_int
    L.jss_step_export.argtypes = [c_void_p, c_void_p, c_void_p]
    L.jss_step_export.restype = c_int
    L.jss_host_set_simd.argtypes = [c_int]
    L.jss_host_set_simd.restype = c_int
    L.jss_host_threads.argtypes = []
    L.jss_host_threads.restype = c_int
    L.jss_stats.argtypes = [c_void_p, POINTER(c_int64), c_void_p]
    L.jss_export_state.argtypes = [c_void_p, c_void_p]
    L.jss_import_state.argtypes = [c_void_p, c_void_p, c_void_p]
    L.jss_host_masked_random.argtypes = [c_void_p, c_int, c_int, c_int64, c_uint64, c_uint64, c_uint64, c_void_p]
    L.jss_set_cr_due_date_factor.argtypes = [c_void_p, ctypes.c_double]
    L.jss_set_cr_due_date_factor.restype = c_int
    L.jss_launch_count.argtypes = [c_void_p]
    L.jss_launch_count.restype = c_int64
    L.jss_assign_generated.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_uint64]
    L.jss_get_env_instances.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    L.jss_generate_instance.argtypes = [c_int, c_int, c_int, c_int, c_uint64, c_uint64, c_uint64, c_void_p, c_void_p]
    for name in ("jss_create", "jss_load_instances", "jss_assign", "jss_get_buffers", "jss_instance_scalars",
                 "jss_reset", "jss_step", "jss_policy", "jss_rollout", "jss_step_host", "jss_host_step_begin", "jss_host_wait", "jss_step_sample", "jss_stats",
                 "jss_export_state", "jss_import_state", "jss_host_masked_random", "jss_assign_generated",
                 "jss_get_env_instances", "jss_generate_instance"):
        getattr(L, name).restype = c_int
    return L


class CudaBackend:
    """Device memory / stream plumbing through torch (plumbing only: every kernel is ours)."""

    name = "cuda"

    def __init__(self):
        self._lib = None

    def library(self):
        if self._lib is None:
            if not os.path.exists(LIB_PATH):
                raise NativeError(
                    f"{LIB_PATH} is missing: build the CUDA extension first "
                    "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
            L = _declare(ctypes.CDLL(LIB_PATH))
            if L.jss_abi_version() != JSS_ABI_VERSION:
                raise NativeError("libjss_b200.so ABI version mismatch; rebuild")
            self._lib = L
        return self._lib

    def torch_device(self, index):
        import torch
        return torch.device("cuda", index)

    def stream(self, device_index):
        import torch
        return c_void_p(torch.cuda.current_stream(device_index).cuda_stream)

    def wrap(self, ptr, shape, dtype, device_index, strides=None):
        """Zero-copy torch view of library-owned device memory."""
        import torch

        class _Holder:
            pass

        h = _Holder()
        npdt = np.dtype(dtype)
        h.__cuda_array_interface__ = {
            "shape": tuple(int(s) for s in shape), "typestr": npdt.str, "data": (int(ptr), False), "version": 3,
            "strides": None if strides is None else tuple(int(s) for s in strides),
        }
        return torch.as_tensor(h, device=torch.device("cuda", device_index))

    def synchronize(self, device_index):
        import torch
        torch.cuda.synchronize(device_index)


backend = CudaBackend()   # tests/emu swaps this object; product code never does


def check(handle, rc, what):
    if rc != 0:
        msg = backend.library().jss_last_error(handle)
        raise NativeError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


def as_i32p(a):
    return a.ctypes.data_as(POINTER(c_int32))
