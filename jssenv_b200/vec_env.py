"""JssVecEnv -- N independent job-shop environments stepped by the sm_100a kernels.

Batched form of the reference's ``JssEnv`` contract (JSSEnv/envs/jss_env.py):
``reset() -> obs`` (jss_env.py:145), ``step(actions) -> (obs, reward, done,
truncated, info)`` (jss_env.py:403-481) with ``obs = {"real_obs": (N, J, 7) float32,
"action_mask": (N, J+1) bool}`` (jss_env.py:112-119, 130-134).  As in the reference,
the observation entries are LIVE ALIASES of the environment's buffers (here: device
memory owned by the native library), the no-op is action index ``J``, actions are
not validated beyond setting a per-env error bit, and ``truncated`` is always False.
"""
import ctypes
from typing import Any, Dict, Optional, Union

import numpy as np

from . import _native as N
from .instances import DEFAULT_INSTANCE, load_instance


def _instance_list(env_config: Optional[Dict[str, Any]]):
    """`env_config` keeps the reference key ``instance_path`` (jss_env.py:35-39) and adds
    ``instance_paths`` (list) + ``env_to_instance`` (int array) for mixed batches."""
    if env_config is None:
        env_config = {"instance_path": DEFAULT_INSTANCE}
    if "instance_paths" in env_config:
        specs = list(env_config["instance_paths"])
    else:
        specs = [env_config["instance_path"]]
    return [load_instance(s) for s in specs], env_config.get("env_to_instance")


class JssVecEnv:
    def __init__(self, num_envs: int, env_config: Optional[Dict[str, Any]] = None, device: int = 0,
                 auto_reset: bool = False, record_solution: bool = False, env_id_base: int = 0, seed: int = 0,
                 host_mirror: bool = False):
        self._h = ctypes.c_void_p()
        self._L = N.backend.library()
        self.num_envs = int(num_envs)
        self.device_index = int(device)
        self.seed = int(seed)
        self.env_id_base = int(env_id_base)
        self.auto_reset = bool(auto_reset)
        self._step_index = 0
        flags = ((N.CREATE_AUTO_RESET if auto_reset else 0) | (N.CREATE_RECORD_SOLUTION if record_solution else 0) |
                 (N.CREATE_HOST_MIRROR if host_mirror else 0))
        rc = self._L.jss_create(ctypes.byref(self._h), self.device_index, self.num_envs, flags, self.env_id_base)
        N.check(None, rc, "jss_create")
        self.generator = None
        if env_config is not None and "generator" in env_config:
            self._assign_generated(env_config["generator"])
        else:
            self._assign_instances(env_config)
        self._bind_buffers()

    def _assign_generated(self, gen: Dict[str, Any]):
        """Generator mode: a fresh random J x M instance per env and episode, drawn on the device (jss_assign_generated)."""
        J, M = int(gen["jobs"]), int(gen["machines"])
        dmin, dmax = (int(v) for v in gen.get("duration", (1, 99)))
        seed = int(gen.get("seed", self.seed))
        self.generator = {"jobs": J, "machines": M, "duration": (dmin, dmax), "seed": seed}
        rc = self._L.jss_assign_generated(self._h, J, M, dmin, dmax, seed)   # also draws instance 0 and resets
        N.check(self._h, rc, "jss_assign_generated")
        self.instances = None
        self.instance_scalars = None
        self.env_to_instance = None
        self.env_jobs = np.full(self.num_envs, J, np.int32)
        self.env_machines = np.full(self.num_envs, M, np.int32)

    def _assign_instances(self, env_config):
        insts, env_to_inst = _instance_list(env_config)
        self.instances = insts
        # instance tables (jss_env.py:72-95)
        jobs = np.array([m.shape[0] for m, _ in insts], np.int32)
        machines = np.array([m.shape[1] for m, _ in insts], np.int32)
        sizes = jobs.astype(np.int64) * machines
        offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
        mach = np.concatenate([m.reshape(-1) for m, _ in insts]).astype(np.int32)
        dur = np.concatenate([d.reshape(-1) for _, d in insts]).astype(np.int32)
        rc = self._L.jss_load_instances(self._h, len(insts), N.as_i32p(jobs), N.as_i32p(machines),
                                        offsets.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                        N.as_i32p(mach), N.as_i32p(dur))
        N.check(self._h, rc, "jss_load_instances")
        if env_to_inst is None:
            env_to_inst = np.arange(self.num_envs) % len(insts)
        self.env_to_instance = np.ascontiguousarray(env_to_inst, dtype=np.int32)
        assert self.env_to_instance.shape == (self.num_envs,)
        rc = self._L.jss_assign(self._h, N.as_i32p(self.env_to_instance))   # also performs the first reset
        N.check(self._h, rc, "jss_assign")
        self.env_jobs = jobs[self.env_to_instance]           # J_i per env (no-op index of env i)
        self.env_machines = machines[self.env_to_instance]
        sc = np.zeros((len(insts), 3), np.int64)
        for k in range(len(insts)):
            N.check(self._h, self._L.jss_instance_scalars(
                self._h, k, sc[k].ctypes.data_as(ctypes.POINTER(ctypes.c_int64))), "jss_instance_scalars")
        self.instance_scalars = sc                           # max_time_op, max_time_jobs, sum_op

    def _bind_buffers(self):
        b = N.JssBuffers()
        N.check(self._h, self._L.jss_get_buffers(self._h, ctypes.byref(b)), "jss_get_buffers")
        self._b = b
        self.jobs, self.machines = int(b.jobs_max), int(b.machines_max)
        n, J, M, w = self.num_envs, self.jobs, self.machines, N.backend.wrap
        d = self.device_index
        self.device = N.backend.torch_device(d)
        import torch
        self._mask_u8 = w(b.action_mask, (n, J + 1), np.uint8, d, strides=(b.mask_stride, 1))
        self.action_mask = self._mask_u8.view(torch.bool)
        self.real_obs = w(b.real_obs, (n, J, 7), np.float32, d)
        ss = (int(b.scalar_stride),)      # the five scalar outputs are fields of one 16-byte record per env
        self.reward = w(b.reward, (n,), np.float32, d, strides=ss)
        self.reward_raw = w(b.reward_raw, (n,), np.int32, d, strides=ss)
        self.done = w(b.done, (n,), np.uint8, d, strides=ss).view(torch.bool)
        self.current_time_step = w(b.time, (n,), np.int32, d, strides=ss)
        self._flags_done = w(b.flags_done, (n,), np.int32, d, strides=ss)
        self.solution = w(b.solution, (n, J, M), np.int32, d) if b.solution else None
        self.episode_count = w(b.episode_count, (n,), np.int32, d)
        self.last_makespan = w(b.last_makespan, (n,), np.int32, d)
        self.last_return = w(b.last_return, (n,), np.int32, d)
        self._x = {
            "todo": w(b.x_todo, (n, J), np.int32, d), "tufco": w(b.x_tufco, (n, J), np.int32, d),
            "idle_last": w(b.x_idle_last, (n, J), np.int32, d), "total_idle": w(b.x_total_idle, (n, J), np.int32, d),
            "col4": w(b.x_col4, (n, J), np.int32, d), "tuam": w(b.x_tuam, (n, M), np.int32, d),
            "legal": w(b.x_legal, (n, J), np.uint8, d), "blocked": w(b.x_blocked, (n, J), np.uint8, d),
        }
        self.host = None
        if b.host_mirror:
            # JSS_CREATE_HOST_MIRROR: the same memory seen from the host (pinned, device-mapped): numpy views, no copies
            def hv(ptr, shape, dt, strides=None):
                dt = np.dtype(dt)
                nbytes = (int(np.prod(shape)) * dt.itemsize if strides is None
                          else sum((sh - 1) * st for sh, st in zip(shape, strides)) + dt.itemsize)
                raw = np.frombuffer((ctypes.c_char * nbytes).from_address(int(ptr)), dtype=np.uint8)
                if strides is None:
                    return raw.view(dt).reshape(shape)
                return np.lib.stride_tricks.as_strided(raw[: nbytes // dt.itemsize * dt.itemsize].view(dt) if dt.itemsize > 1 else raw,
                                                       shape=shape, strides=strides)
            sc = hv(b.reward, (n, 4), np.int32)
            self.host = {
                "action_mask": hv(b.action_mask, (n, J + 1), np.uint8, strides=(int(b.mask_stride), 1)),
                "real_obs": hv(b.real_obs, (n, J, 7), np.float32), "scalars": sc,
                "todo": hv(b.x_todo, (n, J), np.int32), "tufco": hv(b.x_tufco, (n, J), np.int32),
                "idle_last": hv(b.x_idle_last, (n, J), np.int32), "total_idle": hv(b.x_total_idle, (n, J), np.int32),
                "col4": hv(b.x_col4, (n, J), np.int32), "tuam": hv(b.x_tuam, (n, M), np.int32),
                "legal": hv(b.x_legal, (n, J), np.uint8), "blocked": hv(b.x_blocked, (n, J), np.uint8),
                "actions": hv(b.mirror_actions, (n,), np.int32),
            }
            self._mirror_actions = w(b.mirror_actions, (n,), np.int32, d)
        self._truncated = torch.zeros(n, dtype=torch.bool, device=self.device)
        self._actions = torch.zeros(n, dtype=torch.int32, device=self.device)

    @property
    def flags(self):
        """Per-env JSS_FLAG_* bits (done / error / no-op legal) as an int32 tensor."""
        return self._flags_done >> 8

    # ---------------------------------------------------------------- lifetime
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._L.jss_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return N.backend.stream(self.device_index)

    def _obs(self):
        return {"real_obs": self.real_obs, "action_mask": self.action_mask}

    # ---------------------------------------------------------------- reference API, batched
    def reset(self, mask=None):
        """reset() of every env (or of the envs where `mask` is nonzero) -> obs (jss_env.py:145-181)."""
        ptr = None
        if mask is not None:
            import torch
            mask = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            ptr = ctypes.c_void_p(mask.data_ptr())
        N.check(self._h, self._L.jss_reset(self._h, ptr, self._stream()), "jss_reset")
        return self._obs()

    def step(self, actions):
        """actions: int32[N] on the env's device (torch) or anything torch.as_tensor accepts."""
        import torch
        a = torch.as_tensor(actions, device=self.device)
        if a.dtype != torch.int32 or not a.is_contiguous():
            a = a.to(torch.int32).contiguous()
        N.check(self._h, self._L.jss_step(self._h, ctypes.c_void_p(a.data_ptr()), self._stream()), "jss_step")
        return self._obs(), self.reward, self.done, self._truncated, {}

    def step_export_host(self):
        """Host-mirror batches (the single-env facade): apply the actions written to ``self.host["actions"]`` and decode
        the new state into the x_* arrays in ONE launch (jss_step_export), then wait; afterwards every array of
        ``self.host`` is current.  No per-transition copies: the kernels write straight into the pinned block."""
        rc = self._L.jss_step_export(self._h, ctypes.c_void_p(self._mirror_actions.data_ptr()), self._stream())
        N.check(self._h, rc, "jss_step_export")
        N.backend.synchronize(self.device_index)

    def step_sample(self, actions, rule: Union[str, int] = "RANDOM", coin: str = "device", out=None):
        """step(actions) fused with policy(rule) for the next decision (one launch): returns the usual
        step tuple plus the int32[N] tensor of next actions (`out`, default: in place of `actions`)."""
        import torch
        a = torch.as_tensor(actions, device=self.device)
        if a.dtype != torch.int32 or not a.is_contiguous():
            a = a.to(torch.int32).contiguous()
        out = a if out is None else out
        r = N.RULES[rule.upper()] if isinstance(rule, str) else int(rule)
        rc = self._L.jss_step_sample(self._h, ctypes.c_void_p(a.data_ptr()), r,
                                     N.COIN_DEVICE if coin == "device" else N.COIN_NEVER, self.seed,
                                     self._step_index, ctypes.c_void_p(out.data_ptr()), self._stream())
        N.check(self._h, rc, "jss_step_sample")
        self._step_index += 1
        return self._obs(), self.reward, self.done, self._truncated, {}, out

    def get_legal_actions(self):
        return self.action_mask

    # ---------------------------------------------------------------- policies on device
    def policy(self, rule: Union[str, int] = "RANDOM", coin: str = "device", out=None, step_index=None):
        """Device-side action selection (masked-uniform sampler or a dispatching rule)."""
        r = N.RULES[rule.upper()] if isinstance(rule, str) else int(rule)
        out = self._actions if out is None else out
        if step_index is None:
            step_index = self._step_index
            self._step_index += 1
        rc = self._L.jss_policy(self._h, r, N.COIN_DEVICE if coin == "device" else N.COIN_NEVER, self.seed,
                                int(step_index), ctypes.c_void_p(out.data_ptr()), self._stream())
        N.check(self._h, rc, "jss_policy")
        return out

    def set_cr_due_date_factor(self, factor: float):
        """CriticalRatio(due_date_factor) of the reference (dispatching.py:337-349) for later CR launches."""
        N.check(self._h, self._L.jss_set_cr_due_date_factor(self._h, float(factor)), "jss_set_cr_due_date_factor")

    def rollout(self, rule: Union[str, int], n_steps: int, write_obs: bool = True):
        """n_steps x (policy -> step) fused on device (DispatchingRule.run_episode, dispatching.py:55-75)."""
        r = N.RULES[rule.upper()] if isinstance(rule, str) else int(rule)
        rc = self._L.jss_rollout(self._h, r, self.seed, self._step_index, int(n_steps), int(bool(write_obs)),
                                 self._stream())
        N.check(self._h, rc, "jss_rollout")
        self._step_index += int(n_steps)
        return self._obs(), self.reward, self.done, self._truncated, {}

    def rollout_record(self, rule: Union[str, int], n_steps: int, out: Optional[Dict[str, Any]] = None):
        """n_steps x (policy -> step) fused on device WITH the trajectory recorded (jss_rollout_traj): returns
        {"real_obs": (K, N, J, 7) f32, "action_mask": (K, N, J+1) bool, "reward": (K, N) f32, "done": (K, N) bool,
        "actions": (K, N) i32, ...} as device tensors; pass the dict back as `out` to reuse the buffers."""
        import torch
        r = N.RULES[rule.upper()] if isinstance(rule, str) else int(rule)
        K, n, J, ms = int(n_steps), self.num_envs, self.jobs, int(self._b.mask_stride)
        if out is None or out["_obs"].shape[0] != K:
            dev = self.device
            # zero-filled once: rows of envs with fewer jobs than the batch maximum are only written up to J_i
            out = {"_obs": torch.zeros((K, n, J, 7), dtype=torch.float32, device=dev),
                   "_mask": torch.zeros((K, n, ms), dtype=torch.uint8, device=dev),
                   "_scalars": torch.zeros((K, n, 4), dtype=torch.int32, device=dev),
                   "actions": torch.zeros((K, n), dtype=torch.int32, device=dev)}
            out["real_obs"] = out["_obs"]
            out["action_mask"] = out["_mask"][:, :, : J + 1].view(torch.bool)
            out["reward"] = out["_scalars"][:, :, 0].view(torch.float32)
            out["reward_raw"] = out["_scalars"][:, :, 1]
            out["time"] = out["_scalars"][:, :, 2]
            out["done"] = (out["_scalars"][:, :, 3] & 1).bool() if N.backend.name != "cuda" else None
        rc = self._L.jss_rollout_traj(self._h, r, self.seed, self._step_index, K,
                                      ctypes.c_void_p(out["_obs"].data_ptr()), ctypes.c_void_p(out["_mask"].data_ptr()),
                                      ctypes.c_void_p(out["_scalars"].data_ptr()), ctypes.c_void_p(out["actions"].data_ptr()),
                                      self._stream())
        N.check(self._h, rc, "jss_rollout_traj")
        self._step_index += K
        out["done"] = (out["_scalars"][:, :, 3] & 1).bool()       # lazily evaluated view of the done bit
        return out

    # ---------------------------------------------------------------- host-buffer form
    def step_host(self, actions: np.ndarray, want_obs: bool = True):
        """step() with HOST buffers: H2D of the actions and D2H of the results inside the call."""
        a = np.ascontiguousarray(actions, dtype=np.int32)
        n, J = self.num_envs, self.jobs
        if not hasattr(self, "_host"):
            import torch
            pin = N.backend.name == "cuda"
            mk = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=pin)   # noqa: E731
            ms = int(self._b.mask_stride)
            self._host = {"mask": mk((n, ms), torch.uint8), "obs": mk((n, J, 7), torch.float32),
                          "scalars": mk((n, 4), torch.int32)}
            sc = self._host["scalars"].numpy()
            self._host_views = {
                "mask": self._host["mask"].numpy()[:, : J + 1].view(np.bool_), "obs": self._host["obs"].numpy(),
                "reward": sc.view(np.float32)[:, 0], "done": sc.view(np.uint8)[:, 12].view(np.bool_)}
        hb, hv = self._host, self._host_views
        rc = self._L.jss_step_host(self._h, ctypes.c_void_p(a.ctypes.data), ctypes.c_void_p(hb["mask"].data_ptr()),
                                   ctypes.c_void_p(hb["obs"].data_ptr()) if want_obs else None,
                                   ctypes.c_void_p(hb["scalars"].data_ptr()), self._stream())
        N.check(self._h, rc, "jss_step_host")
        obs = {"real_obs": hv["obs"], "action_mask": hv["mask"]}
        return obs, hv["reward"], hv["done"], np.zeros(n, np.bool_), {}

    # pipelined form: begin -> wait_mask -> (choose next actions) -> begin ... ; obs lands in alternating buffers
    def host_step_begin(self, actions: np.ndarray, packed: bool = False, dma_fraction: float = 0.0):
        """Enqueue one host-buffer step and return immediately (see jss_host_step_begin).  Results land
        in this call's slot of two alternating pinned buffer sets; use host_wait_mask()/host_wait_obs().
        packed=True ships the observation as 10-byte integer records per job instead of 28 bytes of fp32
        (jss_host_step_begin_packed); host_wait_obs() then expands them to the exact float observation.
        dma_fraction > 0 (with packed): that share of the envs ships final fp32 rows by DMA instead, so PCIe and the
        host cores each work on their part in parallel (jss_host_step_begin_hybrid)."""
        a = np.ascontiguousarray(actions, dtype=np.int32)
        n, J = self.num_envs, self.jobs
        if not hasattr(self, "_pipe"):
            import torch
            pin = N.backend.name == "cuda"
            mk = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=pin)   # noqa: E731
            ms = int(self._b.mask_stride)
            ws = int(self._L.jss_host_wire_stride(self._h))
            self._pipe = [{"mask": mk((n, ms), torch.uint8), "obs": None, "wire": None, "wire_stride": ws, "n_dma": 0,
                           "scalars": mk((n, 4), torch.int32), "actions": mk((n,), torch.int32), "packed": False,
                           "expanded": True} for _ in range(2)]
            self._pipe_slot = 0
            self._pipe_mk = mk
            self._pipe_inflight = 0
        if self._pipe_inflight >= 2:
            # the slot about to be reused belongs to the begin before the latest one: its transfers must have drained
            N.check(self._h, self._L.jss_host_wait(self._h, N.WAIT_OBS_PREV), "jss_host_wait")
        self._pipe_slot ^= 1
        b = self._pipe[self._pipe_slot]
        if b["obs"] is None:
            import torch
            # fp32 observation buffer: DMA target (pinned) in plain mode, expansion target in packed mode
            b["obs"] = self._pipe_mk((n, J, 7), torch.float32)
        if packed and b["wire"] is None:
            import torch
            b["wire"] = self._pipe_mk((n, b["wire_stride"]), torch.uint8)
        b["actions"].numpy()[:] = a                      # pinned copy: the H2D must not race with the caller's array
        b["packed"] = bool(packed)
        b["expanded"] = not packed
        b["n_dma"] = 0
        if packed and dma_fraction > 0.0:
            g = 256 if n >= 4096 else 1
            b["n_dma"] = min(n, int(dma_fraction * n) // g * g)
        if packed and b["n_dma"] > 0:
            rc = self._L.jss_host_step_begin_hybrid(self._h, ctypes.c_void_p(b["actions"].data_ptr()),
                                                    ctypes.c_void_p(b["mask"].data_ptr()),
                                                    ctypes.c_void_p(b["wire"].data_ptr()),
                                                    ctypes.c_void_p(b["obs"].data_ptr()), b["n_dma"],
                                                    ctypes.c_void_p(b["scalars"].data_ptr()), self._stream())
        elif packed:
            rc = self._L.jss_host_step_begin_packed(self._h, ctypes.c_void_p(b["actions"].data_ptr()),
                                                    ctypes.c_void_p(b["mask"].data_ptr()),
                                                    ctypes.c_void_p(b["wire"].data_ptr()),
                                                    ctypes.c_void_p(b["scalars"].data_ptr()), self._stream())
        else:
            rc = self._L.jss_host_step_begin(self._h, ctypes.c_void_p(b["actions"].data_ptr()),
                                             ctypes.c_void_p(b["mask"].data_ptr()), ctypes.c_void_p(b["obs"].data_ptr()),
                                             ctypes.c_void_p(b["scalars"].data_ptr()), self._stream())
        N.check(self._h, rc, "jss_host_step_begin")
        self._pipe_inflight = min(2, self._pipe_inflight + 1)
        return self._pipe_slot

    def host_wait_mask(self):
        """Block until mask / reward / done of the latest host_step_begin have landed; returns them."""
        N.check(self._h, self._L.jss_host_wait(self._h, N.WAIT_MASK), "jss_host_wait")
        b = self._pipe[self._pipe_slot]
        sc = b["scalars"].numpy()
        return (b["mask"].numpy()[:, : self.jobs + 1].view(np.bool_), sc.view(np.float32)[:, 0],
                sc.view(np.uint8)[:, 12].view(np.bool_))

    def host_wait_obs(self, previous: bool = False):
        """Block until the observation of the latest host_step_begin (or, with previous=True, of the one
        before it, which may be consumed while the latest is still streaming) has landed; returns (N, J, 7)
        float32.  In packed mode the integer rows are expanded here (multi-threaded host helper)."""
        N.check(self._h, self._L.jss_host_wait(self._h, N.WAIT_OBS_PREV if previous else N.WAIT_OBS), "jss_host_wait")
        b = self._pipe[self._pipe_slot ^ (1 if previous else 0)]
        if b["packed"] and not b["expanded"]:
            rc = self._L.jss_host_expand_obs_range(self._h, ctypes.c_void_p(b["wire"].data_ptr()),
                                                   ctypes.c_void_p(b["scalars"].data_ptr()),
                                                   ctypes.c_void_p(b["obs"].data_ptr()), int(b["n_dma"]), self.num_envs)
            N.check(self._h, rc, "jss_host_expand_obs")
            b["expanded"] = True
        return b["obs"].numpy()

    @staticmethod
    def host_configure(threads: int = 0, bind_numa_of_device: int = -1) -> int:
        """Size / bind the host worker pool (jss_host_configure); call before the first host helper runs."""
        return int(N.backend.library().jss_host_configure(int(threads), int(bind_numa_of_device)))

    def host_masked_random(self, mask: np.ndarray, step_index: int) -> np.ndarray:
        """Same draw as policy('RANDOM') but from a host mask (for host-side agents / tests)."""
        m = np.asarray(mask)
        if m.dtype != np.uint8:
            m = m.view(np.uint8) if m.dtype == np.bool_ else m.astype(np.uint8)
        if m.strides[1] != 1:
            m = np.ascontiguousarray(m)
        out = np.empty(m.shape[0], np.int32)
        rc = self._L.jss_host_masked_random(ctypes.c_void_p(m.ctypes.data), m.shape[0], m.shape[1], m.strides[0], self.seed,
                                            self.env_id_base, int(step_index), ctypes.c_void_p(out.ctypes.data))
        if rc != 0:
            raise N.NativeError("jss_host_masked_random failed")
        return out

    # ---------------------------------------------------------------- statistics / state
    def stats(self) -> Dict[str, int]:
        out = np.zeros(len(N.STATS_KEYS), np.int64)
        rc = self._L.jss_stats(self._h, out.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), self._stream())
        N.check(self._h, rc, "jss_stats")
        return dict(zip(N.STATS_KEYS, (int(v) for v in out)))

    def env_instances(self) -> Dict[str, Any]:
        """Generator mode: every env's current instance as device tensors {"machine": (N, J, M), "duration": (N, J, M),
        "index": (N,)} int32 -- index = how many resets the env has had since the first (the k of its instance)."""
        import torch
        if self.generator is None:
            raise N.NativeError("env_instances() needs a generator-mode env ({'generator': ...} config)")
        n, J, M = self.num_envs, self.jobs, self.machines
        out = {"machine": torch.empty((n, J, M), dtype=torch.int32, device=self.device),
               "duration": torch.empty((n, J, M), dtype=torch.int32, device=self.device),
               "index": torch.empty((n,), dtype=torch.int32, device=self.device)}
        rc = self._L.jss_get_env_instances(self._h, *(ctypes.c_void_p(out[k].data_ptr()) for k in ("machine", "duration", "index")),
                                           self._stream())
        N.check(self._h, rc, "jss_get_env_instances")
        return out

    def export_state(self) -> Dict[str, Any]:
        """Canonical per-env integer state as device tensors (snapshot); see jss_b200.h."""
        N.check(self._h, self._L.jss_export_state(self._h, self._stream()), "jss_export_state")
        d = dict(self._x)
        d["t"] = self.current_time_step
        d["flags"] = self._flags_done
        return d

    def import_state(self, state: Dict[str, Any], mask=None):
        """Restore a snapshot taken with export_state() (tensors are copied into the library's buffers)."""
        for k, dst in self._x.items():
            if state[k].data_ptr() != dst.data_ptr():
                dst.copy_(state[k])
        if state["t"].data_ptr() != self.current_time_step.data_ptr():
            self.current_time_step.copy_(state["t"])
        if state["flags"].data_ptr() != self._flags_done.data_ptr():
            self._flags_done.copy_(state["flags"])
        ptr = None
        if mask is not None:
            import torch
            mask = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            ptr = ctypes.c_void_p(mask.data_ptr())
        N.check(self._h, self._L.jss_import_state(self._h, ptr, self._stream()), "jss_import_state")

    @property
    def launch_count(self) -> int:
        return int(self._L.jss_launch_count(self._h))

    def synchronize(self):
        N.backend.synchronize(self.device_index)
