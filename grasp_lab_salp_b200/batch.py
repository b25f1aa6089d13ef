"""SalpBatch: N independent SalpRobotEnv instances on one GPU, behind the C ABI.

Two faces over the same handle:

* host face (numpy): ``reset()`` / ``step()`` call ``salp_reset_host`` / ``salp_step_host`` --
  H2D of the actions, the kernels, D2H of the results, one stream synchronise.  This is what
  the SB3-VecEnv-shaped wrapper (vec_env.py) and the parity tests use.
* device face (torch tensors, zero-copy): ``reset_device()`` / ``step_device()`` pass raw device
  pointers to ``salp_reset`` / ``salp_step`` on the current torch stream, no synchronisation.
  This is what rollouts and bench.py use.

Semantics follow the reference's SalpRobotEnv.reset()/step() (src/salp_robot_env.py:114-155,
196-299) per env; ``auto_reset=True`` adds what an SB3 DummyVecEnv/SubprocVecEnv worker does
around it (reset the finished env, return the post-reset observation, keep the last observation
of the finished episode in ``terminal_obs``).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .params import (NUM_EPISODE_METRICS, NUM_REWARD_TERMS, STEP_AUTORESET, STEP_CHECK_HANDOFF, STEP_FUSED, STEP_GENERIC, STEP_PIPELINE, STEP_SORT_BY_K, SalpParams,
                     default_params, field_dtype, field_id)


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class SalpBatch:
    def __init__(self, num_envs: int, params: SalpParams | None = None, seed: int = 0,
                 env_id_offset: int = 0, device: int = 0, _cdll=None):
        self._L = _cdll if _cdll is not None else _lib.load()
        self.params = (params or default_params()).copy()
        self.num_envs = int(num_envs)
        self.obs_dim = self.params.obs_dim
        self.device = int(device)
        h = C.c_void_p()
        rc = self._L.salp_create(C.byref(self.params), self.num_envs, self.device, C.c_uint64(seed),
                                 int(env_id_offset), C.byref(h))
        if rc != 0:
            raise _lib.SalpError(rc, (self._L.salp_last_error(None) or b"").decode())
        self._h = h
        n, d = self.num_envs, self.obs_dim
        # persistent host buffers of the numpy face (page-locked when torch can provide them, so
        # the D2H copies of salp_step_host are true async DMA)
        self._pinned = []
        self.obs = self.host_buffer((n, d), np.float32)
        self.terminal_obs = self.host_buffer((n, d), np.float32)
        self.reward = self.host_buffer((n,), np.float32)
        self.terminated = self.host_buffer((n,), np.uint8)
        self.truncated = self.host_buffer((n,), np.uint8)
        self.terms = self.host_buffer((n, NUM_REWARD_TERMS), np.float64)
        self.substeps = self.host_buffer((n,), np.int32)
        self.metrics = self.host_buffer((n, NUM_EPISODE_METRICS), np.float64)
        self._io_host = _lib.SalpStepIO()
        self._io_host_extras = None
        self._io_host_ref = None
        self._io_host_bufs = (None,) * 5
        self._dev = None          # lazily created torch output tensors of the device face

    def host_buffer(self, shape, dtype) -> np.ndarray:
        """Zero-filled host array, page-locked if possible (callers can use it for actions too)."""
        if self._cdll_is_cuda():
            try:
                import torch
                tdt = {np.float32: torch.float32, np.float64: torch.float64, np.uint8: torch.uint8,
                       np.int32: torch.int32}[np.dtype(dtype).type]
                t = torch.zeros(tuple(shape), dtype=tdt).pin_memory()
                self._pinned.append(t)
                return t.numpy()
            except Exception:
                pass
        return np.zeros(shape, dtype)

    def _cdll_is_cuda(self) -> bool:
        return b"sm_100a" in (self._L.salp_build_info() or b"")

    # ------------------------------------------------------------------ lifetime / errors
    def close(self):
        if getattr(self, "_h", None):
            self._L.salp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise _lib.SalpError(rc, (self._L.salp_last_error(self._h) or b"").decode())

    def check(self):
        """Raise if a kernel recorded a device-side error (synchronises)."""
        self._check(self._L.salp_check(self._h))

    @property
    def launch_count(self) -> int:
        return int(self._L.salp_launch_count(self._h))

    @property
    def last_step_kernel(self) -> str:
        """Name of the step kernel the library launched for the last step (salp_last_step_kernel)."""
        return (self._L.salp_last_step_kernel(self._h) or b"").decode()

    # ------------------------------------------------------------------ host (numpy) face
    def set_scene_pool(self, targets, obstacles):
        """Replace the built-in Philox scene sampler by caller-given scenes (parity with an
        external oracle): targets [N,P,2], obstacles [N,P,num_obstacles,2]; None = built-in."""
        if targets is None:
            self._check(self._L.salp_set_scene_pool(self._h, None, None, 0))
            return
        targets = np.ascontiguousarray(targets, np.float32)
        obstacles = np.ascontiguousarray(obstacles, np.float32)
        P = targets.shape[1]
        if targets.shape != (self.num_envs, P, 2) or obstacles.shape != (self.num_envs, P, self.params.num_obstacles, 2):
            raise ValueError("scene pool shapes must be [N,P,2] and [N,P,num_obstacles,2]")
        self._check(self._L.salp_set_scene_pool(self._h, _np_ptr(targets), _np_ptr(obstacles), P))

    def reset(self, mask=None) -> np.ndarray:
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        if m is not None and m.shape != (self.num_envs,):
            raise ValueError("mask must have shape [num_envs]")
        if m is None:
            self._check(self._L.salp_reset_host(self._h, None, _np_ptr(self.obs)))
        else:
            tmp = np.empty_like(self.obs)
            self._check(self._L.salp_reset_host(self._h, _np_ptr(m), _np_ptr(tmp)))
            sel = m.astype(bool)
            self.obs[sel] = tmp[sel]
        return self.obs

    def step(self, actions, auto_reset: bool = False, sort_by_k: bool = False, extras: bool = True,
             pipeline=None, generic: bool = False, check_handoff: bool = False):
        a = actions
        if not (type(a) is np.ndarray and a.dtype == np.float32 and a.flags.c_contiguous):
            a = np.ascontiguousarray(actions, np.float32)
        if a.shape != (self.num_envs, 3):
            raise ValueError(f"actions must have shape [{self.num_envs}, 3]")
        io = self._io_host
        bufs = (self.obs, self.reward, self.terminated, self.truncated, self.terminal_obs)
        if self._io_host_extras is not extras or any(x is not y for x, y in zip(bufs, self._io_host_bufs)):
            # (output pointers only change with `extras` or when a caller swaps in its own arrays)
            self._io_host_bufs = bufs
            io.obs = self.obs.ctypes.data
            io.reward = self.reward.ctypes.data
            io.terminated = self.terminated.ctypes.data
            io.truncated = self.truncated.ctypes.data
            io.terminal_obs = self.terminal_obs.ctypes.data
            io.reward_terms = self.terms.ctypes.data if extras else None
            io.substeps = self.substeps.ctypes.data if extras else None
            io.episode_metrics = self.metrics.ctypes.data if extras else None
            self._io_host_extras = extras
            self._io_host_ref = C.byref(io)
        io.actions = a.__array_interface__["data"][0]
        flags = ((STEP_AUTORESET if auto_reset else 0) | (STEP_SORT_BY_K if sort_by_k else 0)
                 | (0 if pipeline is None else (STEP_PIPELINE if pipeline else STEP_FUSED))
                 | (STEP_GENERIC if generic else 0) | (STEP_CHECK_HANDOFF if check_handoff else 0))
        rc = self._L.salp_step_host(self._h, self._io_host_ref, flags)
        if rc != 0:
            self._check(rc)
        return self.obs, self.reward, self.terminated, self.truncated

    def get_state(self, name: str) -> np.ndarray:
        out = np.zeros(self.num_envs, field_dtype(name))
        self._check(self._L.salp_get_state(self._h, field_id(name), _np_ptr(out), 0, self.num_envs))
        return out

    def set_state(self, name: str, values):
        v = np.ascontiguousarray(np.broadcast_to(values, (self.num_envs,)), field_dtype(name))
        self._check(self._L.salp_set_state(self._h, field_id(name), _np_ptr(v), 0, self.num_envs))

    TRACE_COLUMNS = ("position_world", "euler_angle", "velocity", "angular_velocity", "length", "width")

    def trace_cycle(self, env: int, action) -> dict:
        """History feed: the per-substep histories the reference records with
        Robot.enable_history_recording() (robot.py:681-776) for the NEXT cycle of one env, computed
        in float64 reference arithmetic WITHOUT advancing the env.  Returns arrays of K rows."""
        a = np.ascontiguousarray(action, np.float32).reshape(3)
        cap = 4096
        buf = np.zeros((cap, 14), np.float64)
        K = C.c_int32(0)
        self._check(self._L.salp_trace_cycle(self._h, int(env), _np_ptr(a), _np_ptr(buf), cap, C.byref(K)))
        k = min(K.value, cap)
        t = buf[:k]
        return dict(substeps=K.value, position_world=t[:, 0:3].copy(), euler_angle=t[:, 3:6].copy(),
                    velocity=t[:, 6:9].copy(), angular_velocity=t[:, 9:12].copy(), length=t[:, 12].copy(),
                    width=t[:, 13].copy())

    # ------------------------------------------------------------------ device (torch) face
    def _device_buffers(self):
        if self._dev is None:
            import torch
            dev = torch.device("cuda", self.device)
            n, d = self.num_envs, self.obs_dim
            self._dev = dict(
                obs=torch.zeros((n, d), dtype=torch.float32, device=dev),
                terminal_obs=torch.zeros((n, d), dtype=torch.float32, device=dev),
                reward=torch.zeros(n, dtype=torch.float32, device=dev),
                terminated=torch.zeros(n, dtype=torch.uint8, device=dev),
                truncated=torch.zeros(n, dtype=torch.uint8, device=dev),
                substeps=torch.zeros(n, dtype=torch.int32, device=dev),
                terms=torch.zeros((n, NUM_REWARD_TERMS), dtype=torch.float64, device=dev),
                metrics=torch.zeros((n, NUM_EPISODE_METRICS), dtype=torch.float64, device=dev),
            )
            self._io_dev = _lib.SalpStepIO()
        return self._dev

    @staticmethod
    def _stream_ptr(device: int):
        import torch
        return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)

    def reset_device(self, mask=None):
        """mask: optional uint8/bool CUDA tensor [N].  Returns the obs tensor [N,D] (device)."""
        import torch
        bufs = self._device_buffers()
        mptr = None
        if mask is not None:
            mask = mask.to(torch.uint8).contiguous()
            mptr = C.c_void_p(mask.data_ptr())
            tmp = torch.empty_like(bufs["obs"])
            self._check(self._L.salp_reset(self._h, mptr, C.c_void_p(tmp.data_ptr()), self._stream_ptr(self.device)))
            bufs["obs"] = torch.where(mask.bool()[:, None], tmp, bufs["obs"])
        else:
            self._check(self._L.salp_reset(self._h, None, C.c_void_p(bufs["obs"].data_ptr()),
                                           self._stream_ptr(self.device)))
        return bufs["obs"]

    def step_device(self, actions, auto_reset: bool = True, sort_by_k: bool = False, extras: bool = False,
                    pipeline=None, generic: bool = False, extra_flags: int = 0, out=None):
        """actions: float32 CUDA tensor [N,3] on this batch's device.  Asynchronous on the current
        torch stream.  Returns (obs, reward, terminated, truncated) device tensors (reused every
        call); ``self.dev["terminal_obs"]`` etc. hold the rest.

        out: optional dict of caller-owned tensors that receive this step's obs / reward / terminated /
        truncated / terminal_obs instead of the batch's own buffers (any subset; e.g. views into a replay
        ring, so that a step is stored with no copy).  Contiguous, on this device: obs and terminal_obs
        float32 [N, D], reward float32 [N], terminated and truncated 1-byte (uint8 / bool) [N]."""
        import torch
        bufs = self._device_buffers()
        if actions.dtype != torch.float32 or not actions.is_cuda or tuple(actions.shape) != (self.num_envs, 3):
            raise ValueError("actions must be a float32 CUDA tensor of shape [num_envs, 3]")
        if out:
            n, d = self.num_envs, self.obs_dim
            want = dict(obs=(n, d), terminal_obs=(n, d), reward=(n,), terminated=(n,), truncated=(n,))
            bufs = dict(bufs)
            for k, t in out.items():
                if k not in want:
                    raise ValueError(f"out: unknown buffer {k!r} (expected a subset of {sorted(want)})")
                ok_dtype = t.dtype == torch.float32 if k in ("obs", "terminal_obs", "reward") else t.element_size() == 1
                if not (ok_dtype and tuple(t.shape) == want[k] and t.is_contiguous() and t.is_cuda
                        and t.device.index == self.device):
                    raise ValueError(f"out[{k!r}] must be a contiguous {'float32' if k in ('obs', 'terminal_obs', 'reward') else 'uint8 / bool'} "
                                     f"tensor of shape {list(want[k])} on cuda:{self.device}")
                bufs[k] = t
        actions = actions.contiguous()
        io = self._io_dev
        io.actions = actions.data_ptr()
        io.obs = bufs["obs"].data_ptr()
        io.reward = bufs["reward"].data_ptr()
        io.terminated = bufs["terminated"].data_ptr()
        io.truncated = bufs["truncated"].data_ptr()
        io.terminal_obs = bufs["terminal_obs"].data_ptr()
        io.substeps = bufs["substeps"].data_ptr()
        io.reward_terms = bufs["terms"].data_ptr() if extras else None
        io.episode_metrics = bufs["metrics"].data_ptr() if extras else None
        flags = ((STEP_AUTORESET if auto_reset else 0) | (STEP_SORT_BY_K if sort_by_k else 0)
                 | (0 if pipeline is None else (STEP_PIPELINE if pipeline else STEP_FUSED))
                 | (STEP_GENERIC if generic else 0) | int(extra_flags))
        self._check(self._L.salp_step(self._h, C.byref(io), flags, self._stream_ptr(self.device)))
        return bufs["obs"], bufs["reward"], bufs["terminated"], bufs["truncated"]

    @property
    def dev(self):
        return self._device_buffers()

    def state_tensor(self, name: str):
        """Zero-copy (strided) torch view of one state field over all envs (salp_state_ptr)."""
        import torch
        p = C.c_void_p()
        stride = C.c_int64(0)
        self._check(self._L.salp_state_ptr(self._h, field_id(name), C.byref(p), C.byref(stride)))
        dt = {np.float64: torch.float64, np.float32: torch.float32, np.int32: torch.int32}[field_dtype(name)]
        iface = {"shape": (self.num_envs,), "typestr": np.dtype(field_dtype(name)).str,
                 "data": (p.value, False), "version": 2, "strides": (int(stride.value),)}

        class _Holder:
            __cuda_array_interface__ = iface
        t = torch.as_tensor(_Holder(), device=torch.device("cuda", self.device))
        assert t.dtype == dt
        t._salp_owner = self   # keep the handle alive as long as the view
        return t
