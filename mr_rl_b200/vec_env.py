"""VecMREnv — the batched, device-resident MR_Env (reference: MR_env.py:21-229, MR_simulator.py:8-94).

Same gym surface as the reference (``reset`` / ``step`` / ``observation_space`` / ``action_space`` /
``init_space`` / ``last_pos`` / ``state_prime`` / ``counter``), vectorised over ``num_envs`` envs
whose state lives structure-of-arrays in HBM.  Every method launches hand-written sm_100a
kernels through the C ABI (include/mr_rl_b200.h); there is no CPU path.

PyTorch is used for device memory, streams and (optionally) torch.distributed — nothing else.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import _lib as L
from .learning_module import HeadingTrackingPolicy
from .spaces import Box

_DT = {torch.float64: L.MR_F64, torch.float32: L.MR_F32}
_NOISE = {"none": L.NOISE_NONE, "table": L.NOISE_TABLE, "philox": L.NOISE_PHILOX}
_PAD = 16          # rows are padded so every SoA row starts 16-byte aligned for any dtype


def _row_stride(n):
    """Elements between the SoA rows of one tensor: n rounded up to 16, plus 256 when that is a large power-of-two multiple.
    The rows of a tile are fetched together (one tensor-map box, or back-to-back bulk copies); with a power-of-two row
    stride they all land on the same DRAM channels.  Measured on B200 at 2^20 envs (noise-free fp64 step, us per launch):
    stride 2^20 -> 28.8 (1-D copies) / 29.5 (tensor maps), stride 2^20 + 256 -> 28.0 / 27.9."""
    npad = (n + _PAD - 1) // _PAD * _PAD
    if npad >= (1 << 16) and npad % 4096 == 0:
        npad += 256
    return npad


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def raise_for_status(status):
    """Raise what the reference raises for the first failed envs of the sticky status flags ``status`` [N] (uint8)."""
    flags = int(status.max().item()) if status.numel() else 0
    if flags == 0:
        return
    idx = torch.nonzero(status)[:8, 0].tolist()
    if flags & L.ENV_NOISE_OVERFLOW:
        raise L.MRLibraryError(f"noise table exhausted for envs {idx}")
    if flags & L.ENV_NONFINITE:
        raise ValueError(f"non-finite state in envs {idx} (scipy: 'All components of the initial state `y0` must be finite')")
    raise RuntimeError(f"integrator failed in envs {idx} (scipy: 'Attempt to step on a failed or finished solver')")


class VecMREnv:
    """``num_envs`` independent MR_Env instances stepped by one kernel launch.

    Parameters
    ----------
    num_envs : int
    device : torch device (must be CUDA)
    dtype : torch.float64 (parity: 1e-9) or torch.float32 (storage only; 1e-4)
    noise : "philox" (in-kernel counter-based generator), "table" (shared pre-generated
        standard-normal tensor ``noise_table[L, num_envs]`` — the parity mode) or "none"
    seed, env_base : Philox key and the global index of local env 0 (sharding across GPUs
        keeps trajectories independent of the number of ranks)
    auto_reset : restart an env from ``init_space`` right after a terminal step
    reward_mode : "const" (rew = 10, MR_env.py:89) or "shaped" (calculate_reward, MR_env.py:118-134)
    per_env_params : keep Simulator.a0 / noise_var / is_mismatched (MR_simulator.py:16-19, per-instance attributes set
        by every reset, MR_env.py:179-183) as per-env rows instead of launch scalars: ``reset`` then takes scalars or
        [N] arrays for them, a masked reset may change them, and one launch steps envs with different models
    """

    def __init__(self, num_envs, device="cuda", dtype=torch.float64, noise="philox", seed=0, env_base=0,
                 auto_reset=False, reward_mode="const", noise_table=None, time_table_len=4096, host_mapped_aux=False,
                 per_env_params=False):
        self.lib = L.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.MRLibraryError("VecMREnv needs a CUDA device: there is no CPU fallback")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if dtype not in _DT:
            raise ValueError("dtype must be torch.float64 or torch.float32")
        self.num_envs = int(num_envs)
        self.dtype = dtype
        self._dt = _DT[dtype]
        n = self.num_envs
        self._np = npad = _row_stride(n)
        dev = self.device

        # --- spaces and constants, MR_env.py:34-63 -------------------------------------------
        # (max_timesteps, min_dist2goal, init_space, action_space, observation_space are properties further down: the
        #  kernels read them from self.params, so assigning them — as users of the reference do — writes through)
        self.params = L.default_params()
        self.action_space = Box(low=np.array([0, 0]), high=np.array([20, np.pi * 2]))
        self.params.action_high[1] = 2 * math.pi     # the default keeps the float64 bound (a Box stores float32)
        self.observation_space = Box(low=np.array([-5000, -5000, -5000, -5000, 0]),
                                     high=np.array([5000, 5000, 5000, 5000, 80000]))
        self.init_space = Box(low=np.array([100, 100]), high=np.array([120, 120]))
        self.max_timesteps = 50
        self.min_dist2goal = 30
        self.init_goal = np.zeros(2)

        # --- Simulator parameters, MR_simulator.py:12-19 --------------------------------------
        self.params.a0 = 0.0
        self.params.noise_var = 0.0
        self.params.auto_reset = 1 if auto_reset else 0
        self.params.reward_mode = {"const": L.REWARD_CONST10, "shaped": L.REWARD_SHAPED}[reward_mode]
        self.number_iterations = 100

        # --- device state: SoA rows --------------------------------------------------------------
        self._state = torch.zeros(5, npad, dtype=dtype, device=dev)          # x, y, fx, fy, h
        self._counter = torch.zeros(npad, dtype=torch.int32, device=dev)
        self._cursor = torch.zeros(npad, dtype=torch.int32, device=dev)
        # host_mapped_aux (the single-env facade): status flags and state_prime live in page-locked HOST memory that the
        # kernels address directly, so a step needs no device->host read besides the one stream synchronisation
        aux = (lambda *s, **k: torch.zeros(*s, **k).pin_memory()) if host_mapped_aux else (lambda *s, **k: torch.zeros(*s, device=dev, **k))
        self._status = aux(npad, dtype=torch.uint8)
        self._obs = torch.zeros(5, npad, dtype=dtype, device=dev)            # x, y, gx, gy, d
        self._rew = torch.zeros(npad, dtype=dtype, device=dev)
        self._done = torch.zeros(npad, dtype=torch.uint8, device=dev)
        self._sp = aux(2, npad, dtype=dtype)                                 # Simulator.state_prime
        self._stats = torch.zeros(L.STATS_LEN, dtype=torch.float64, device=dev)
        tt = np.zeros(int(time_table_len), dtype=np.float64)
        self.lib.mr_fill_time_table_host(tt.ctypes.data_as(C.c_void_p), len(tt), self.params.time_span)
        self._tt = torch.from_numpy(tt).to(dev)

        self.per_env_params = bool(per_env_params)
        self._a0_row = self._sigma_row = self._mism_row = None
        if self.per_env_params:
            self._a0_row = torch.zeros(npad, dtype=torch.float64, device=dev)
            self._sigma_row = torch.zeros(npad, dtype=torch.float64, device=dev)
            self._mism_row = torch.zeros(npad, dtype=torch.uint8, device=dev)
        self._c_state = L.EnvState(*[_ptr(self._state[i]) for i in range(5)], _ptr(self._counter),
                                   _ptr(self._cursor), _ptr(self._status), _ptr(self._a0_row), _ptr(self._sigma_row),
                                   _ptr(self._mism_row))
        self._c_tt = L.TimeTable(_ptr(self._tt), len(tt), 0)
        self._c_out = L.StepOut(_ptr(self._obs), _ptr(self._rew), _ptr(self._done), _ptr(self._sp), npad)
        self._c_out_lean = L.StepOut(_ptr(self._obs), _ptr(self._rew), _ptr(self._done), C.c_void_p(0), npad)

        # --- noise -----------------------------------------------------------------------------
        self.noise_kind = noise
        self._noise_table = None
        self._c_noise = L.Noise(_NOISE[noise], 0, C.c_void_p(0), 0, int(seed) & (2**64 - 1), 0, int(env_base), C.c_void_p(0))
        if noise == "table":
            if noise_table is None:
                raise ValueError("noise='table' needs noise_table[L, num_envs] (standard normals, float64)")
            self.set_noise_table(noise_table)
        self._step_index = 0
        self.want_state_prime = True
        self._pinned = {}
        self.kernel_launches = 0
        # per-step call overhead: argument references and result views are built once
        self._dev_index = self.device.index
        self._call_step = self.lib.mr_env_step
        self._b_state, self._b_params, self._b_tt = C.byref(self._c_state), C.byref(self.params), C.byref(self._c_tt)
        self._b_out, self._b_out_lean = C.byref(self._c_out), C.byref(self._c_out_lean)
        self._views = (self._obs[:, :n].t(), self._rew[:n], self._done[:n], {})

    # ---- properties mirroring the reference attributes ------------------------------------
    # MR_env.py:34-63 — plain attributes in the reference; here every assignment also updates the launch parameters
    @property
    def max_timesteps(self):
        return self.params.max_timesteps

    @max_timesteps.setter
    def max_timesteps(self, v):
        self.params.max_timesteps = int(v)

    @property
    def min_dist2goal(self):
        return self.params.min_dist2goal

    @min_dist2goal.setter
    def min_dist2goal(self, v):
        self.params.min_dist2goal = float(v)

    @property
    def init_space(self):
        return self._init_space

    @init_space.setter
    def init_space(self, box):
        self._init_space = box
        for i in range(2):
            self.params.init_low[i] = float(box.low[i])
            self.params.init_high[i] = float(box.high[i])

    @property
    def action_space(self):
        return self._action_space

    @action_space.setter
    def action_space(self, box):
        self._action_space = box
        for i in range(2):
            self.params.action_high[i] = float(box.high[i])      # in-kernel random / actor policies scale by the upper bound

    @property
    def observation_space(self):
        return self._observation_space

    @observation_space.setter
    def observation_space(self, box):
        # the kernels test |x|, |y| <= bound_xy and 0 <= d <= bound_d (MR_env.py:37-39 is symmetric in x, y)
        lo, hi = np.asarray(box.low, dtype=np.float64), np.asarray(box.high, dtype=np.float64)
        if not (lo[0] == -hi[0] and lo[1] == -hi[1] and hi[0] == hi[1] and lo[4] == 0):
            raise ValueError("observation_space must be [-b, b] in x and y and [0, bd] in the distance")
        self._observation_space = box
        self.params.bound_xy = float(hi[0])
        self.params.bound_d = float(hi[4])

    @property
    def a0(self):
        """Simulator.a0: the launch scalar, or the [N] device row with ``per_env_params``."""
        return self._a0_row[:self.num_envs] if self.per_env_params else self.params.a0

    @property
    def noise_var(self):
        return self._sigma_row[:self.num_envs] if self.per_env_params else self.params.noise_var

    @property
    def is_mismatched(self):
        return self._mism_row[:self.num_envs].bool() if self.per_env_params else bool(self.params.is_mismatched)

    @property
    def time_span(self):
        return self.params.time_span

    @property
    def last_pos(self):
        """[N, 2] positions (MR_Env.last_pos / Simulator.last_state)."""
        return self._state[:2, :self.num_envs].t()

    @property
    def state_prime(self):
        """[N, 2] last RHS evaluation (Simulator.state_prime, MR_simulator.py:87)."""
        return self._sp[:, :self.num_envs].t()

    @property
    def counter(self):
        return self._counter[:self.num_envs]

    @property
    def obs(self):
        """[N, 5] view of the SoA observation rows [x, y, goal_x, goal_y, distance]."""
        return self._obs[:, :self.num_envs].t()

    @property
    def status(self):
        return self._status[:self.num_envs]

    @property
    def stats(self):
        return self._stats

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def set_noise_table(self, table):
        t = torch.as_tensor(table, dtype=torch.float64).to(self.device).contiguous()
        if t.dim() != 2 or t.shape[1] != self.num_envs:
            raise ValueError(f"noise_table must be [L, {self.num_envs}] (draw-major), got {tuple(t.shape)}")
        self._noise_table = t
        self._c_noise.table = t.data_ptr()
        self._c_noise.table_len = t.shape[0]

    def _noise_for(self, sigma):
        """sigma == 0 consumes no draws unless the parity table is in use (cursor discipline)."""
        nz = self._c_noise
        if self.noise_kind == "table":
            nz.mode = L.NOISE_TABLE
        elif self.per_env_params and self.noise_kind == "philox":
            nz.mode = L.NOISE_PHILOX              # the noise levels live in the per-env row
        elif sigma == 0.0:
            nz.mode = L.NOISE_NONE
        elif self.noise_kind == "philox":
            nz.mode = L.NOISE_PHILOX
        else:
            raise ValueError("noise_var != 0 needs noise='philox' or noise='table'")
        nz.offset = self._step_index
        return nz

    # ---- MR_Env.reset, MR_env.py:164-201 -----------------------------------------------------
    def reset(self, init=None, noise_var=1, a0=1, is_mismatched=False, mask=None, reset_cursor=True):
        """Reset all envs (or those with ``mask[i] != 0``).  ``init``: None (sample init_space on
        device), a (2,) position for every env, or an [N, 2] tensor.  With ``per_env_params`` the three simulator
        arguments may be scalars or [N] arrays (only the masked envs take the new values).  Returns obs [N, 5]."""
        if torch.cuda.current_device() != self._dev_index:
            with torch.cuda.device(self.device):
                return self.reset(init, noise_var, a0, is_mismatched, mask, reset_cursor)
        n = self.num_envs
        p = self.params
        rp, keep = None, []
        if self.per_env_params:
            def row(v, dt):
                if np.ndim(v) == 0 and not torch.is_tensor(v):
                    return None
                t = torch.as_tensor(v).to(device=self.device, dtype=dt).contiguous()
                if t.numel() != n:
                    raise ValueError(f"per-env reset arguments must have {n} entries")
                keep.append(t)
                return t
            ra, rs, rm = row(a0, torch.float64), row(noise_var, torch.float64), row(is_mismatched, torch.uint8)
            rp = L.ResetParams(_ptr(ra), _ptr(rs), _ptr(rm))
            # scalars go through the launch parameters (the kernel writes them into the rows of the envs it resets)
            a0 = 0.0 if ra is not None else a0
            noise_var = 0.0 if rs is not None else noise_var
            is_mismatched = False if rm is not None else is_mismatched
            if self.noise_kind == "none" and (rs is not None and float(rs.abs().max()) != 0.0 or float(noise_var) != 0.0):
                raise ValueError("noise_var != 0 needs noise='philox' or noise='table'")
        elif mask is not None and (float(noise_var) != p.noise_var or float(a0) != p.a0
                                   or bool(is_mismatched) != bool(p.is_mismatched)):
            raise ValueError("a masked reset cannot change noise_var / a0 / is_mismatched when they are launch scalars "
                             "(construct the env with per_env_params=True)")
        p.mism_at_reset = p.is_mismatched          # the integrator is built before the flag changes (:181 vs :183)
        p.noise_var = float(noise_var)
        p.a0 = float(a0)
        if self.per_env_params:
            p.is_mismatched = 1 if is_mismatched else 0       # the NEW flag for the envs being reset (old one: their row)
        init_t = None
        if init is not None:
            init_t = torch.as_tensor(np.asarray(init) if not torch.is_tensor(init) else init)
            init_t = init_t.to(device=self.device, dtype=self.dtype)
            if init_t.dim() == 1:
                init_t = init_t.reshape(1, 2).expand(n, 2)
            init_t = init_t.contiguous()
            if tuple(init_t.shape) != (n, 2):
                raise ValueError(f"init must be (2,) or ({n}, 2)")
        mask_t = None
        if mask is not None:
            mask_t = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).contiguous()
        nz = self._noise_for(p.noise_var)
        rc = self.lib.mr_env_reset_ex(C.byref(self._c_state), n, self._dt, C.byref(p), C.byref(nz), _ptr(init_t),
                                      _ptr(mask_t), 1 if reset_cursor else 0, C.byref(rp) if rp is not None else None,
                                      C.byref(self._c_out), self._stream())
        L.check(rc, "mr_env_reset")
        self.kernel_launches += 1
        self._step_index += 1
        p.is_mismatched = 1 if is_mismatched else 0
        p.mism_at_reset = p.is_mismatched
        return self.obs

    # ---- MR_Env.step, MR_env.py:70-98 -----------------------------------------------------------
    def step(self, actions):
        """actions: [N, 2] (f_t, alpha_t) device tensor.  Returns (obs [N,5], rew [N], done [N] uint8, info).
        The returned tensors are views of buffers that the next step overwrites."""
        if not torch.is_tensor(actions):
            return self.step_host(actions)
        n = self.num_envs
        a = actions
        if a.device != self.device or a.dtype is not self.dtype or not a.is_contiguous():
            a = a.to(device=self.device, dtype=self.dtype).contiguous()
        if a.numel() != 2 * n:
            raise ValueError(f"actions must be [{n}, 2]")
        nz = self._noise_for(self.params.noise_var)
        if torch.cuda.current_device() != self._dev_index:      # kernels launch on the runtime's current device
            with torch.cuda.device(self.device):
                return self.step(a)
        rc = self._call_step(self._b_state, n, self._dt, self._b_params, C.byref(nz), self._b_tt, a.data_ptr(),
                             self._b_out if self.want_state_prime else self._b_out_lean,
                             torch.cuda.current_stream(self.device).cuda_stream)
        if rc:
            L.check(rc, "mr_env_step")
        self.kernel_launches += 1
        self._step_index += 1
        return self._views

    # ---- K single-step launches as ONE CUDA graph ---------------------------------------------------------------
    def capture_steps(self, action_buffers, k_steps=None):
        """Capture ``k_steps`` launches of the single-step kernel into a CUDA graph (step k reads
        ``action_buffers[k % len(action_buffers)]``, each an [N, 2] device tensor whose CONTENTS may change between
        replays) and return a ``StepGraph``; ``graph.replay()`` then costs one graph launch instead of K kernel launches —
        what a rank of a sharded population needs once a launch is only a few microseconds of work.
        The Philox env-step index is read from a device counter (mr_noise.offset_dev) that every replay advances, so
        replays keep drawing fresh noise; results are identical to K ``step`` calls (tested)."""
        return StepGraph(self, action_buffers, k_steps)

    # A caller that steps with the SAME plain numpy action array every time (the usual control loop) should not pay a
    # 16 MB staging copy per step: the array's pages are page-locked in place once (cudaHostRegister) and the step kernel
    # reads them directly, like a pinned tensor.  At most `host_register_max` arrays are kept registered (oldest dropped).
    host_register_max = 16

    def _registered_view(self, a_np, hdt):
        """A torch view of the caller's numpy array after page-locking it in place, or None if it cannot be used as it
        is (wrong dtype, not C-contiguous, too small to be worth it, registration refused)."""
        want = np.float64 if hdt is torch.float64 else np.float32
        if a_np.dtype != want or not a_np.flags.c_contiguous or not a_np.flags.writeable or a_np.nbytes < (1 << 16):
            return None
        reg = self._pinned.setdefault("registered", {})
        key = (a_np.ctypes.data, a_np.nbytes)
        hit = reg.get(key)
        if hit is not None:
            return hit[0]
        with torch.cuda.device(self.device):
            if self.lib.mr_host_register(a_np.ctypes.data, a_np.nbytes) != 0:
                return None                       # e.g. the platform cannot address registered memory by its host pointer
        while len(reg) >= self.host_register_max:
            old_key = next(iter(reg))
            self.lib.mr_host_unregister(old_key[0])
            del reg[old_key]
        view = torch.from_numpy(a_np).view(-1, 2)
        reg[key] = (view, a_np)                   # keeps the array alive while it is registered
        return view

    def _pinned_buf(self, key, shape, dtype):
        b = self._pinned.get(key)
        if b is None or tuple(b.shape) != tuple(shape) or b.dtype != dtype:
            b = torch.empty(shape, dtype=dtype, pin_memory=True)
            self._pinned[key] = b
        return b

    def step_host(self, actions):
        """The reference-facing call with HOST buffers: actions [N, 2] (numpy array, or a pinned torch
        tensor which is used without a staging copy) in, numpy (obs [N,5], rew [N], done [N] bool) out.
        The call returns when the host arrays are filled; they are views of pinned buffers reused by the next call.
        ``host_mode = "direct"`` (default): the step kernel reads the actions from and writes the results to the pinned
        host buffers itself — the device-side obs / rew / done rows are NOT refreshed by this call (state, counters
        and state_prime are).  ``host_mode = "staged"``: copies through the device rows in pipelined chunks."""
        n = self.num_envs
        fast = self._pinned.get("fast")            # the same pinned action tensor as last time, direct mode: everything cached
        if fast is not None and actions is fast[0] and self.host_mode == "direct" \
                and actions.dtype == (self.host_io_dtype or self.dtype):
            _, io_ref, ret = fast
            if torch.cuda.current_device() != self._dev_index:
                with torch.cuda.device(self.device):
                    return self.step_host(actions)
            nz = self._noise_for(self.params.noise_var)
            rc = self.lib.mr_env_step_host(None, self._b_state, n, self._dt, self._b_params, C.byref(nz), self._b_tt, io_ref,
                                           self._b_out if self.want_state_prime else self._b_out_lean, 0,
                                           torch.cuda.current_stream(self.device).cuda_stream)
            if rc:
                L.check(rc, "mr_env_step_host")
            self.kernel_launches += 1
            self._step_index += 1
            return ret
        direct = self.host_mode == "direct"
        io32 = direct and self.dtype is torch.float64 and self.host_io_dtype is torch.float32
        hdt = torch.float32 if io32 else self.dtype          # dtype of the host action / observation buffers
        if torch.is_tensor(actions) and actions.device.type == "cpu" and actions.is_pinned() \
                and actions.dtype == hdt and actions.is_contiguous() and actions.numel() == 2 * n:
            a_pin = actions.view(n, 2)
            in_place = True
        else:
            in_place = False
            a_np = np.asarray(actions.numpy() if torch.is_tensor(actions) else actions)
            if a_np.size != 2 * n:
                raise ValueError(f"actions must be [{n}, 2]")
            a_pin = self._registered_view(a_np, hdt) if direct or self.host_mode == "staged_zc" else None
            if a_pin is None:                     # staging copy into pinned memory (dtype / layout / registration not usable)
                a_pin = self._pinned_buf("act", (n, 2), hdt)
                np.copyto(a_pin.numpy(), a_np.reshape(n, 2), casting="same_kind")
        a_dev = self._pinned.get("act_dev")
        zc_in = self.host_mode == "staged_zc"      # chunk kernels read the pinned actions themselves, results by copy engine
        if a_dev is None and not direct and not zc_in:
            a_dev = self._pinned["act_dev"] = torch.empty(n, 2, dtype=self.dtype, device=self.device)
        if zc_in:
            a_dev = None
        fresh = "obs" not in self._pinned or self._pinned["obs"].dtype != hdt
        o_pin = self._pinned_buf("obs", (5, self._np), hdt)           # same row stride as the device rows
        d_pin = self._pinned_buf("done", (n,), torch.uint8)
        # the constant reward of MR_env.py:89 is not sent at all in direct mode: one cached array of 10s
        const_rew = self.params.reward_mode == L.REWARD_CONST10
        if const_rew:
            r_np = self._pinned.get("rew_const")
            if r_np is None or r_np.dtype != o_pin.numpy().dtype:
                r_np = self._pinned["rew_const"] = np.full(n, 10.0, dtype=o_pin.numpy().dtype)
            r_ptr = 0
        else:
            r_pin = self._pinned_buf("rew", (n,), hdt)
            r_np, r_ptr = r_pin.numpy(), r_pin.data_ptr()
        if fresh:
            o_pin.zero_()          # goal rows 2, 3 are always 0 (MR_env.py:57): written once, never re-copied
        # one C call.  "direct": the step kernel reads / writes the pinned host buffers itself (zero-copy over PCIe);
        # "staged": H2D, kernel(s) and D2H pipelined over env chunks on the library's own streams
        chunks = 0 if direct else self._host_chunks(n)
        with torch.cuda.device(self.device):
            pl = self._pinned.get("pipeline")
            if pl is None and chunks:
                h = C.c_void_p()
                L.check(self.lib.mr_host_pipeline_create(8, C.byref(h)), "mr_host_pipeline_create")
                pl = self._pinned["pipeline"] = h
            io = L.HostStepIO(a_pin.data_ptr(), a_dev.data_ptr() if a_dev is not None else 0, o_pin.data_ptr(), r_ptr,
                              d_pin.data_ptr(), self._np, 0, 1 if io32 else 0)
            nz = self._noise_for(self.params.noise_var)
            rc = self.lib.mr_env_step_host(pl, self._b_state, n, self._dt, self._b_params, C.byref(nz), self._b_tt, C.byref(io),
                                           self._b_out if self.want_state_prime else self._b_out_lean, chunks,
                                           torch.cuda.current_stream(self.device).cuda_stream)
        L.check(rc, "mr_env_step_host")
        self.kernel_launches += max(chunks, 1)
        self._step_index += 1
        ret = (o_pin[:, :n].numpy().T, r_np, d_pin.numpy().view(np.bool_), {})
        if in_place and chunks == 0:       # a caller that reuses its pinned action tensor skips all of the above next time
            self._pinned["fast"] = (actions, C.byref(io), ret)
            self._pinned["fast_io"] = io           # keep the struct alive
        return ret

    # Host-buffer step strategy.  Measured at 2^20 envs (fp64, sigma = 1): staged 1 / 2 / 4 / 8 chunks 1.01 / 0.91 / 0.91 /
    # 0.99 ms (each of the 5 D2H pieces per chunk costs a few us of DMA set-up); direct 0.82 ms.  Round 2, constant reward
    # not sent: direct 0.66-0.68 ms; staged with ONE 2-D copy for the x, y rows 0.86 / 0.73 / 0.75 ms (1 / 2 / 4 chunks);
    # "staged_zc" (chunk kernels read the pinned actions themselves, results by copy engine) 0.83-0.88 ms with 2-8 chunks
    # (gpurun_out/e2e_zc.log -> profiles/r02_e2e_host_modes.txt) — direct stays the default.  Tried and dropped: a
    # hybrid (copy-engine H2D of the actions in chunks + kernel writing straight to the host) 0.89 / 0.93 / 0.97 ms with
    # 2 / 4 / 8 chunks — the smaller launches lose more than the DMA read gains; and a "streamed" variant (ONE kernel whose
    # loader waits on per-chunk arrival flags while the copy engine delivers the actions) 0.88 / 0.91 / 1.03 ms with
    # 4 / 8 / 16 chunks: correct, but DMA reads + SM writes to the host interfere more than SM reads + SM writes do.
    host_mode = "direct"
    host_chunks = 2
    # dtype of the HOST action / observation buffers of step_host in direct mode: None = the storage dtype;
    # torch.float32 with float64 storage = float32 on the wire (north_star's 1e-4 tier for the transferred values, half
    # the bytes over PCIe), state and all decisions stay float64 on the device
    host_io_dtype = None

    def _host_chunks(self, n, min_chunk=1 << 16):
        """Number of env ranges for the staged host step; small batches and table noise stay in one piece."""
        if self.noise_kind == "table":
            return 1
        return max(1, min(int(self.host_chunks), n // min_chunk))

    def __del__(self):
        try:
            pl = self._pinned.get("pipeline")
            if pl is not None:
                self.lib.mr_host_pipeline_destroy(pl)
                self._pinned["pipeline"] = None
            for key in list(self._pinned.get("registered", {})):
                self.lib.mr_host_unregister(key[0])
            self._pinned["registered"] = {}
        except Exception:
            pass

    def _c_state_ptr(self, field, lo):
        t = {"x": self._state[0], "y": self._state[1], "fx": self._state[2], "fy": self._state[3], "h": self._state[4],
             "counter": self._counter, "cursor": self._cursor, "status": self._status}[field]
        return t.data_ptr() + lo * t.element_size()

    # ---- fused K-step rollout: utils.run_sim (utils.py:43-61) / the DDPG acting loop --------------
    def rollout(self, actions=None, k_steps=None, policy=None, record=False, record_state_prime=False,
                record_done=False, accumulate_stats=True, record_episodes=False, reset_init=None, ddpg_collect=None,
                ddpg_population=None):
        """K env steps in ONE launch with the state held in registers.

        actions : [K, N, 2] per-env actions, or [K, 2] / [K, >=2] one action row for every env
                  (what utils.run_sim does), or None with ``policy``:
        policy  : "random" -> U[0,20) x U[0,2pi) generated in-kernel (Philox);
                  a packed float32 actor tensor (see actor.pack_actor) -> DDPG actor in the loop;
                  a ``LearningModule.tracking_policy(ref, gain)`` -> GP-corrected heading control in the loop
                  (``k_steps`` defaults to the K rows of its ``ref``; per-env parameter rows are not supported).
        record_episodes : per-episode logging on the device (what MRExperiment.new_iter / new_transition record,
                  MR_data.py:27-57): adds ``actions_traj`` [K,N,2], ``rew_traj`` [K,N], ``reset_xy`` [K,2,N] (start of the
                  episode that follows a terminal step, with auto_reset), ``episode`` / ``step`` [K,N] int32 keys and
                  ``start_xy`` [N,2] (positions before the first step); ``recording.experiment_from_rollout`` turns them into
                  the reference's pickle layout.  Episode ordinals continue across launches (``self._episode_counter``).
        reset_init : [E, N, 2] start positions for the auto resets (episode e of env i restarts at reset_init[(e-1) % E, i])
                  instead of sampling init_space.
        ddpg_collect : with an actor ``policy``, the ``_lib.DDPGCollect`` of ``ddpg.collect``: the launch also adds OU
                  noise to the actions and writes every transition into the replay ring (mr_env_rollout_ddpg_collect).
        ddpg_population : with ``ddpg_collect``, ``(members, stats)`` of ``ddpg.collect_population``: ``policy`` is the
                  stacked actors [members, count], the ring arrays are stacked per member, and the statistics accumulate
                  into ``stats`` [members, 8] instead of the env's vector (mr_env_rollout_ddpg_collect_population).
        Returns dict(obs, rew, done[, xy [K,2,N], state_prime [K,2,N], done_traj [K,N]]).
        """
        if torch.cuda.current_device() != self._dev_index:
            with torch.cuda.device(self.device):
                return self.rollout(actions, k_steps, policy, record, record_state_prime, record_done, accumulate_stats,
                                    record_episodes, reset_init, ddpg_collect, ddpg_population)
        n = self.num_envs
        io = L.RolloutIO()
        keep = []
        gp_pol = None
        if actions is not None:
            a = torch.as_tensor(actions) if not torch.is_tensor(actions) else actions
            a = a.to(device=self.device, dtype=self.dtype)
            if a.dim() == 2:
                a = a[:, :2].contiguous()
                io.action_source = L.ACTIONS_BROADCAST
            elif a.dim() == 3 and a.shape[1] == n and a.shape[2] == 2:
                a = a.contiguous()
                io.action_source = L.ACTIONS_TENSOR
            else:
                raise ValueError(f"actions must be [K, {n}, 2] or [K, 2]")
            k = a.shape[0]
            io.actions = a.data_ptr()
            keep.append(a)
        elif isinstance(policy, str) and policy == "random":
            io.action_source = L.ACTIONS_PHILOX
            k = int(k_steps)
        elif torch.is_tensor(policy):
            w = policy.to(device=self.device, dtype=torch.float32).contiguous()
            members = ddpg_population[0] if ddpg_population is not None else 1
            if w.numel() != members * self.lib.mr_actor_param_count():
                raise ValueError("actor tensor has the wrong number of parameters (use actor.pack_actor)")
            io.action_source = L.ACTIONS_ACTOR
            io.actor = w.data_ptr()
            keep.append(w)
            k = int(k_steps)
        elif isinstance(policy, HeadingTrackingPolicy):
            k = policy.k_steps if k_steps is None else int(k_steps)
            if k > policy.k_steps:
                raise ValueError(f"k_steps = {k} exceeds the {policy.k_steps} rows of the policy's ref")
            io.action_source = L.ACTIONS_GP_HEADING
            gp_pol, tensors = policy.c_policy(self.device)
            keep.extend(tensors)
        else:
            raise ValueError("give actions or policy")
        if ddpg_collect is not None and io.action_source != L.ACTIONS_ACTOR:
            raise ValueError("ddpg_collect needs an actor policy")
        if ddpg_population is not None and ddpg_collect is None:
            raise ValueError("ddpg_population needs ddpg_collect")
        io.k_steps = k
        res = {}
        if record_episodes:
            record = record_done = True
            res["start_xy"] = self.last_pos.clone()
            res["actions_traj"] = torch.empty(k, n, 2, dtype=self.dtype, device=self.device)
            res["rew_traj"] = torch.empty(k, n, dtype=self.dtype, device=self.device)
            res["reset_xy"] = torch.zeros(k, 2, n, dtype=self.dtype, device=self.device)
            res["episode"] = torch.empty(k, n, dtype=torch.int32, device=self.device)
            res["step"] = torch.empty(k, n, dtype=torch.int32, device=self.device)
            if getattr(self, "_episode_counter", None) is None:
                self._episode_counter = torch.zeros(n, dtype=torch.int32, device=self.device)
            io.traj_actions, io.traj_rew = res["actions_traj"].data_ptr(), res["rew_traj"].data_ptr()
            io.traj_reset_xy = res["reset_xy"].data_ptr()
            io.traj_episode, io.traj_step = res["episode"].data_ptr(), res["step"].data_ptr()
            io.episode_counter = self._episode_counter.data_ptr()
        if reset_init is not None:
            ri = torch.as_tensor(reset_init).to(device=self.device, dtype=self.dtype).contiguous()
            if ri.dim() != 3 or ri.shape[1] != n or ri.shape[2] != 2:
                raise ValueError(f"reset_init must be [E, {n}, 2]")
            if getattr(self, "_episode_counter", None) is None:
                self._episode_counter = torch.zeros(n, dtype=torch.int32, device=self.device)
            io.episode_counter = self._episode_counter.data_ptr()
            io.reset_init, io.reset_init_len = ri.data_ptr(), ri.shape[0]
            keep.append(ri)
        if record:
            res["xy"] = torch.empty(k, 2, n, dtype=self.dtype, device=self.device)
            io.traj_xy = res["xy"].data_ptr()
        if record_state_prime:
            res["state_prime"] = torch.empty(k, 2, n, dtype=self.dtype, device=self.device)
            io.traj_state_prime = res["state_prime"].data_ptr()
        if record_done:
            res["done_traj"] = torch.empty(k, n, dtype=torch.uint8, device=self.device)
            io.traj_done = res["done_traj"].data_ptr()
        if accumulate_stats:
            io.stats = self._stats.data_ptr() if ddpg_population is None else ddpg_population[1].data_ptr()
        nz = self._noise_for(self.params.noise_var)
        if gp_pol is not None:
            rc = self.lib.mr_env_rollout_gp_heading(C.byref(self._c_state), n, self._dt, C.byref(self.params), C.byref(nz),
                                                    C.byref(self._c_tt), C.byref(io), C.byref(gp_pol), C.byref(self._c_out),
                                                    self._stream())
            L.check(rc, "mr_env_rollout_gp_heading")
        elif ddpg_population is not None:
            rc = self.lib.mr_env_rollout_ddpg_collect_population(C.byref(self._c_state), n, self._dt, C.byref(self.params),
                                                                 C.byref(nz), C.byref(self._c_tt), C.byref(io),
                                                                 C.byref(ddpg_collect), int(ddpg_population[0]),
                                                                 C.byref(self._c_out), self._stream())
            L.check(rc, "mr_env_rollout_ddpg_collect_population")
        elif ddpg_collect is not None:
            rc = self.lib.mr_env_rollout_ddpg_collect(C.byref(self._c_state), n, self._dt, C.byref(self.params), C.byref(nz),
                                                      C.byref(self._c_tt), C.byref(io), C.byref(ddpg_collect),
                                                      C.byref(self._c_out), self._stream())
            L.check(rc, "mr_env_rollout_ddpg_collect")
        else:
            rc = self.lib.mr_env_rollout(C.byref(self._c_state), n, self._dt, C.byref(self.params), C.byref(nz),
                                         C.byref(self._c_tt), C.byref(io), C.byref(self._c_out), self._stream())
            L.check(rc, "mr_env_rollout")
        self.kernel_launches += 1
        self._step_index += k
        res.update(obs=self.obs, rew=self._rew[:n], done=self._done[:n])
        return res

    # ---- episode statistics (NCCL all-reduce is the only collective of the path) -------------------
    def reset_stats(self):
        self._stats.zero_()

    def allreduce_stats(self, group=None):
        """Sum the episode-statistics vector over all ranks (torch.distributed, NCCL on GPUs).
        Returns the global statistics; the local accumulators are left untouched."""
        from .dist import merge_stats
        return merge_stats(self._stats, group)

    def stats_dict(self):
        v = self._stats.tolist()
        d = dict(zip(L.STAT_NAMES, v))
        d["mean_episode_length"] = d["sum_length"] / d["episodes"] if d["episodes"] else math.nan
        return d

    # ---- failure reporting: the reference raises from scipy; kernels set sticky flags ---------------
    def check_status(self):
        raise_for_status(self._status[:self.num_envs])

    # ---- checkpoint / resume ----------------------------------------------------------------------------
    def state_dict(self):
        p = self.params
        return {
            "state": self._state.clone(), "counter": self._counter.clone(), "cursor": self._cursor.clone(),
            "status": self._status.clone(), "stats": self._stats.clone(), "step_index": self._step_index,
            "params": {"a0": p.a0, "noise_var": p.noise_var, "is_mismatched": int(p.is_mismatched),
                       "max_timesteps": int(p.max_timesteps), "min_dist2goal": float(p.min_dist2goal),
                       "bound_xy": float(p.bound_xy), "bound_d": float(p.bound_d),
                       "init_low": [p.init_low[0], p.init_low[1]], "init_high": [p.init_high[0], p.init_high[1]],
                       "action_high": [p.action_high[0], p.action_high[1]],
                       "auto_reset": int(p.auto_reset), "reward_mode": int(p.reward_mode)},
            "seed": int(self._c_noise.seed), "env_base": int(self._c_noise.env_base),
        }

    def load_state_dict(self, sd):
        self._state.copy_(sd["state"]); self._counter.copy_(sd["counter"]); self._cursor.copy_(sd["cursor"])
        self._status.copy_(sd["status"]); self._stats.copy_(sd["stats"])
        self._step_index = int(sd["step_index"])
        self.params.a0 = sd["params"]["a0"]; self.params.noise_var = sd["params"]["noise_var"]
        self.params.is_mismatched = self.params.mism_at_reset = sd["params"]["is_mismatched"]
        q = sd["params"]
        if "max_timesteps" in q:                      # older checkpoints carry only the three simulator parameters
            self.max_timesteps, self.min_dist2goal = q["max_timesteps"], q["min_dist2goal"]
            self.init_space = Box(low=np.array(q["init_low"]), high=np.array(q["init_high"]))
            self.action_space = Box(low=np.array([0, 0]), high=np.array(q["action_high"]))
            b, bd = q["bound_xy"], q["bound_d"]
            self.observation_space = Box(low=np.array([-b, -b, -b, -b, 0]), high=np.array([b, b, b, b, bd]))
            self.params.auto_reset, self.params.reward_mode = int(q["auto_reset"]), int(q["reward_mode"])
        self._c_noise.seed = sd["seed"]; self._c_noise.env_base = sd["env_base"]

    # ---- no-op hooks kept for drop-in compatibility (MR_env.py:203-229) --------------------------------
    def render(self, mode="human"):
        return None

    def close(self):
        return None


class StepGraph:
    """K MR_Env.step launches of a VecMREnv captured in one CUDA graph (see VecMREnv.capture_steps)."""

    def __init__(self, env, action_buffers, k_steps=None):
        bufs = list(action_buffers)
        n = env.num_envs
        for a in bufs:
            if not (torch.is_tensor(a) and a.device == env.device and a.dtype is env.dtype and a.is_contiguous()
                    and a.numel() == 2 * n):
                raise ValueError(f"action buffers must be contiguous [{n}, 2] {env.dtype} tensors on {env.device}")
        self.env, self.buffers = env, bufs
        self.k_steps = int(k_steps if k_steps is not None else len(bufs))
        self._ctr = torch.zeros(1, dtype=torch.int64, device=env.device)      # mr_noise.offset_dev
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.device(env.device):
            env.step(bufs[0])                       # first-launch set-up (function attributes) must not be captured
            torch.cuda.synchronize(env.device)
            nz = env._noise_for(env.params.noise_var)
            out = env._b_out if env.want_state_prime else env._b_out_lean
            with torch.cuda.graph(self.graph):
                stream = torch.cuda.current_stream(env.device).cuda_stream
                nz.offset_dev = self._ctr.data_ptr()
                try:
                    for k in range(self.k_steps):
                        nz.offset = k
                        rc = env._call_step(env._b_state, n, env._dt, env._b_params, C.byref(nz), env._b_tt,
                                            bufs[k % len(bufs)].data_ptr(), out, stream)
                        if rc:
                            L.check(rc, "mr_env_step (graph capture)")
                finally:
                    nz.offset_dev = None
        # the launch parameters are baked into the captured kernel nodes
        self._baked = self._param_key()

    def _param_key(self):
        p = self.env.params
        return (p.a0, p.noise_var, p.is_mismatched, p.auto_reset, p.max_timesteps, p.min_dist2goal, p.reward_mode,
                p.bound_xy, p.bound_d, tuple(p.init_low), tuple(p.init_high), self.env.want_state_prime)

    def replay(self):
        """Run the K captured steps; returns the views (obs, rew, done, info) after the last one."""
        env = self.env
        if self._baked != self._param_key():
            raise RuntimeError("env parameters changed since the graph was captured: capture again")
        with torch.cuda.device(env.device):
            rc = env.lib.mr_counter_set(self._ctr.data_ptr(), env._step_index, env._stream())
            if rc:
                L.check(rc, "mr_counter_set")
            self.graph.replay()
        env._step_index += self.k_steps
        env.kernel_launches += self.k_steps + 1
        return env._views


from .dist import shard_range  # noqa: E402,F401  (re-exported)
