"""Batched T-rex simulator: thin Python host over the C ABI, torch tensors as zero-copy buffers.

PyTorch is plumbing here (device memory, streams); all arithmetic happens in
``libtrex_b200.so`` (``csrc/trex_core.h``).  Requires a CUDA device: there is no CPU path.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native
from .model_compiler import CompiledModel, load_builtin


class TrexBatchSim:
    """``num_envs`` independent T-rex environments on one GPU, one warp each.

    Buffers are one row per environment: ``action [N,25]``, ``obs [N,75]``, ``reward [N]``,
    ``done [N]`` (uint8), ``state [N,160]`` (layout: ``include/trex_b200.h``).  Joint order
    of action/obs = revolute joints sorted by name (trex_robot.py:311-314).
    """

    def __init__(self, num_envs: int, device: int | str | torch.device = 0, model: CompiledModel | None = None,
                 num_substeps: int = 5, distance_weight: float = 1.0, energy_weight: float = 0.005,
                 drift_weight: float = 0.002, max_episode_steps: int = 0, contacts: bool = True,
                 seed: int = 0, warps_per_block: int | None = None, reset_mode: int = 0, env_offset: int = 0,
                 deferred_solve: bool = True, defer_contacts: bool = True, heavy_solver: bool = True,
                 heavy_share_div: int = 0, pipelines: int = 0, heavy_memory: int = 0, chunk_envs: int = 0, contact_memory: int = 0,
                 env_params: bool = False, external_forces: bool = False, actuation: str = "position"):
        """``actuation``: ``"position"`` (default: an action is a motor target, clipped to the joint limits) or ``"torque"``
        (joint torque control: an action is the joint torque in N m, clipped to the model's ``motor_max_torque`` -- or an
        ``env_params`` row's element 29 -- and applied in every physics substep; the motors have no gain or strength; the
        observation's torque block and the energy term report the clipped command).  See ``include/trex_b200.h``."""
        if actuation not in _native.ACTUATION:
            raise ValueError("actuation must be 'position' or 'torque', not %r" % (actuation,))
        if not torch.cuda.is_available():
            raise RuntimeError("trex_gym_b200 needs a CUDA device (no CPU fallback)")
        dev = torch.device(device if not isinstance(device, int) else "cuda:%d" % device)
        if dev.type != "cuda":
            raise ValueError("device must be a CUDA device")
        self.device = dev
        self.num_envs = int(num_envs)
        self.env_offset = int(env_offset)  # global id of environment 0 of this shard
        self.seed = int(seed)
        self.model = model if model is not None else load_builtin()
        self._L = _native.lib()
        cfg = _native.TrexConfig()
        cfg.num_substeps = int(num_substeps)
        cfg.distance_weight = float(distance_weight)
        cfg.energy_weight = float(energy_weight)
        cfg.drift_weight = float(drift_weight)
        cfg.max_episode_steps = int(max_episode_steps)
        cfg.enable_contacts = int(bool(contacts))
        cfg.reset_mode = int(reset_mode)
        cfg.env_offset = int(env_offset)
        cfg.seed = int(seed) & 0xFFFFFFFF
        # solver placement (diagnostics; include/trex_b200.h TREX_SOLVE_*)
        cfg.solver_placement = ((_native.SOLVE_DEFAULT if heavy_solver else _native.SOLVE_NO_HEAVY) if defer_contacts
                                else _native.SOLVE_FREE_ONLY) if deferred_solve else _native.SOLVE_FRONT
        cfg.heavy_share_div = int(heavy_share_div)
        cfg.warps_per_block = int(warps_per_block or 0)
        cfg.heavy_memory = int(heavy_memory)  # _native.HEAVY_BOTH / HEAVY_SHARED / HEAVY_TENSOR: where solve2 keeps its Delassus matrices
        cfg.pipelines = int(pipelines)  # 0 = default; independent groups of environments on separate streams
        cfg.contact_memory = int(contact_memory)  # _native.CONTACT_TENSOR (default) / CONTACT_SHARED: where solve4 keeps its contact stash
        cfg.chunk_envs = int(chunk_envs)  # 0 = default; L2-resident work records (include/trex_b200.h), -1 = off
        cfg.env_params = int(bool(env_params))  # per-environment dynamics parameters (set_env_params)
        self.env_params = bool(env_params)
        cfg.external_forces = int(bool(external_forces))  # per-environment external wrenches (set_external_forces)
        self.external_forces = bool(external_forces)
        cfg.actuation = _native.ACTUATION[actuation]
        self.actuation = actuation
        blob = self.model.blob()
        h = ctypes.c_void_p()
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        _native.check(self._L.trex_create(blob, len(blob), self.num_envs, idx, ctypes.byref(cfg), ctypes.byref(h)),
                      "trex_create")
        self._h = h
        self.num_substeps = int(num_substeps)
        with torch.cuda.device(dev):
            self.obs = torch.zeros(self.num_envs, _native.OBS_DIM, device=dev, dtype=torch.float32)
            self.reward = torch.zeros(self.num_envs, device=dev, dtype=torch.float32)
            self.done = torch.zeros(self.num_envs, device=dev, dtype=torch.uint8)
            # motor position targets last set through TrexRobot.set_actions (trex_robot.py:413-422): the counterpart of
            # pybullet's motor state, which persists between setJointMotorControlArray calls; step(None) consumes it
            self.targets = torch.zeros(self.num_envs, _native.NUM_JOINTS, device=dev, dtype=torch.float32)
        lo = np.zeros(_native.NUM_JOINTS, np.float32)
        hi = np.zeros(_native.NUM_JOINTS, np.float32)
        _native.check(self._L.trex_get_joint_limits(self._h, lo.ctypes.data, hi.ctypes.data), "trex_get_joint_limits")
        self.action_low, self.action_high = lo, hi  # the joint limits (the observation space uses them in both modes)

    def action_limits(self) -> tuple[np.ndarray, np.ndarray]:
        """(low, high) [25] of the action space, name-sorted: the joint limits in position mode, -/+ the model's
        ``motor_max_torque`` in torque mode."""
        lo = np.zeros(_native.NUM_JOINTS, np.float32)
        hi = np.zeros(_native.NUM_JOINTS, np.float32)
        _native.check(self._L.trex_get_action_limits(self._h, lo.ctypes.data, hi.ctypes.data), "trex_get_action_limits")
        return lo, hi

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._L.trex_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check_tensor(self, t: torch.Tensor, shape, dtype, name):
        if not isinstance(t, torch.Tensor) or t.device != self.device or t.dtype != dtype or tuple(t.shape) != tuple(shape) \
                or not t.is_contiguous():
            raise ValueError("%s must be a contiguous %s tensor of shape %s on %s" % (name, dtype, tuple(shape), self.device))

    # -- the hot path -------------------------------------------------------------------------
    def reset(self, mask: torch.Tensor | None = None) -> torch.Tensor:
        """``TrexBulletEnv.reset`` (trex_env.py:98-122) for all (or the masked) environments."""
        mp = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if mask.shape != (self.num_envs,):
                raise ValueError("mask must have shape (num_envs,)")
            mp = ctypes.c_void_p(mask.data_ptr())
        _native.check(self._L.trex_reset(self._h, mp, ctypes.c_void_p(self.obs.data_ptr()), self._stream()), "trex_reset")
        return self.obs

    def step(self, action: torch.Tensor | None = None):
        """``TrexBulletEnv.step`` (trex_env.py:128-154) for every environment; returns views of the
        simulator-owned ``obs``, ``reward``, ``done`` tensors (overwritten by the next call).
        ``action=None`` steps with the targets last written through ``TrexRobot.set_actions`` (``self.targets``)."""
        if action is None:
            action = self.targets
        self._check_tensor(action, (self.num_envs, _native.NUM_JOINTS), torch.float32, "action")
        _native.check(
            self._L.trex_step(self._h, ctypes.c_void_p(action.data_ptr()), ctypes.c_void_p(self.obs.data_ptr()),
                              ctypes.c_void_p(self.reward.data_ptr()), ctypes.c_void_p(self.done.data_ptr()), self._stream()),
            "trex_step")
        return self.obs, self.reward, self.done

    # -- CUDA-graph replay of the step (small batches are launch bound: 26 launches + events per group and env step) --------
    def capture_graph(self):
        """Capture one ``trex_step`` (every kernel, fork / join event and counter reset of the step) into a CUDA graph with
        simulator-owned static buffers; afterwards ``step_graph(action)`` copies the action in and replays the graph.  The step
        is capturable because the library forks from and joins back into the caller's stream by events only
        (``include/trex_b200.h``).  State is untouched by the capture.  Results are bit-identical to ``step``."""
        if getattr(self, "_graph", None) is not None:
            return
        self._g_action = torch.zeros(self.num_envs, _native.NUM_JOINTS, device=self.device, dtype=torch.float32)
        torch.cuda.synchronize(self.device)
        side = torch.cuda.Stream(device=self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            pre = self.get_state().clone()
            self.step(self._g_action)          # warm-up on the capture stream (kernel attributes get configured here)
            self.set_state(pre)
            side.synchronize()
            with torch.cuda.graph(g, stream=side):
                self.step(self._g_action)
        torch.cuda.synchronize(self.device)
        self.set_state(pre)                    # (capture does not execute, the warm-up step is undone)
        torch.cuda.synchronize(self.device)
        self._graph = g

    def step_graph(self, action: torch.Tensor):
        """``step`` through the captured graph: one device-to-device copy of the actions + one graph launch."""
        if getattr(self, "_graph", None) is None:
            self.capture_graph()
        self._check_tensor(action, (self.num_envs, _native.NUM_JOINTS), torch.float32, "action")
        self._g_action.copy_(action, non_blocking=True)
        self._graph.replay()
        return self.obs, self.reward, self.done

    def step_into(self, action: torch.Tensor, obs: torch.Tensor, reward: torch.Tensor, done: torch.Tensor):
        """Step writing into caller-provided buffers (e.g. slices of a rollout buffer)."""
        self._check_tensor(action, (self.num_envs, _native.NUM_JOINTS), torch.float32, "action")
        self._check_tensor(obs, (self.num_envs, _native.OBS_DIM), torch.float32, "obs")
        self._check_tensor(reward, (self.num_envs,), torch.float32, "reward")
        self._check_tensor(done, (self.num_envs,), torch.uint8, "done")
        _native.check(
            self._L.trex_step(self._h, ctypes.c_void_p(action.data_ptr()), ctypes.c_void_p(obs.data_ptr()),
                              ctypes.c_void_p(reward.data_ptr()), ctypes.c_void_p(done.data_ptr()), self._stream()),
            "trex_step")

    def step_host(self, action: np.ndarray | torch.Tensor, obs=None, reward=None, done=None):
        """Host-buffer step (numpy or pinned CPU tensors in, numpy / CPU tensors out): H2D copy of the
        actions, step, D2H copy of obs/reward/done, synchronise.  This is the end-to-end call."""
        def ptr(x):
            return x.data_ptr() if isinstance(x, torch.Tensor) else x.ctypes.data
        if isinstance(action, np.ndarray):
            action = np.ascontiguousarray(action, np.float32)
        if tuple(action.shape) != (self.num_envs, _native.NUM_JOINTS):
            raise ValueError("action must have shape (num_envs, 25)")
        if obs is None:
            obs = np.empty((self.num_envs, _native.OBS_DIM), np.float32)
        if reward is None:
            reward = np.empty(self.num_envs, np.float32)
        if done is None:
            done = np.empty(self.num_envs, np.uint8)
        _native.check(self._L.trex_step_host(self._h, ctypes.c_void_p(ptr(action)), ctypes.c_void_p(ptr(obs)),
                                             ctypes.c_void_p(ptr(reward)), ctypes.c_void_p(ptr(done))), "trex_step_host")
        return obs, reward, done

    def step_host_async(self, action, obs, reward, done):
        """``step_host`` as a depth-1 pipeline (``trex_step_host_async``): when call k returns, the outputs of call k-1
        are complete; the copies of call k overlap call k+1.  Alternate between two sets of caller-owned (ideally pinned)
        arrays and finish with ``host_wait()``."""
        def ptr(x):
            return x.data_ptr() if isinstance(x, torch.Tensor) else x.ctypes.data
        for x, shape in ((action, (self.num_envs, _native.NUM_JOINTS)), (obs, (self.num_envs, _native.OBS_DIM)),
                         (reward, (self.num_envs,)), (done, (self.num_envs,))):
            if tuple(x.shape) != shape:
                raise ValueError("step_host_async: expected shape %s" % (shape,))
        _native.check(self._L.trex_step_host_async(self._h, ctypes.c_void_p(ptr(action)), ctypes.c_void_p(ptr(obs)),
                                                   ctypes.c_void_p(ptr(reward)), ctypes.c_void_p(ptr(done))), "trex_step_host_async")

    def host_wait(self) -> None:
        _native.check(self._L.trex_host_wait(self._h), "trex_host_wait")

    def reset_host(self) -> np.ndarray:
        obs = np.empty((self.num_envs, _native.OBS_DIM), np.float32)
        _native.check(self._L.trex_reset_host(self._h, ctypes.c_void_p(obs.ctypes.data)), "trex_reset_host")
        return obs

    # -- per-environment dynamics parameters (env_params=True) ------------------------------------------------
    # A row has 32 floats (include/trex_b200.h): [0:25] mass scale of the body of joint k (pybullet link order), [25] of the
    # base, [26] friction, [27] kp, [28] kd, [29] max torque (N m), [30] impulse bound (derived), [31] reserved.
    _ROW_FIELDS = {"friction": 26, "kp": 27, "kd": 28, "max_torque": 29}

    def _body_index(self, name) -> int:
        """Row element of a body named by its joint (``meta["body_joint_names"]``) or ``"base"``."""
        if name == "base":
            return 25
        names = self.model.meta["body_joint_names"]
        if name not in names[1:]:
            raise ValueError("unknown body %r: use 'base' or a name of meta['body_joint_names']" % (name,))
        return names.index(name) - 1

    def default_env_params(self) -> torch.Tensor:
        """The row that reproduces the model's own constants ([32] on the CPU): unit mass scales, the model's friction,
        motor gains and torque."""
        p = self.model.meta["params"]
        row = np.zeros(_native.ENV_PARAM_DIM, np.float32)
        row[:26] = 1.0
        row[26], row[27], row[28], row[29] = p["friction"], p["motor_kp"], p["motor_kd"], p["motor_max_torque"]
        row[30] = np.float32(p["motor_max_torque"] * (p["time_step"] / self.num_substeps))
        return torch.from_numpy(row)

    def _row(self, spec, base) -> np.ndarray:
        """A [32] row from an array, or from names (``mass_scale``: a scalar or {body: scale}; ``friction``, ``kp``,
        ``kd``, ``max_torque``) applied on top of ``base``."""
        if not isinstance(spec, dict):
            row = np.asarray(spec.cpu() if isinstance(spec, torch.Tensor) else spec, np.float32).reshape(-1)
            if row.shape != (_native.ENV_PARAM_DIM,):
                raise ValueError("a parameter row has %d elements" % _native.ENV_PARAM_DIM)
            return row.copy()
        row = np.array(base, np.float32)
        for k, v in spec.items():
            if k == "mass_scale":
                if isinstance(v, dict):
                    for body, sc in v.items():
                        row[self._body_index(body)] = sc
                else:
                    row[:26] = v
            elif k in self._ROW_FIELDS:
                row[self._ROW_FIELDS[k]] = v
            else:
                raise ValueError("unknown parameter %r (mass_scale, friction, kp, kd, max_torque)" % (k,))
        return row

    def _need_env_params(self):
        if not self.env_params:
            raise ValueError("the simulator was created with env_params=False")

    def get_env_params(self) -> torch.Tensor:
        """[N,32] copy of every environment's parameter row (element 30 as the library derived it)."""
        self._need_env_params()
        t = torch.empty(self.num_envs, _native.ENV_PARAM_DIM, device=self.device, dtype=torch.float32)
        _native.check(self._L.trex_get_env_params(self._h, ctypes.c_void_p(t.data_ptr()), self._stream()), "trex_get_env_params")
        return t

    def set_env_params(self, t, mask: torch.Tensor | None = None) -> None:
        """Set the rows of all (or the masked) environments: ``t`` is an [N,32] tensor, one [32] row for every
        environment, or a dict of names (see ``_row``) applied to the default row.  Element 30 is derived by the library."""
        self._need_env_params()
        if isinstance(t, torch.Tensor) and t.dim() == 2:
            rows = t.to(device=self.device, dtype=torch.float32).contiguous()
        else:
            rows = torch.from_numpy(self._row(t, self.default_env_params().numpy())).to(self.device).repeat(self.num_envs, 1)
        self._check_tensor(rows, (self.num_envs, _native.ENV_PARAM_DIM), torch.float32, "env params")
        if not bool(torch.isfinite(rows).all()):
            raise ValueError("env params must be finite")
        if bool((rows[:, :26] <= 0).any()) or bool((rows[:, 26:30] < 0).any()):
            raise ValueError("mass scales must be > 0; friction, kp, kd and max_torque >= 0")
        mp = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if mask.shape != (self.num_envs,):
                raise ValueError("mask must have shape (num_envs,)")
            mp = ctypes.c_void_p(mask.data_ptr())
        _native.check(self._L.trex_set_env_params(self._h, ctypes.c_void_p(rows.data_ptr()), mp, self._stream()),
                      "trex_set_env_params")
        self._env_param_src = (rows, mask)  # kept alive until the stream has consumed them

    def set_env_param_ranges(self, low=None, high=None) -> None:
        """Randomizer: from now on every reset of an environment (``reset``, masked too, and the auto-reset) draws its row
        uniformly in [low, high] (Philox keyed by the seed, global environment id and episode).  ``low`` / ``high``: [32]
        rows, or dicts of names (see ``_row``) applied to the default row; elements 30-31 are ignored.  ``None, None``
        turns the randomizer off."""
        self._need_env_params()
        if low is None and high is None:
            _native.check(self._L.trex_set_env_param_ranges(self._h, None, None), "trex_set_env_param_ranges")
            return
        base = self.default_env_params().numpy()
        lo, hi = self._row(low, base), self._row(high, base)
        lo[30:] = 0.0
        hi[30:] = 0.0
        _native.check(self._L.trex_set_env_param_ranges(self._h, lo.ctypes.data, hi.ctypes.data), "trex_set_env_param_ranges")

    # -- external forces and torques (external_forces=True) ------------------------------------------------------
    # A wrench is [fx fy fz tx ty tz] in the world frame on one of 26 bodies (body k < 25: the body of joint k in pybullet link
    # order, 25: the base); the force acts at the body's centre of mass (body_com), the torque is free.  Unlike pybullet's
    # applyExternalForce, which lasts one stepSimulation, the wrenches stay until set again; they act in every physics
    # substep of a step, never in the physics step of a reset, and survive resets.

    def _need_external_forces(self):
        if not self.external_forces:
            raise ValueError("the simulator was created with external_forces=False")

    def _mask_ptr(self, mask):
        if mask is None:
            return None, None
        mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        if mask.shape != (self.num_envs,):
            raise ValueError("mask must have shape (num_envs,)")
        return mask, ctypes.c_void_p(mask.data_ptr())

    def body_com(self) -> np.ndarray:
        """[26, 3] centre of mass of every body in its own frame (the point the force of a wrench acts at), float32, in
        wrench-body order.  A torque about another point p of body k is the torque at the COM plus (p - com) x F in world
        coordinates."""
        from .model_blob import unpack
        sec = unpack(self.model.blob())
        mass, mc = sec["mb_mass"], sec["mb_mc"].reshape(-1, 3)
        bodies = [k + 1 for k in range(_native.EXT_BODIES - 1)] + [0]
        return np.stack([(mc[b] / mass[b]) if mass[b] > 0 else np.zeros(3) for b in bodies]).astype(np.float32)

    def set_external_forces(self, force, torque=None, bodies=None, mask: torch.Tensor | None = None) -> None:
        """Replace the wrenches of all (or the masked) environments.  ``force`` / ``torque`` (None: zero): [N, 26, 3], or
        [N, len(bodies), 3] with ``bodies`` a list of body names (joint names of ``meta["body_joint_names"]`` or
        ``"base"``); bodies not named get zero."""
        self._need_external_forces()
        n = self.num_envs
        cols = list(range(_native.EXT_BODIES)) if bodies is None else [self._body_index(b) for b in bodies]
        if len(set(cols)) != len(cols):
            raise ValueError("a body is named twice")

        def part(x, what):
            if x is None:
                return torch.zeros(n, len(cols), 3, device=self.device, dtype=torch.float32)
            x = torch.as_tensor(x, dtype=torch.float32).to(self.device)
            if tuple(x.shape) != (n, len(cols), 3):
                raise ValueError("%s must have shape %s" % (what, (n, len(cols), 3)))
            return x
        w = torch.zeros(n, _native.EXT_BODIES, 6, device=self.device, dtype=torch.float32)
        w[:, cols, 0:3] = part(force, "force")
        w[:, cols, 3:6] = part(torque, "torque")
        if not bool(torch.isfinite(w).all()):
            raise ValueError("external forces must be finite")
        mask, mp = self._mask_ptr(mask)
        _native.check(self._L.trex_set_external_forces(self._h, ctypes.c_void_p(w.data_ptr()), mp, self._stream()),
                      "trex_set_external_forces")
        self._extf_src = (w, mask)  # kept alive until the stream has consumed them

    def get_external_forces(self) -> torch.Tensor:
        """[N, 26, 6] copy of every environment's wrenches."""
        self._need_external_forces()
        t = torch.empty(self.num_envs, _native.EXT_BODIES, 6, device=self.device, dtype=torch.float32)
        _native.check(self._L.trex_get_external_forces(self._h, ctypes.c_void_p(t.data_ptr()), self._stream()),
                      "trex_get_external_forces")
        return t

    def clear_external_forces(self, mask: torch.Tensor | None = None) -> None:
        """Zero the wrenches of all (or the masked) environments."""
        self.set_external_forces(None, mask=mask)

    def set_push_schedule(self, body="base", interval: int = 100, duration: int = 10, probability: float = 1.0,
                          force=(0.0, 0.0), first_step: int = 0) -> None:
        """Random horizontal pushes on ``body``, drawn on the device per environment and ``interval``-step window: with
        chance ``probability`` a window holds one push of ``duration`` steps, magnitude uniform in ``force = (lo, hi)`` N and
        one of 32 horizontal directions; none before ``first_step`` of an episode (include/trex_b200.h,
        trex_set_push_schedule).  The push adds to the body's force in the record.  ``set_push_schedule(None)`` turns it off."""
        self._need_external_forces()
        if body is None:
            _native.check(self._L.trex_set_push_schedule(self._h, None), "trex_set_push_schedule")
            return
        lo, hi = force
        s = _native.TrexPushSchedule(body=self._body_index(body), interval=int(interval), duration=int(duration),
                                     first_step=int(first_step), probability=float(probability), force_min=float(lo),
                                     force_max=float(hi))
        _native.check(self._L.trex_set_push_schedule(self._h, ctypes.byref(s)), "trex_set_push_schedule")

    # -- state / diagnostics -----------------------------------------------------------------------
    def get_state(self) -> torch.Tensor:
        s = torch.empty(self.num_envs, _native.STATE_DIM, device=self.device, dtype=torch.float32)
        _native.check(self._L.trex_get_state(self._h, ctypes.c_void_p(s.data_ptr()), self._stream()), "trex_get_state")
        return s

    def set_state(self, state: torch.Tensor) -> None:
        self._check_tensor(state, (self.num_envs, _native.STATE_DIM), torch.float32, "state")
        _native.check(self._L.trex_set_state(self._h, ctypes.c_void_p(state.data_ptr()), self._stream()), "trex_set_state")

    def aux(self) -> torch.Tensor:
        """[N,8]: head xyz, lifting / station-keeping / energy penalties (trex_env.py:193-195), PGS
        iterations of the last step, active contacts."""
        a = torch.empty(self.num_envs, _native.AUX_DIM, device=self.device, dtype=torch.float32)
        _native.check(self._L.trex_get_aux(self._h, ctypes.c_void_p(a.data_ptr()), self._stream()), "trex_get_aux")
        return a

    # -- per-body world states and floor contact forces (every simulator) ------------------------------------------------
    # Bodies in the order of body_names(): body k < 25 is the body moved by joint k (pybullet link order, fixed links folded
    # in), 25 the base -- the order of an env-param row and of the wrench record.

    def body_names(self) -> list[str]:
        """The 26 body names in query order: the joint names of ``meta["body_joint_names"]``, then ``"base"`` (the names
        ``set_external_forces(bodies=)`` and ``set_env_params`` accept)."""
        return list(self.model.meta["body_joint_names"][1:]) + ["base"]

    def _body_query(self, states, forces):
        _native.check(self._L.trex_get_body_states(self._h, None if states is None else ctypes.c_void_p(states.data_ptr()),
                                                   None if forces is None else ctypes.c_void_p(forces.data_ptr()),
                                                   self._stream()), "trex_get_body_states")

    def body_states(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """[N, 26, 13] world state of every body, computed on the device from the current records (include/trex_b200.h,
        trex_get_body_states): COM position | body -> world quaternion x y z w | COM velocity | angular velocity.  The body
        frame is the joint frame with the joint axis along +z (the base's: its inertial frame, the record's pose)."""
        if out is None:
            out = torch.empty(self.num_envs, _native.EXT_BODIES, _native.BODY_STATE_DIM, device=self.device, dtype=torch.float32)
        self._check_tensor(out, (self.num_envs, _native.EXT_BODIES, _native.BODY_STATE_DIM), torch.float32, "out")
        self._body_query(out, None)
        return out

    def contact_forces(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """[N, 26] the floor's normal force on every body in the last physics substep (N): pybullet's
        ``getContactPoints(robot, floor)[9]`` summed over the body's links.  Friction forces are not reported."""
        if out is None:
            out = torch.empty(self.num_envs, _native.EXT_BODIES, device=self.device, dtype=torch.float32)
        self._check_tensor(out, (self.num_envs, _native.EXT_BODIES), torch.float32, "out")
        self._body_query(None, out)
        return out

    # -- joint-space dynamics (every simulator) ---------------------------------------------------------------------------
    # Coordinates u of dof_names(): base angular velocity and the velocity of the base link's COM (world frame, the record's
    # [7:13]), then the 25 joint rates in pybullet link order (the record's [38:63]; NOT the name-sorted action order).

    def dof_names(self) -> list[str]:
        """The 31 coordinate names of ``mass_matrix`` / ``bias_forces`` / ``jacobians``: six base coordinates, then the joint
        names in pybullet link order (``meta["body_joint_names"]``)."""
        return ["base_wx", "base_wy", "base_wz", "base_vx", "base_vy", "base_vz"] + list(self.model.meta["body_joint_names"][1:])

    def _dynamics_query(self, mass_matrix, bias, jacobian):
        ptrs = [None if t is None else ctypes.c_void_p(t.data_ptr()) for t in (mass_matrix, bias, jacobian)]
        _native.check(self._L.trex_get_dynamics(self._h, *ptrs, self._stream()), "trex_get_dynamics")

    def mass_matrix(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """[N, 31, 31] joint-space mass matrix M of the current records (include/trex_b200.h, trex_get_dynamics): kinetic
        energy = u^T M u / 2 in the coordinates of ``dof_names()``, with the environments' mass scales; exactly symmetric."""
        shape = (self.num_envs, _native.NUM_DOFS, _native.NUM_DOFS)
        if out is None:
            out = torch.empty(shape, device=self.device, dtype=torch.float32)
        self._check_tensor(out, shape, torch.float32, "out")
        self._dynamics_query(out, None, None)
        return out

    def bias_forces(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """[N, 31] b with M du/dt + b = tau: gravity, Coriolis and centrifugal terms (pybullet's calculateInverseDynamics with
        zero accelerations).  Damping, motors, joint limits, contacts and external wrenches are not included.  Torques of
        given accelerations: ``(sim.mass_matrix() @ udot[..., None])[..., 0] + sim.bias_forces()``."""
        shape = (self.num_envs, _native.NUM_DOFS)
        if out is None:
            out = torch.empty(shape, device=self.device, dtype=torch.float32)
        self._check_tensor(out, shape, torch.float32, "out")
        self._dynamics_query(None, out, None)
        return out

    def jacobians(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """[N, 26, 6, 31] Jacobian of every body in ``body_names()`` order: rows [COM velocity; angular velocity] in the world
        frame, so that ``J[:, k] @ u`` is ``body_states()[:, k, 7:13]`` and ``J[:, k].transpose(-1, -2) @ [f; t]`` is the
        generalized force of a wrench on body k."""
        shape = (self.num_envs, _native.EXT_BODIES, _native.JACOBIAN_ROWS, _native.NUM_DOFS)
        if out is None:
            out = torch.empty(shape, device=self.device, dtype=torch.float32)
        self._check_tensor(out, shape, torch.float32, "out")
        self._dynamics_query(None, None, out)
        return out

    def random_actions(self, step: int, seed: int = 0, env_offset: int = 0, out: torch.Tensor | None = None) -> torch.Tensor:
        """U(low, high) actions from Philox keyed by (seed, env_offset + env, step)."""
        if out is None:
            out = torch.empty(self.num_envs, _native.NUM_JOINTS, device=self.device, dtype=torch.float32)
        self._check_tensor(out, (self.num_envs, _native.NUM_JOINTS), torch.float32, "out")
        _native.check(self._L.trex_fill_random_actions(self._h, ctypes.c_void_p(out.data_ptr()), int(seed) & 0xFFFFFFFF,
                                                       int(step), int(env_offset), self._stream()), "trex_fill_random_actions")
        return out

    def stats(self) -> dict:
        s = _native.TrexStats()
        _native.check(self._L.trex_get_stats(self._h, ctypes.byref(s)), "trex_get_stats")
        return {f: getattr(s, f) for f, _ in _native.TrexStats._fields_}

    @property
    def kernel_launches(self) -> int:
        return int(self._L.trex_kernel_launches(self._h))
