"""``TrexBulletEnv`` / ``TrexVecEnv``: the gym surface of the reference (trex_gym/trex_env.py) over
the batched CUDA simulator.

``TrexBulletEnv`` is the drop-in single-environment class (same constructor, ``reset``/``step``/
``seed``/``render``, ``action_space``/``observation_space``/``model``/``metadata``).
``TrexVecEnv`` is the batched form with the baselines ``VecEnv`` call signature
(``reset() -> obs[N,75]``, ``step(actions[N,25]) -> (obs, rews, dones, infos)``) that returns
torch CUDA tensors instead of numpy arrays.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import spaces
from .model_compiler import BLOB_PATH, CompiledModel, compile_model, load_builtin
from .reference_loader import ReferenceToolsNotFound
from .sim import TrexBatchSim
from .trex_robot import TrexRobot

NUM_SUBSTEPS = 5  # trex_env.py:18
FLOOR_URDF_FILENAME = "floor.urdf"
EARTH_GRAVITATIONAL_CONSTANT = 9.81
RENDER_HEIGHT = 720
RENDER_WIDTH = 960


def _load_model(urdf_path, contact_model="points") -> CompiledModel:
    """Compile ``urdf_path`` through the reference's ``tools/urdf_parsing`` when that checkout is
    reachable; otherwise fall back to the compiled model shipped with the package (generated from
    the reference's assets/trex.urdf by the same compiler)."""
    if urdf_path and os.path.isfile(urdf_path):
        try:
            return compile_model(urdf_path, contact_model=contact_model)
        except ReferenceToolsNotFound:
            pass
    if not os.path.isfile(BLOB_PATH):
        raise FileNotFoundError("no URDF at %r and no built-in model blob" % (urdf_path,))
    return load_builtin(contact_model)


class TrexBulletEnv(spaces.Env):
    """The gym environment for the T-rex model (trex_env.py:25-196), CUDA-backed."""

    metadata = {"render.modes": ["human", "rgb_array"], "video.frames_per_second": 50}

    def __init__(self, urdf_path=None, action_repeat=1, distance_weight=1.0, energy_weight=0.005, drift_weight=0.002,
                 render=False, device=0, model=None, contacts=True, contact_model="points", literal_reference=False,
                 actuation="position"):
        """``actuation="torque"``: an action is the joint torque (N m) of every joint, applied in every physics substep
        (``TrexBatchSim``); ``action_space`` is then -/+ the motor torque bound."""
        self._time_step = 0.01
        self._urdf_path = urdf_path
        self._action_repeat = action_repeat
        self._num_bullet_solver_iterations = 300
        self._observation = []
        self._env_step_counter = 0
        self._is_render = render
        self._last_base_position = [0.0] * 3
        self._weight_distance = distance_weight
        self._weight_energy = energy_weight
        self._weight_drift = drift_weight
        # trex_env.py:70-73
        self._time_step /= NUM_SUBSTEPS
        self._num_bullet_solver_iterations /= NUM_SUBSTEPS
        self._action_repeat *= NUM_SUBSTEPS
        self._starting_configuration = {  # trex_env.py:81-87 (legacy names; mapped by TrexRobot)
            "femur_L_joint": -0.6, "tibia_L_joint": 0.4, "tarsometatarsus_L_joint": -1.2,
            "femur_R_joint": -0.6, "tibia_R_joint": 0.4, "tarsometatarsus_R_joint": -1.2,
        }
        # contact_model: "points" (support points of the visual meshes) or "primitives" (spheres / capsules fitted to them).
        # literal_reference=True reproduces what the reference's own pybullet calls do with the checked-in URDF [RECALL]:
        # inertia recomputed from the (absent) collision shapes and no floor contact at all (the URDF has no <collision>:
        # the animal free-falls).  The DEFAULT is the physically meaningful configuration -- inertia tensors from the file
        # and floor contact on derived geometry -- which is NOT what the literal reference simulates (INTEGRATION.md).
        if literal_reference:
            contacts = False
            mdl = model if model is not None else load_builtin("literal")
        else:
            mdl = model if model is not None else _load_model(urdf_path, contact_model)
        # dt = 0.01/NUM_SUBSTEPS and int(300/NUM_SUBSTEPS) iterations per physics step; the env step runs
        # action_repeat * NUM_SUBSTEPS physics steps (trex_env.py:148-150)
        self._sim = TrexBatchSim(1, device=device, model=mdl, num_substeps=NUM_SUBSTEPS,
                                 distance_weight=distance_weight, energy_weight=energy_weight,
                                 drift_weight=drift_weight, contacts=contacts, actuation=actuation)
        self._repeat_env_steps = int(action_repeat)
        self.model = None
        self.np_random = None
        self.seed()
        self.reset()
        action_low, action_high = self.model.get_action_limits()
        self.action_space = spaces.Box(low=action_low, high=action_high, dtype=np.float32)
        observation_low, observation_high = self.model.get_observation_limits()
        self.observation_space = spaces.Box(low=observation_low, high=observation_high, dtype=np.float32)

    def reset(self):
        if self.model is None:
            self.model = TrexRobot(self._sim, 0, starting_configuration=self._starting_configuration)
        self._sim.reset()  # reset pose + zero-gain motors + one physics step (trex_env.py:115-120)
        self._env_step_counter = 0
        self._last_base_position = self.model.get_base_position()
        return self.model.get_observations()

    def seed(self, seed=None):
        self.np_random, seed = spaces.np_random(seed)
        return [seed]

    def step(self, action):
        action = np.asarray(action, dtype=np.float32)
        if action.shape != (25,):
            raise ValueError("The action dimension is not the same as the number of motors.")
        clipped_action = np.clip(action, self.action_space.low, self.action_space.high)  # trex_env.py:147
        # trex_env.py:148-150: `for _ in range(action_repeat): model.set_actions(clipped); stepSimulation()` -- the targets
        # persist in the simulator (TrexRobot.set_actions) and one sim.step() runs NUM_SUBSTEPS physics steps on them
        self.model.set_actions(clipped_action)
        for _ in range(self._repeat_env_steps):
            self._sim.step()
        self._env_step_counter += 1
        self._observation = self.model.get_observations()
        return self._observation, self.compute_reward(), self.should_terminate(), {}

    def render(self, mode="rgb_array", close=False):
        return np.array([])  # rendering is out of scope (SURVEY.md section 2 #15)

    def should_terminate(self):
        return False  # trex_env.py:183-184

    def compute_reward(self):
        self._last_base_position = self.model.get_head_position()
        return float(self._sim.reward[0].item())  # trex_env.py:186-196, computed in-kernel

    def close(self):
        self._sim.close()


TrexEnv = TrexBulletEnv  # north-star name


class TrexVecEnv(object):
    """Batched environment with the baselines ``VecEnv`` surface (what ``DummyVecEnv`` ->
    ``VecNormalize`` -> ``ppo2.Runner`` call, trex_train.py:44-49), torch CUDA tensors in/out."""

    def __init__(self, num_envs, urdf_path=None, distance_weight=1.0, energy_weight=0.005, drift_weight=0.002,
                 device=0, model=None, num_substeps=NUM_SUBSTEPS, max_episode_steps=0, contacts=True, seed=0, contact_model="points",
                 literal_reference=False, randomize=None, pushes=None, actuation="position"):
        """``randomize``: None, or a dict of parameter name -> (low, high) -- ``mass_scale`` (a scale, or {body: scale}),
        ``friction``, ``kp``, ``kd``, ``max_torque`` -- drawn per environment at every reset (``TrexBatchSim.set_env_param_ranges``);
        parameters not named keep the model's value.
        ``pushes``: None, or the keyword arguments of ``TrexBatchSim.set_push_schedule`` (``body``, ``interval``, ``duration``,
        ``probability``, ``force=(lo, hi)``, ``first_step``): random horizontal pushes drawn on the device.
        ``actuation``: ``"position"`` (motor targets) or ``"torque"`` (joint torques, ``action_space`` -/+ the motor torque
        bound; see ``TrexBatchSim``)."""
        if literal_reference:  # see TrexBulletEnv
            contacts = False
            mdl = model if model is not None else load_builtin("literal")
        else:
            mdl = model if model is not None else _load_model(urdf_path, contact_model)
        self.sim = TrexBatchSim(num_envs, device=device, model=mdl, num_substeps=num_substeps,
                                distance_weight=distance_weight, energy_weight=energy_weight, drift_weight=drift_weight,
                                max_episode_steps=max_episode_steps, contacts=contacts, seed=seed, env_params=randomize is not None,
                                external_forces=pushes is not None, actuation=actuation)
        if randomize is not None:
            self.sim.set_env_param_ranges({k: v[0] for k, v in randomize.items()}, {k: v[1] for k, v in randomize.items()})
        if pushes is not None:
            self.sim.set_push_schedule(**pushes)
        self.num_envs = int(num_envs)
        alo, ahi = self.sim.action_limits()
        self.action_space = spaces.Box(low=alo, high=ahi, dtype=np.float32)
        lo, hi = self.sim.action_low, self.sim.action_high  # the joint limits bound the observed positions in either mode
        n = lo.shape[0]
        self.observation_space = spaces.Box(low=np.concatenate([lo, np.full(2 * n, -1.0e12, np.float32)]),
                                            high=np.concatenate([hi, np.full(2 * n, 1.0e12, np.float32)]), dtype=np.float32)

    def reset(self):
        return self.sim.reset()

    def step(self, actions):
        if not isinstance(actions, torch.Tensor):
            actions = torch.as_tensor(np.asarray(actions, np.float32))
        actions = actions.to(device=self.sim.device, dtype=torch.float32).contiguous()
        if tuple(actions.shape) != (self.num_envs, 25):
            raise ValueError("The action dimension is not the same as the number of motors.")
        obs, rew, done = self.sim.step(actions)
        return obs, rew, done, [{} for _ in range(self.num_envs)]  # one empty info dict per environment (trex_env.py:154)

    def step_async(self, actions):
        self._pending = actions

    def step_wait(self):
        return self.step(self._pending)

    def close(self):
        self.sim.close()
