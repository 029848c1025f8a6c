"""``TrexRobot``: the reference robot adapter's surface (trex_gym/trex_robot.py:256-433) over the
batched CUDA simulator.  One instance fronts environment ``env_index`` of a :class:`TrexBatchSim`.

pybullet client handles are gone; what remains is exactly what ``TrexBulletEnv`` and
``trex_train.py`` read: ``reset``, ``get_observations``, ``set_actions``, ``get_action_limits``,
``get_observation_limits``, ``get_base_position``, ``get_head_position``,
``get_total_joint_power``, ``_revolute_joint_indices``, ``_total_mass``.
"""
from __future__ import annotations

import numpy as np
import torch

from .model_compiler import map_legacy_joint_name
from .sim import TrexBatchSim


class TrexRobot(object):
    _MAX_JOINT_TORQUE_IN_NM = 300000.0  # trex_robot.py:260

    def __init__(self, sim: TrexBatchSim, env_index: int = 0, starting_configuration=None):
        self.sim = sim
        self.env_index = int(env_index)
        meta = sim.model.meta
        # pybullet joint indices of the revolute joints, sorted by joint name (trex_robot.py:311-314)
        self._revolute_joint_indices = list(meta["obs_pybullet_link_index"])
        self._joint_names = list(meta["obs_joint_names"])
        self._head_link_index = int(meta["head_pybullet_link_index"])  # trex_robot.py:316 (N1 applied)
        # trex_robot.py:318-320: sum of getDynamicsInfo(link).mass over links, base excluded
        self._total_mass = float(meta["golden"]["links_mass_excluding_base"])
        self._starting_configuration = {}
        if starting_configuration:
            known = dict(meta["starting_configuration"])
            for k, v in starting_configuration.items():
                name = map_legacy_joint_name(k)  # femur_L_joint -> joint_femur_left
                if name not in known or abs(known[name] - float(v)) > 1e-12:
                    raise ValueError(
                        "starting configuration %s=%r differs from the compiled model (%r); recompile the model"
                        % (k, v, known.get(name)))
                self._starting_configuration[name] = float(v)

    # --- reset --------------------------------------------------------------------------------
    def reset(self, reload_urdf=False):
        """trex_robot.py:39-65 + 300-320.  (The env's reset adds the one physics step.)"""
        mask = torch.zeros(self.sim.num_envs, dtype=torch.uint8, device=self.sim.device)
        mask[self.env_index] = 1
        self.sim.reset(mask)

    def reset_configuration(self):
        self.reset()

    # --- reads ----------------------------------------------------------------------------------
    def _row(self, t: torch.Tensor) -> np.ndarray:
        return t[self.env_index].detach().cpu().numpy().astype(np.float64)

    def get_observations(self):
        """q | qd | appliedJointMotorTorque of the name-sorted revolute joints (trex_robot.py:359-365)."""
        return self._row(self.sim.obs).tolist()

    get_observation = get_observations  # north-star alias

    def get_base_position(self):
        s = self._row(self.sim.get_state())
        return (float(s[0]), float(s[1]), float(s[2]))  # trex_robot.py:322-328

    def get_head_position(self):
        """World COM of link_atlas_axis after the last step (trex_robot.py:330-335)."""
        a = self._row(self.sim.aux())
        return (float(a[0]), float(a[1]), float(a[2]))

    def get_total_joint_power(self):
        o = np.asarray(self.get_observations())
        return float(np.sum(np.fabs(np.multiply(o[25:50], o[50:75]))))  # trex_robot.py:367-375

    def _get_joint_limits(self):
        return self.sim.action_low.astype(np.float64).tolist(), self.sim.action_high.astype(np.float64).tolist()

    def get_action_limits(self):
        """The joint limits (trex_robot.py:424-433); -/+ the motor torque bound on a torque-actuated simulator."""
        lo, hi = self.sim.action_limits()
        return lo.astype(np.float64), hi.astype(np.float64)

    def get_observation_limits(self):
        n = len(self._revolute_joint_indices)  # trex_robot.py:348-357
        lo, hi = self._get_joint_limits()
        lo.extend([-1.0e12] * 2 * n)
        hi.extend([1.0e12] * 2 * n)
        return np.array(lo), np.array(hi)

    # --- actions ----------------------------------------------------------------------------------
    def set_actions(self, actions):
        """trex_robot.py:413-422: position targets for the 25 motors (kp = 5e-3, kd = 0.1, 3e5 N m), name-sorted order.
        Like ``setJointMotorControlArray`` the targets persist: they are written to this environment's row of the
        simulator's target buffer and every following physics substep (``sim.step()`` without an argument, which is
        what ``TrexBulletEnv.step`` calls, trex_env.py:148-150) servoes towards them until the next call.  On a simulator
        created with ``actuation="torque"`` the values are joint torques (N m), applied in every substep instead."""
        n = len(self._revolute_joint_indices)
        a = np.asarray(actions, dtype=np.float32).reshape(-1)[:n]  # the reference slices actions[:num_joints]
        if a.shape != (n,):
            raise ValueError("expected %d actions" % n)
        self.sim.targets[self.env_index].copy_(torch.from_numpy(np.ascontiguousarray(a)), non_blocking=False)

    apply_action = set_actions  # north-star alias
