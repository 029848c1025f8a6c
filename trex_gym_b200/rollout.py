"""On-device rollout plumbing for the caller of the path (SURVEY.md section 8f row 1; BASELINE.json configs[3]).

The reference trains with baselines PPO2 (trex_train.py:35-63): ``DummyVecEnv`` -> ``VecNormalize`` ->
``ppo2.Runner`` collects ``nsteps`` transitions, then GAE(lambda=0.95, gamma=0.99).  Here the simulator writes
observations / rewards / dones straight into preallocated time-major device buffers (no host round trip per
step) and the advantage scan runs as one CUDA kernel (``trex_gae``).  The RL algorithm itself stays out of scope.
"""
from __future__ import annotations

import ctypes

import torch

from . import _native
from .sim import TrexBatchSim


class RunningMeanStd:
    """baselines ``RunningMeanStd`` (VecNormalize) on the device: parallel-variance update per batch."""

    def __init__(self, dim: int, device, epsilon: float = 1e-4):
        self.mean = torch.zeros(dim, device=device, dtype=torch.float64)
        self.var = torch.ones(dim, device=device, dtype=torch.float64)
        self.count = float(epsilon)

    def update(self, x: torch.Tensor) -> None:
        x = x.reshape(-1, self.mean.shape[0]).double()
        b_mean, b_var, b_count = x.mean(0), x.var(0, unbiased=False), x.shape[0]
        delta = b_mean - self.mean
        tot = self.count + b_count
        self.mean = self.mean + delta * (b_count / tot)
        m2 = self.var * self.count + b_var * b_count + delta * delta * (self.count * b_count / tot)
        self.var = m2 / tot
        self.count = tot


class RolloutBuffer:
    """Time-major device buffers ``[T, N, ...]`` filled in place by :class:`TrexBatchSim`."""

    def __init__(self, sim: TrexBatchSim, horizon: int):
        if getattr(sim, "actuation", "position") != "position":
            # the on-device PPO loop drives motor targets only
            raise ValueError("RolloutBuffer supports position-actuated simulators only; this one was created with "
                             "actuation=%r" % (sim.actuation,))
        self.sim, self.T, self.N = sim, int(horizon), sim.num_envs
        dev = sim.device
        f32, u8 = torch.float32, torch.uint8
        self.obs = torch.zeros(self.T + 1, self.N, _native.OBS_DIM, device=dev, dtype=f32)  # obs[t] = state step t acts in
        self.actions = torch.zeros(self.T, self.N, _native.NUM_JOINTS, device=dev, dtype=f32)
        self.rewards = torch.zeros(self.T, self.N, device=dev, dtype=f32)
        self.dones = torch.zeros(self.T + 1, self.N, device=dev, dtype=u8)  # dones[t] = obs[t] starts an episode
        self.values = torch.zeros(self.T, self.N, device=dev, dtype=f32)
        self.neglogp = torch.zeros(self.T, self.N, device=dev, dtype=f32)
        self.advantages = torch.zeros(self.T, self.N, device=dev, dtype=f32)
        self.returns = torch.zeros(self.T, self.N, device=dev, dtype=f32)
        self.obs[0].copy_(sim.obs)

    def collect(self, policy=None, seed: int = 0, step_offset: int = 0):
        """Run ``T`` env steps.  ``policy(obs[N,75]) -> (action[N,25], value[N], neglogp[N])`` on the device, or
        ``None`` for uniform random actions (the benchmark's synthetic input)."""
        sim = self.sim
        for t in range(self.T):
            if policy is None:
                sim.random_actions(step=step_offset + t, seed=seed, env_offset=sim.env_offset, out=self.actions[t])
            elif isinstance(policy, MlpPolicy):
                # fused kernel: reads obs[t] in place, writes the three rollout rows, no intermediate tensors
                policy.act_into(self.obs[t], self.actions[t], self.values[t], self.neglogp[t], step=step_offset + t, seed=seed,
                                env_offset=sim.env_offset)
            else:
                a, v, nlp = policy(self.obs[t])
                self.actions[t].copy_(a)
                self.values[t].copy_(v)
                self.neglogp[t].copy_(nlp)
            # obs[t+1], rewards[t], dones[t+1] written by the kernels, no copies
            sim.step_into(self.actions[t], self.obs[t + 1], self.rewards[t], self.dones[t + 1])
        return self

    def compute_gae(self, last_value: torch.Tensor, gamma: float = 0.99, lam: float = 0.95):
        """trex_train.py:52-53 (lam=0.95, gamma=0.99); one kernel, one thread per environment."""
        last_value = last_value.to(self.sim.device, torch.float32).contiguous()
        stream = ctypes.c_void_p(torch.cuda.current_stream(self.sim.device).cuda_stream)
        p = lambda x: ctypes.c_void_p(x.data_ptr())  # noqa: E731
        idx = self.sim.device.index if self.sim.device.index is not None else torch.cuda.current_device()
        _native.check(_native.lib().trex_gae(idx, p(self.rewards), p(self.values), p(self.dones[: self.T]), p(last_value),
                                             p(self.dones[self.T]), float(gamma), float(lam), p(self.advantages), p(self.returns),
                                             self.T, self.N, stream), "trex_gae")
        return self.advantages, self.returns

    def roll(self):
        """Start the next rollout from the last observation."""
        self.obs[0].copy_(self.obs[self.T])
        self.dones[0].copy_(self.dones[self.T])


def normalize(x: torch.Tensor, rms: RunningMeanStd, clip: float = 10.0, eps: float = 1e-8) -> torch.Tensor:
    """VecNormalize observation filter (clip 10) as one CUDA kernel."""
    x = x.contiguous()
    out = torch.empty_like(x)
    dim = x.shape[-1]
    stream = ctypes.c_void_p(torch.cuda.current_stream(x.device).cuda_stream)
    mean, var = rms.mean.float().contiguous(), rms.var.float().contiguous()
    idx = x.device.index if x.device.index is not None else torch.cuda.current_device()
    _native.check(_native.lib().trex_normalize(idx, ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(mean.data_ptr()),
                                               ctypes.c_void_p(var.data_ptr()), float(eps), float(clip),
                                               ctypes.c_void_p(out.data_ptr()), x.numel() // dim, dim, stream), "trex_normalize")
    return out


class MlpPolicy:
    """The trainer's policy / value networks (trex_train.py:48,107: baselines ``MlpPolicy`` [RECALL]) as ONE kernel:
    observation filter, two tanh trunks 75 -> 64 -> 64, Gaussian-mean head (25) with a state-independent log-std,
    value head, sampling and neglogp.  Parameters live in one packed device vector (layout: ``include/trex_b200.h``)."""

    OBS, HID, ACT = _native.OBS_DIM, 64, _native.NUM_JOINTS
    _FIELDS = (("pi_w1", (75, 64)), ("pi_b1", (64,)), ("pi_w2", (64, 64)), ("pi_b2", (64,)), ("pi_wo", (64, 25)), ("pi_bo", (25,)),
               ("vf_w1", (75, 64)), ("vf_b1", (64,)), ("vf_w2", (64, 64)), ("vf_b2", (64,)), ("vf_wo", (64, 1)), ("vf_bo", (1,)),
               ("logstd", (25,)))

    def __init__(self, device, seed: int = 0, rms: RunningMeanStd | None = None, clip: float = 10.0, eps: float = 1e-8):
        self.device = torch.device(device if not isinstance(device, int) else "cuda:%d" % device)
        n = int(_native.lib().trex_policy_param_count())
        assert n == sum(int(torch.tensor(s).prod()) for _, s in self._FIELDS)
        self.params = torch.zeros(n, device=self.device, dtype=torch.float32)
        self.rms, self.clip, self.eps = rms, float(clip), float(eps)
        g = torch.Generator(device="cpu").manual_seed(int(seed))
        # baselines initialisation: orthogonal weights (gain sqrt(2); 0.01 for the action head, 1 for the value head), zero biases
        for name, shape in self._FIELDS:
            if len(shape) == 2:
                w = torch.empty(shape[1], shape[0])
                torch.nn.init.orthogonal_(w, gain={"pi_wo": 0.01, "vf_wo": 1.0}.get(name, 2.0 ** 0.5), generator=g)
                self.view(name).copy_(w.t())

    def view(self, name: str) -> torch.Tensor:
        """Writable view of one parameter block, weights as ``[in, out]``."""
        off = 0
        for f, shape in self._FIELDS:
            size = 1
            for d in shape:
                size *= d
            if f == name:
                return self.params[off:off + size].view(*shape)
            off += size
        raise KeyError(name)

    def act_into(self, obs, action, value=None, neglogp=None, mean=None, step: int = 0, seed: int = 0, env_offset: int = 0,
                 deterministic: bool = False):
        n = obs.shape[0]
        for t, shape in ((obs, (n, self.OBS)), (action, (n, self.ACT)), (value, (n,)), (neglogp, (n,)), (mean, (n, self.ACT))):
            if t is not None and (tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_contiguous() or t.device != self.device):
                raise ValueError("policy buffers must be contiguous float32 tensors on %s with shapes [N,75] / [N,25] / [N]" % self.device)
        p = lambda x: None if x is None else ctypes.c_void_p(x.data_ptr())  # noqa: E731
        om = ov = None
        if self.rms is not None:
            om, ov = self.rms.mean.float().contiguous(), self.rms.var.float().contiguous()
        stream = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        _native.check(_native.lib().trex_policy_forward(idx, p(obs), p(om), p(ov), self.eps, self.clip, p(self.params), int(seed) & 0xFFFFFFFF,
                                                        int(step), int(env_offset), int(bool(deterministic)), p(action), p(neglogp),
                                                        p(value), p(mean), n, stream), "trex_policy_forward")
        return action, value, neglogp

    def __call__(self, obs, step: int = 0, seed: int = 0, deterministic: bool = False, env_offset: int = 0):
        n = obs.shape[0]
        a = torch.empty(n, self.ACT, device=self.device, dtype=torch.float32)
        v = torch.empty(n, device=self.device, dtype=torch.float32)
        nlp = torch.empty(n, device=self.device, dtype=torch.float32)
        return self.act_into(obs.contiguous(), a, v, nlp, step=step, seed=seed, env_offset=env_offset, deterministic=deterministic)

    def reference_forward(self, obs: torch.Tensor):
        """The same networks in plain PyTorch FP32 (tests: numerics reference of the kernel)."""
        x = obs.float()
        if self.rms is not None:
            x = torch.clamp((x - self.rms.mean.float()) / torch.sqrt(self.rms.var.float() + self.eps), -self.clip, self.clip)
        v = self.view
        hp = torch.tanh(torch.tanh(x @ v("pi_w1") + v("pi_b1")) @ v("pi_w2") + v("pi_b2"))
        hv = torch.tanh(torch.tanh(x @ v("vf_w1") + v("vf_b1")) @ v("vf_w2") + v("vf_b2"))
        return hp @ v("pi_wo") + v("pi_bo"), (hv @ v("vf_wo") + v("vf_bo")).squeeze(-1)
