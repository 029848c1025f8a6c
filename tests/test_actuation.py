"""Joint torque control (trex_config.actuation = TREX_ACTUATION_TORQUE): actions are joint torques, applied in every physics
substep.

CPU (the product kernel source through tests/emu, and the oracle with torque control inserted, tests/emu/oracle_tau.py): the
TAU instances against the oracle variant, against the zero-gain position path with the torque applied as a wrench pair, and
against a zero-gain position handle byte for byte at zero torque.  GPU (-m gpu): the library's TAU kernels."""
import ctypes

import numpy as np
import pytest

from conftest import STATE_BLOCKS, rel_err
from trex_gym_b200.model_compiler import with_params

T_MODEL = 300000.0  # the builtin model's motor_max_torque (N m)
TAU = slice(63, 88)  # the applied joint torque in the record


def _bytes(x):
    return np.ascontiguousarray(x).view(np.uint8)


def _random_torques(rng, shape, scale=2000.0):
    """Joint torques of a size that moves the joints without throwing the animal around (the bound itself is 3e5 N m)."""
    return rng.uniform(-scale, scale, shape).astype(np.float32)


def _zero_gain(model):
    """The position-mode model whose motors do what torque-mode motors do: no gain, no strength."""
    return with_params(model, motor_kp=0.0, motor_kd=0.0, motor_max_torque=0.0)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the oracle variant
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_variant_without_torque_mode_is_the_oracle(model, action_limits):
    """Check 1: the oracle built with torque control steps exactly as the oracle does while torque mode is off."""
    from oracle.oracle import Oracle
    from oracle_tau import OracleTau

    lo, hi = action_limits
    rng = np.random.default_rng(13)
    a, b = Oracle(model.blob()), OracleTau(model.blob())
    assert np.array_equal(a.reset(), b.reset())
    for t in range(6):
        act = rng.uniform(lo, hi)
        oa, ra = a.step(act)
        ob, rb = b.step(act)
        assert np.array_equal(a.get_state(), b.get_state()) and np.array_equal(oa, ob) and ra == rb, t


def test_joint_torques_are_internal_forces(model):
    """Check 2: contacts off, no link damping, one physics substep from rest at configurations along a random-torque
    trajectory: the total linear momentum changes by M g dt (1e-9 relative) and the angular momentum about the COM stays 0
    (relative to dt max|tau|).  Joint torques, joint damping and
    limit rows are internal, so this holds whatever the insertion does, as long as it only adds joint torques.  The torques
    are scaled by each joint's inverse inertia (about 20 rad/s^2) so that no joint reaches the velocity clamp, which is not
    momentum-conserving."""
    from oracle_tau import OracleTau

    m = with_params(model, linear_damping=0.0, angular_damping=0.0)
    dt = m.meta["params"]["time_step"]
    g = m.meta["params"]["gravity"]
    obs_dof = np.asarray(model["obs_dof"])
    o = OracleTau(m.blob(), num_substeps=1, contacts=False)
    o.set_torque_mode(True, T_MODEL)
    o.reset()
    scale = np.array([20.0 / o.minv_column(6 + d)[6 + d] for d in obs_dof])
    rng = np.random.default_rng(3)
    worst_p, worst_l, fastest = 0.0, 0.0, 0.0
    for t in range(40):
        # one substep from rest at the configuration the trajectory has reached: the momentum of the velocity change (with
        # velocities, the velocity-product terms move momentum by order dt |u|^2 within a substep, and the configuration's
        # own change adds a term of order dt^2 tau^2: measured up to 3e-2 of M g dt)
        s = o.get_state()
        s0 = s.copy()
        s0[7:13] = 0.0
        s0[38:88] = 0.0
        o.set_state(s0)
        p0 = o.momentum()
        a = rng.uniform(-1.0, 1.0, 25) * scale
        o.step(a)
        s1 = o.get_state()
        sv = s0.copy()
        sv[7:13], sv[38:63] = s1[7:13], s1[38:63]
        o.set_state(sv)
        p1 = o.momentum()
        mass = p0["mass"]
        ref = np.array([0.0, 0.0, -mass * g * dt])
        worst_p = max(worst_p, np.abs(p1["P"] - p0["P"] - ref).max() / (mass * g * dt))
        L1 = p1["L"] - np.cross(p1["com"], p1["P"])  # about the COM (L0 = 0 from rest)
        worst_l = max(worst_l, np.abs(L1).max() / (np.abs(a).max() * dt))
        # the trajectory goes on from where it was, with its velocities
        o.set_state(s)
        o.step(a)
        fastest = max(fastest, np.abs(o.get_state()[38:63]).max())
    assert 1.0 < fastest < 100.0, fastest  # the joints move, and stay below the clamp
    # measured: 3.6e-15 and 8.2e-14
    assert worst_p < 1e-9, worst_p
    assert worst_l < 1e-11, worst_l


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the emulator's TAU instances
# ---------------------------------------------------------------------------------------------------------------------
def _parity(e, o, rng, steps, hold_for=5, scale=2000.0):
    errs, sigs, n_contact = [], 0, 0
    a = _random_torques(rng, 25, scale)
    for t in range(steps):
        if t % hold_for == 0:
            a = _random_torques(rng, 25, scale)
        o.set_state(e.get_state(o.num_candidates))
        o.step(a.astype(np.float64))
        e.step(a)
        so, se = o.get_state(), e.get_state(o.num_candidates)
        errs.append(max(rel_err(so[sl], se[sl]) for sl in STATE_BLOCKS.values()))
        sigs += int(e.rec[158]) == o.signature
        n_contact += o.last_num_contacts > 0
    return np.asarray(errs), sigs, n_contact


@pytest.mark.parametrize("with_", ["alone", "env_params", "external_forces"])
def test_random_torques_contact_free_match_the_oracle(model, with_):
    """Check 3 (contact-free): random torques, per env step < 2e-5 against the oracle variant, every active-set signature
    equal; alone and together with ENVP (a row equal to the model's constants but a torque bound of 1,500 N m, so that
    clipping happens) and EXTF (a zero record)."""
    from emu_tau import EmuTauEnv
    from oracle_tau import OracleTau

    rng = np.random.default_rng(7)
    e = EmuTauEnv(model.blob(), contacts=False, torque=True)
    bound = T_MODEL
    if with_ == "env_params":
        r = e.default_env_params()
        bound = r[29] = 1500.0
        e.set_env_params(r)
    elif with_ == "external_forces":
        e.set_external_forces(np.zeros((26, 6), np.float32))
    o = OracleTau(model.blob(), contacts=False)
    o.set_torque_mode(True, bound)
    e.reset()
    errs, sigs, _ = _parity(e, o, rng, 20)
    assert errs.max() < 2e-5, errs.max()
    assert sigs == 20


def test_random_torques_with_contacts_match_the_oracle(model):
    """Check 3 (contacts): single substeps against the oracle variant, p50 < 2e-5 and p99 < 2e-3 (the external-forces
    bounds)."""
    from emu_tau import EmuTauEnv
    from oracle_tau import OracleTau

    rng = np.random.default_rng(8)
    sub = with_params(model, time_step=0.002, solver_iterations=60)
    e = EmuTauEnv(sub.blob(), num_substeps=1, deferred=1, torque=True)
    o = OracleTau(sub.blob(), num_substeps=1)
    o.set_torque_mode(True, T_MODEL)
    e.reset()
    errs, _, n_contact = _parity(e, o, rng, 220, scale=500.0)
    assert n_contact > 60
    assert np.percentile(errs, 50) < 2e-5 and np.percentile(errs, 99) < 2e-3, (np.percentile(errs, [50, 99]), errs.max())


def test_torque_equals_the_wrench_pair(model):
    """Check 4: one substep, contacts off: a torque tau on joint k does what a zero-gain position handle does with the wrench
    pair +tau axis on the joint's body and -tau axis on its parent, set from the same pose (FP32 round-off, not bitwise)."""
    from emu_bodies import EmuBodiesEnv
    from emu_extf import EmuExtfEnv
    from emu_tau import EmuTauEnv

    obs_dof = np.asarray(model["obs_dof"])
    parent = np.asarray(model["mb_parent"])
    a = EmuTauEnv(model.blob(), num_substeps=1, contacts=False, torque=True)
    b = EmuExtfEnv(_zero_gain(model).blob(), num_substeps=1, contacts=False)
    q = EmuBodiesEnv(model.blob(), num_substeps=1, contacts=False)
    a.reset()
    rng = np.random.default_rng(4)
    worst = 0.0
    for t in range(12):
        tau = _random_torques(rng, 25)
        states, _ = q.body_states(a.rec)
        w = np.zeros((26, 6), np.float64)
        for slot in range(25):
            k = obs_dof[slot]
            x, y, z, s = states[k, 3:7].astype(np.float64)
            axis = np.array([2 * (x * z + s * y), 2 * (y * z - s * x), 1 - 2 * (x * x + y * y)])  # body +z in the world
            p = parent[k + 1]
            w[k, 3:] += tau[slot] * axis
            w[p - 1 if p > 0 else 25, 3:] -= tau[slot] * axis
        b.set_external_forces(w.astype(np.float32))
        b.rec[:] = a.rec
        a.step(tau)
        b.step(np.zeros(25, np.float32))
        worst = max(worst, max(rel_err(a.rec[sl], b.rec[sl]) for name, sl in STATE_BLOCKS.items() if name != "tau"))
    # measured: 1.1e-6
    assert worst < 1e-5, worst


SCENARIOS = {  # (n envs, emulator flags, EmuEnv kwargs, steps, start) -- the scenarios of test_env_params.py
    "contact": (4, 1, {}, 6, "perturbed"),
    "contact_solve4_shared_memory": (4, 1, {}, 4, "perturbed"),
    "contact_solve4_tensor_memory": (4, 1 | 64, {}, 4, "perturbed"),
    "packed_4warp": (4, 1 | 8, {}, 4, "perturbed"),
    "front_solve": (4, 0, {}, 4, "perturbed"),
    "contact_free": (4, 1, {"contacts": False}, 4, "perturbed"),
    "fallen_start": (4, 1, {"reset_mode": 1, "seed": 3, "max_episode_steps": 3}, 5, "reset"),
    "standing_solve2_shared_memory": (3, 1, {}, 40, "standing"),
    "standing_solve2_tensor_memory": (3, 1 | 32, {}, 40, "standing"),
}


def _compare_zero_torque(a, b):
    """a: the torque handle's outputs, b: the zero-gain position handle's; byte for byte except the applied torque, which is
    compared by value (the torque handle reports the command +0, the position handle the motor's impulse / dt = +-0)."""
    for t, (x, y) in enumerate(zip(a, b)):
        rx, ry = x[0].copy(), y[0].copy()
        assert np.array_equal(rx[..., TAU], ry[..., TAU]), t
        rx[..., TAU] = 0.0
        ry[..., TAU] = 0.0
        assert np.array_equal(_bytes(rx), _bytes(ry)), t
        if len(x) > 2:
            assert np.array_equal(x[1], y[1]), t  # obs (its torque block by value)
            assert np.array_equal(_bytes(x[1][:, :50]), _bytes(y[1][:, :50])), t
            for k in (2, 3, 4):
                assert np.array_equal(_bytes(x[k]), _bytes(y[k])), (t, k)


@pytest.mark.parametrize("extf", [False, True], ids=["", "external_forces"])
@pytest.mark.parametrize("envp", [False, True], ids=["", "env_params"])
@pytest.mark.parametrize("scen", list(SCENARIOS))
def test_zero_torque_is_the_zero_gain_position_path(model, scen, envp, extf):
    """Check 5: zero torque gives the records, obs, reward, done and aux of a position handle built from
    with_params(motor_kp=0, motor_kd=0, motor_max_torque=0) byte for byte (the applied torque by value), for the emulated
    warps / ENVP / EXTF combinations; ENVP: random rows, the position handle's with [27:30] = 0."""
    from emu_extf import EmuExtfWarp4
    from emu_tau import EmuTauWarp4
    from test_external_forces import _random_env_row, _states

    n, flags, kw, nsteps, how = SCENARIOS[scen]
    start = _states(model, 4, np.random.default_rng(11))
    rows_t = rows_p = None
    if envp:
        from emu_envp import EmuEnvpEnv

        rng = np.random.default_rng(3)
        rows_t = np.stack([_random_env_row(rng, EmuEnvpEnv(model.blob()).default_env_params()) for _ in range(n)])
        rows_p = rows_t.copy()
        rows_p[:, 27:30] = 0.0
    rng = np.random.default_rng(9)
    wrench = (rng.normal(size=(n, 26, 6)) * 20.0).astype(np.float32) if extf else None

    def run(w, rows, torque):
        if rows is not None:
            w.env.set_env_params(rows)
        if wrench is not None:
            w.env.set_external_forces(wrench)
        if torque:
            w.env.set_torque_mode()
        out = [(w.rec.copy(),), ]
        w.reset()
        out.append((w.rec.copy(),))
        if how == "perturbed":
            w.rec[:] = start[:n]
        for t in range(nsteps):
            obs, rew, done = w.step(np.zeros((n, 25), np.float32))
            out.append((w.rec.copy(), obs.copy(), rew.copy(), done.copy(), w.aux.copy()))
        return out, w

    a, wa = run(EmuTauWarp4(model.blob(), n=n, deferred=flags, **kw), rows_t, True)
    b, _ = run(EmuExtfWarp4(_zero_gain(model).blob(), n=n, deferred=flags, **kw), rows_p, False)
    _compare_zero_torque(a, b)
    if scen == "packed_4warp":
        assert wa.env.packed_rounds() > 0
    if scen.startswith("standing") and not extf:  # (the pushed animals settle with fewer contacts)
        assert wa.env.heavy_solves() > 0


def test_applied_torque_is_the_clipped_command(model):
    """Obs [50:75] and record [63:88] hold the clipped command bit for bit, the reward's energy term is w_e sum |qd tau| of
    the observation (sequential float32), and a reset step reports zero torque."""
    from emu_tau import EmuTauEnv

    obs_dof = np.asarray(model["obs_dof"])
    e = EmuTauEnv(model.blob(), torque=True, max_episode_steps=3)
    r = e.default_env_params()
    r[29] = 1000.0
    e.set_env_params(r)
    e.reset()
    rng = np.random.default_rng(1)
    for t in range(6):
        a = rng.uniform(-3000.0, 3000.0, 25).astype(np.float32)
        obs, rew, done = e.step(a)
        clipped = np.clip(a, np.float32(-1000.0), np.float32(1000.0))
        if done:
            assert np.all(obs[50:75] == 0.0), t
            continue
        assert np.array_equal(_bytes(obs[50:75]), _bytes(clipped)), t
        rec_tau = np.zeros(25, np.float32)
        rec_tau[:] = e.rec[63:88][obs_dof]
        assert np.array_equal(_bytes(rec_tau), _bytes(clipped)), t
        power = np.float32(0.0)
        for k in range(25):
            power = np.float32(power + np.abs(np.float32(obs[25 + k] * obs[50 + k])))
        assert e.aux[5] == np.float32(np.float32(0.005) * power), t


def test_python_and_c_surface_without_a_device():
    """The config struct keeps its size; the new call refuses a NULL handle; an unknown actuation is refused in Python."""
    from trex_gym_b200 import _native
    from trex_gym_b200.sim import TrexBatchSim

    assert ctypes.sizeof(_native.TrexConfig) == 96
    lo = np.zeros(25, np.float32)
    L = _native.lib()
    assert L.trex_get_action_limits(None, lo.ctypes.data, lo.ctypes.data) == -1
    with pytest.raises(ValueError):
        TrexBatchSim(4, actuation="velocity")


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _sim(n, **kw):
    from trex_gym_b200.sim import TrexBatchSim

    return TrexBatchSim(n, device=0, **kw)


def _zero_gain_sim(n, **kw):
    from trex_gym_b200.model_compiler import load_builtin

    return _sim(n, model=_zero_gain(load_builtin()), **kw)


def _np(x):
    return x.detach().cpu().numpy()


def _equal_but_torque(sa, sb):
    """States / obs of a torque handle and a zero-gain position handle: bytes equal outside the torque block, values inside."""
    a, b = _np(sa).copy(), _np(sb).copy()
    blk = TAU if a.shape[1] != 75 else slice(50, 75)
    if not np.array_equal(a[:, blk], b[:, blk]):
        return False
    a[:, blk] = 0.0
    b[:, blk] = 0.0
    return np.array_equal(a.view(np.uint8), b.view(np.uint8))


def _hold_actions(sim):
    import torch

    from test_external_forces import _hold

    return torch.tensor(_hold(sim.model), device=sim.device).repeat(sim.num_envs, 1).contiguous()


GPU_ZERO_CONFIGS = dict(
    __import__("test_env_params").GPU_CONFIGS,
    env_params=(1024, {"env_params": True}, "random"),
    external_forces=(1024, {"external_forces": True}, "random"),
)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", list(GPU_ZERO_CONFIGS))
def test_gpu_zero_torque_is_the_zero_gain_position_path(cfg):
    """Check 6: zero torque gives the obs, reward, done and state of a zero-gain position handle byte for byte (the applied
    torque by value), across the env-params configurations and with env_params / external_forces on."""
    import torch

    n, kw, acts = GPU_ZERO_CONFIGS[cfg]
    a = _sim(n, actuation="torque", **kw)
    b = _zero_gain_sim(n, **kw)
    if kw.get("env_params"):
        rows = b.get_env_params()
        rows[:, 27:30] = 0.0
        b.set_env_params(rows)
        assert float(a.get_env_params()[:, 30].abs().max()) == 0.0
    zero = torch.zeros(n, 25, device=a.device)
    steps = 24 if acts == "standing" else 8
    for t in range(steps):
        oa, ra, da = [x.clone() for x in a.step(zero)]
        ob, rb, db = b.step(zero)
        assert _equal_but_torque(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db), (cfg, t)
        assert _equal_but_torque(a.get_state(), b.get_state()), (cfg, t)


@pytest.mark.gpu
def test_gpu_zero_torque_under_graph_capture():
    import torch

    a, b = _sim(1024, actuation="torque"), _zero_gain_sim(1024)
    zero = torch.zeros(1024, 25, device=a.device)
    for t in range(4):
        oa = a.step_graph(zero)[0].clone()
        ob = b.step_graph(zero)[0]
        assert _equal_but_torque(oa, ob), t
    assert _equal_but_torque(a.get_state(), b.get_state())


@pytest.mark.gpu
def test_gpu_random_torques_match_the_oracle(model):
    """Check 7: 4,096 environments under random torques, 64 checked per step against the oracle variant."""
    import torch

    from oracle_tau import OracleTau

    n, rng = 4096, np.random.default_rng(12)
    s = _sim(n, actuation="torque")
    check = list(range(0, n, n // 64))
    oracles = {e: OracleTau(model.blob()) for e in check}
    for o in oracles.values():
        o.set_torque_mode(True, T_MODEL)
    nc = oracles[0].num_candidates
    free, contact = [], []
    for t in range(16):
        pre = _np(s.get_state())
        act = torch.from_numpy(_random_torques(rng, (n, 25))).to(s.device)
        s.step(act)
        post = _np(s.get_state())
        acts = _np(act).astype(np.float64)
        for e in check:
            o = oracles[e]
            o.set_state(np.concatenate([pre[e, :88], pre[e, 88:88 + nc]]).astype(np.float64))
            o.step(acts[e])
            so = o.get_state()
            err = max(rel_err(so[sl], post[e, :88 + nc][sl]) for sl in STATE_BLOCKS.values())
            (contact if o.last_num_contacts else free).append(err)
    assert len(free) > 0 and np.percentile(free, 99) < 2e-5 and max(free) < 5e-5, (np.percentile(free, 99), max(free))
    # whole env steps in contact: the bound of the external-forces GPU test
    assert len(contact) > 0 and np.percentile(contact, 50) < 1e-3 and np.percentile(contact, 99) < 2e-2, np.percentile(contact, [50, 99])


@pytest.mark.gpu
def test_gpu_observation_and_energy_report_the_clipped_command():
    """Check 8: obs [50:75] is the clipped command bit for bit; aux's energy term is w_e sum |qd tau| of the observation."""
    import torch

    n = 512
    s = _sim(n, actuation="torque")
    lo, hi = s.action_limits()
    assert np.all(hi == np.float32(T_MODEL)) and np.all(lo == -hi)
    jl, jh = s.action_low, s.action_high
    assert np.all(jl < jh) and not np.array_equal(jh, hi)  # the observation space keeps the joint limits
    rng = np.random.default_rng(2)
    for t in range(6):
        a = _random_torques(rng, (n, 25), 4000.0)
        a[:, 0] = 4.0e5  # above the bound
        obs, rew, done = s.step(torch.from_numpy(a).to(s.device))
        o = _np(obs)
        d = _np(done).astype(bool)
        clipped = np.clip(a, -np.float32(T_MODEL), np.float32(T_MODEL))
        assert np.array_equal(o[~d, 50:75].view(np.uint32), clipped[~d].view(np.uint32)), t
        aux = _np(s.aux())
        power = np.zeros(n, np.float32)
        for k in range(25):
            power = (power + np.abs(o[:, 25 + k] * o[:, 50 + k])).astype(np.float32)
        assert np.array_equal(aux[~d, 5], (np.float32(0.005) * power[~d]).astype(np.float32)), t
    r = s.random_actions(step=0)
    assert float(r.abs().max()) <= T_MODEL and float(r.min()) < 0.0 < float(r.max())


@pytest.mark.gpu
def test_gpu_env_params_bounds_clip_per_environment():
    """Check 9: per-environment bounds clip per environment; element 30 stays 0 after a set and after randomized resets."""
    import torch

    n = 256
    s = _sim(n, actuation="torque", env_params=True, max_episode_steps=3)
    rows = s.get_env_params()
    assert float(rows[:, 30].abs().max()) == 0.0
    bounds = torch.linspace(100.0, 2000.0, n, device=s.device)
    rows[:, 29] = bounds
    rows[:, 30] = 123.0  # ignored
    s.set_env_params(rows)
    assert float(s.get_env_params()[:, 30].abs().max()) == 0.0
    a = torch.full((n, 25), 5000.0, device=s.device)
    a[:, 1::2] = -5000.0
    obs, _, _ = s.step(a)
    exp = torch.clamp(a, -bounds[:, None], bounds[:, None])
    assert torch.equal(obs[:, 50:75], exp)
    s.set_env_param_ranges({"max_torque": 50.0}, {"max_torque": 500.0})
    for t in range(8):
        s.step(a)
    got = s.get_env_params()
    assert float(got[:, 30].abs().max()) == 0.0
    assert float(got[:, 29].min()) >= 50.0 and float(got[:, 29].max()) <= 500.0


@pytest.mark.gpu
def test_gpu_position_handles_and_wrappers():
    """Position handles keep the joint limits as action limits; the environment classes take actuation=; the rollout loop
    refuses a torque handle; an unknown trex_config.actuation is refused."""
    from trex_gym_b200 import _native
    from trex_gym_b200.rollout import RolloutBuffer
    from trex_gym_b200.trex_env import TrexBulletEnv, TrexVecEnv

    p = _sim(8)
    lo, hi = p.action_limits()
    assert np.array_equal(lo, p.action_low) and np.array_equal(hi, p.action_high)
    v = TrexVecEnv(8, actuation="torque")
    assert np.all(v.action_space.high == np.float32(T_MODEL))
    assert np.array_equal(v.observation_space.low[:25], p.action_low)
    e = TrexBulletEnv(actuation="torque")
    assert np.all(e.action_space.high == np.float32(T_MODEL))
    e.step(np.full(25, 100.0, np.float32))
    assert np.all(np.asarray(e._observation)[50:75] == 100.0)
    with pytest.raises(ValueError):
        RolloutBuffer(v.sim, 4)
    cfg = _native.TrexConfig()
    cfg.actuation = 2
    h = ctypes.c_void_p()
    blob = p.model.blob()
    assert _native.lib().trex_create(blob, len(blob), 8, 0, ctypes.byref(cfg), ctypes.byref(h)) == -1
