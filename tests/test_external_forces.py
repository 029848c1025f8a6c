"""External forces and torques on the bodies (trex_config.external_forces = 1), and the on-device push schedule.

CPU (the product kernel source through tests/emu, and the oracle): the EXTF instances against the external_forces = 0 path,
against the oracle fed the links' share of each wrench (model_compiler.link_wrenches), against a changed-gravity model, and
the push schedule against a numpy reference.  GPU (-m gpu): the library's EXTF kernels."""
import ctypes
import math

import numpy as np
import pytest

from conftest import STATE_BLOCKS, rel_err
from trex_gym_b200.model_compiler import link_wrenches, with_params

BASE = 25
G = 9.81
PUSH_KEY = 0x9E57


def _hold(model):
    names = list(model.meta["obs_joint_names"])
    hold = np.zeros(25, np.float32)
    for k, v in model.meta["starting_configuration"].items():
        hold[names.index(k)] = v
    return hold


def _body_mass(model):
    """[26] merged-body masses in wrench-record order (k: body k + 1, 25: the base)."""
    m = np.asarray(model["mb_mass"], np.float64)
    return np.concatenate([m[1:], m[:1]])


def _random_wrenches(rng, model, n=None, scale=0.3):
    """Forces up to about scale * m_b g per body in random directions, torques up to 0.1 m times that."""
    mb = _body_mass(model)
    shape = (26,) if n is None else (n, 26)
    f = rng.normal(size=shape + (3,)) * (scale * G * mb / math.sqrt(3.0))[:, None]
    t = rng.normal(size=shape + (3,)) * (0.1 * scale * G * mb / math.sqrt(3.0))[:, None]
    return np.concatenate([f, t], axis=-1).astype(np.float32)


def _bytes(x):
    return np.ascontiguousarray(x).view(np.uint8)


def _equal(a, b):
    for t, (x, y) in enumerate(zip(a, b)):
        for k, (u, v) in enumerate(zip(x, y)):
            assert np.array_equal(_bytes(u), _bytes(v)), (t, k)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the emulator
# ---------------------------------------------------------------------------------------------------------------------
# scenario: (n envs, emulator flags, EmuEnv kwargs, steps, start) -- the scenario list of test_env_params.py
SCENARIOS = {
    "contact": (4, 1, {}, 8, "perturbed"),
    "contact_solve4_tensor_memory": (4, 1 | 64, {}, 6, "perturbed"),
    "packed_4warp": (4, 1 | 8, {}, 6, "perturbed"),
    "front_solve": (4, 0, {}, 5, "perturbed"),
    "contact_free": (4, 1, {"contacts": False}, 6, "perturbed"),
    "fallen_start": (4, 1, {"reset_mode": 1, "seed": 3, "max_episode_steps": 3}, 6, "reset"),
    "standing_solve2": (3, 1, {}, 50, "standing"),
}


def _states(model, n, rng):
    """n perturbed reset states: joints off the crouch, the later ones on / near the floor."""
    from emu import EmuWarp4

    w = EmuWarp4(model.blob(), n=n)
    w.reset()
    qlo, qhi = model["mb_lower"][1:], model["mb_upper"][1:]
    rec = w.rec.copy()
    for e in range(n):
        rec[e, 13:38] = np.clip(rec[e, 13:38] + rng.uniform(-0.3, 0.3, 25), qlo - 0.02, qhi + 0.02)
        rec[e, 2] -= 0.12 * e
    return rec


@pytest.fixture(scope="module")
def starts(model):
    return _states(model, 4, np.random.default_rng(11))


def _run(model, scen, start, warp, wrench=None, rows=None, per_step=None, seed=0):
    """Steps one emulated work unit; returns (rec, obs[, reward, done, aux]) after the reset and every step.
    per_step(t, warp) runs before step t (to change the record)."""
    n, flags, kw, nsteps, how = SCENARIOS[scen]
    w = warp(model.blob(), n=n, deferred=flags, **kw)
    if rows is not None:
        w.env.set_env_params(rows)
    if wrench is not None:
        w.env.set_external_forces(wrench)
    out = [(w.rec.copy(), w.reset())]
    if how == "perturbed":
        w.rec[:] = start[:n]
    rng = np.random.default_rng(seed)
    hold = _hold(model)
    for t in range(nsteps):
        if how == "standing":
            acts = np.stack([hold + rng.uniform(-0.02, 0.02, 25) * (e > 0) for e in range(n)]).astype(np.float32)
        else:
            acts = rng.uniform(-1.0, 1.0, (n, 25)).astype(np.float32)
        if per_step is not None:
            per_step(t, w)
        obs, rew, done = w.step(acts)
        out.append((w.rec.copy(), obs.copy(), rew.copy(), done.copy(), w.aux.copy()))
    return out, w


def _random_env_row(rng, default):
    r = default.copy()
    r[:26] = rng.uniform(0.8, 1.25, 26)
    r[26] = rng.uniform(0.15, 0.5)
    r[27] = default[27] * rng.uniform(0.8, 1.25)
    r[28] = default[28] * rng.uniform(0.8, 1.25)
    r[29] = default[29] * rng.uniform(0.7, 1.0)
    return r.astype(np.float32)


@pytest.mark.parametrize("envp", [False, True], ids=["no_env_params", "env_params"])
@pytest.mark.parametrize("scen", list(SCENARIOS))
def test_zero_record_reproduces_the_path_without_it_bit_for_bit(model, scen, envp, starts):
    """Check 1: the EXTF instances with a zero record give the records, obs, reward and done of external_forces = 0 byte
    for byte, alone and together with ENVP rows."""
    from emu_envp import EmuEnvpWarp4
    from emu_extf import EmuExtfWarp4

    n = SCENARIOS[scen][0]
    rows = None
    if envp:
        from emu_envp import EmuEnvpEnv

        rng = np.random.default_rng(3)
        rows = np.stack([_random_env_row(rng, EmuEnvpEnv(model.blob()).default_env_params()) for _ in range(n)])
    a, _ = _run(model, scen, starts, EmuEnvpWarp4, rows=rows)
    b, wb = _run(model, scen, starts, EmuExtfWarp4, wrench=np.zeros((n, 26, 6), np.float32), rows=rows)
    _equal(a, b)
    if scen == "packed_4warp":
        assert wb.env.packed_rounds() > 0
    if scen.startswith("standing"):
        assert wb.env.heavy_solves() > 0


def _kat_model(model):
    return with_params(model, gravity=0.0, linear_damping=0.0, angular_damping=0.0)


def test_oracle_wrench_changes_momentum_as_newton_says(model):
    """Check 2 (oracle KATs), one substep from rest, gravity, damping, motors and contacts off:
    linear momentum changes by dt sum F (1e-9 relative) for random wrenches; angular momentum about the world origin by
    dt sum (c_b x F_b + T_b) within an O(dt) bound, for a uniform field F_b = m_b a (sum c_b x F_b = M c x a) plus random
    torques."""
    from oracle_extf import OracleExtf

    m = _kat_model(model)
    dt = m.meta["params"]["time_step"] / 5
    rng = np.random.default_rng(2)
    o = OracleExtf(m.blob(), contacts=False)
    o.reset()
    s0 = o.get_state()
    s0[7:13] = 0.0
    s0[38:88] = 0.0
    target = s0[13:38].copy()  # dof order
    def momentum_after(w):
        """momentum at the starting configuration with the velocities after one substep under w (the momentum of the
        velocity change; the configuration's own change within the substep would add a term of order dt^2)"""
        o.set_state(s0)
        o.set_external_forces(link_wrenches(m, w))
        o.substep(target, 0.0)
        s1 = s0.copy()
        s1[7:13] = o.get_state()[7:13]
        s1[38:63] = o.get_state()[38:63]
        o.set_state(s1)
        return o.momentum()

    o.set_state(s0)
    p0 = o.momentum()
    for trial in range(3):
        w = _random_wrenches(rng, model).astype(np.float64)
        p1 = momentum_after(w)
        dP = p1["P"] - p0["P"]
        ref = dt * w[:, :3].sum(axis=0)
        assert np.abs(dP - ref).max() <= 1e-9 * np.abs(ref).max(), (dP, ref)
        # uniform field + random torques
        a = rng.normal(size=3) * 2.0
        w2 = w.copy()
        w2[:, :3] = _body_mass(m)[:, None] * a[None, :]
        p1 = momentum_after(w2)
        refL = dt * (p0["mass"] * np.cross(p0["com"], a) + w2[:, 3:].sum(axis=0))
        assert np.abs(p1["L"] - p0["L"] - refL).max() <= 10 * dt * np.abs(refL).max(), (p1["L"] - p0["L"], refL)
    o.set_external_forces(None)


def test_oracle_variant_without_wrench_is_the_oracle(model, action_limits):
    """The oracle built with the wrench input (tests/emu/oracle_extf.py) steps exactly as the oracle does while no wrench is
    set, and a wrench set to zero changes nothing either."""
    from oracle.oracle import Oracle
    from oracle_extf import OracleExtf

    lo, hi = action_limits
    rng = np.random.default_rng(13)
    a, b = Oracle(model.blob()), OracleExtf(model.blob())
    c = OracleExtf(model.blob())
    c.set_external_forces(np.zeros((int(model["full_n_links"][0]) + 1, 6)))
    assert np.array_equal(a.reset(), b.reset()) and np.array_equal(a.reset(), c.reset())
    for t in range(6):
        act = rng.uniform(lo, hi)
        for o in (a, b, c):
            o.step(act)
        assert np.array_equal(a.get_state(), b.get_state()) and np.array_equal(a.get_state(), c.get_state()), t


def test_link_wrenches_reproduce_the_body_wrench(model):
    """Check 2: the links' forces sum to the body force and their moments about the body COM to the body torque (1e-12)."""
    rng = np.random.default_rng(4)
    w = _random_wrenches(rng, model).astype(np.float64)
    lw = link_wrenches(model, w)
    tb = np.asarray(model["mb_task_body"])
    mass = np.asarray(model["full_mass"])
    # the split is by mass share, so the moment of the link forces about the body COM is
    # sum_l (m_l / m_b) (x_l - c_b) x F = 0 (the mass-weighted link COMs average to c_b): the body torque is all there is
    for k in range(26):
        b = k + 1 if k < 25 else 0
        links = tb == b
        assert np.abs(lw[links, :3].sum(axis=0) - w[k, :3]).max() <= 1e-12 * max(np.abs(w[k, :3]).max(), 1.0)
        assert np.abs(lw[links, 3:].sum(axis=0) - w[k, 3:]).max() <= 1e-12 * max(np.abs(w[k, 3:]).max(), 1.0)
        share = mass[links] / mass[links].sum()
        assert np.allclose(lw[links, :3], share[:, None] * w[k, :3][None, :], rtol=1e-12, atol=0)
    assert np.isclose(mass.sum(), np.asarray(model["mb_mass"]).sum(), rtol=1e-12)
    assert lw.shape == (int(model["full_n_links"][0]) + 1, 6)
    with pytest.raises(ValueError):
        link_wrenches(model, np.zeros((25, 6)))


def _rest_state(o):
    s = o.get_state()
    s[7:13] = 0.0
    s[38:88] = 0.0
    return s


def test_gravity_cancellation(model):
    """Check 3: F_b = m_b g z on every body, from rest at the reset pose with the motor targets at that pose: the oracle's
    velocities stay below 1e-12, the emulator's below 1e-4 over 50 steps."""
    from emu_extf import EmuExtfEnv
    from oracle_extf import OracleExtf

    mb = _body_mass(model)
    w = np.zeros((26, 6))
    w[:, 2] = mb * model.meta["params"]["gravity"]
    obs_dof = np.asarray(model["obs_dof"])
    o = OracleExtf(model.blob())
    o.reset()
    s = _rest_state(o)
    o.set_state(s)
    o.set_external_forces(link_wrenches(model, w))
    act = s[13:38][obs_dof]
    for t in range(10):
        o.step(act)
        st = o.get_state()
        assert np.abs(st[7:13]).max() < 1e-12 and np.abs(st[38:63]).max() < 1e-12, t
    e = EmuExtfEnv(model.blob())
    e.set_external_forces(w.astype(np.float32))
    e.reset()
    e.rec[7:13] = 0.0
    e.rec[38:63] = 0.0
    act32 = e.rec[13:38][obs_dof].copy()
    for t in range(50):
        e.step(act32)
        assert np.abs(e.rec[7:13]).max() < 1e-4 and np.abs(e.rec[38:63]).max() < 1e-4, (t, np.abs(e.rec[38:63]).max())


def test_uniform_field_equals_changed_gravity(model):
    """Check 4: F_b = m_b (0, 0, d) on the emulator matches the emulator on with_params(gravity = g - d) over 20 env steps,
    each from the same state, within 1e-5 relative (independent of the oracle).  The two paths round differently -- the
    wrench is m_b d in FP32 rotated as a force, gravity m (g Rw) -- and the motor solve ends on a residual threshold, so
    last-bit differences of its inputs show at the solver's tolerance (measured: 5.6e-6 at most)."""
    from emu import EmuEnv
    from emu_extf import EmuExtfEnv

    d = 2.5
    g = model.meta["params"]["gravity"]
    w = np.zeros((26, 6), np.float32)
    w[:, 2] = (_body_mass(model) * d).astype(np.float32)
    a = EmuExtfEnv(model.blob(), contacts=False)
    a.set_external_forces(w)
    b = EmuEnv(with_params(model, gravity=g - d).blob(), contacts=False)
    a.reset()
    b.reset()
    rng = np.random.default_rng(6)
    worst = 0.0
    for t in range(20):
        b.rec[:] = a.rec  # (the reset steps differ too: a reset takes no wrench)
        act = rng.uniform(-1.0, 1.0, 25).astype(np.float32)
        a.step(act)
        b.step(act)
        worst = max(worst, max(rel_err(b.rec[sl], a.rec[sl]) for sl in STATE_BLOCKS.values()))
    assert worst < 1e-5, worst


def _oracle_parity(model, e, o, w_model, rng, lo, hi, steps, substeps):
    errs, n_contact = [], 0
    a = rng.uniform(lo, hi)
    for t in range(steps):
        if t % 5 == 0:
            a = rng.uniform(lo, hi)
        o.set_state(e.get_state(o.num_candidates))
        o.step(a)
        e.step(a)
        so, se = o.get_state(), e.get_state(o.num_candidates)
        errs.append(max(rel_err(so[sl], se[sl]) for sl in STATE_BLOCKS.values()))
        n_contact += o.last_num_contacts > 0
    return np.asarray(errs), n_contact


@pytest.mark.parametrize("envp", [False, True], ids=["wrench", "wrench_and_env_params"])
def test_random_wrenches_contact_free_match_the_oracle(model, action_limits, envp):
    """Check 5 (contact-free): random wrenches (forces up to ~0.3 m_b g, torques), per env step < 2e-5 against the oracle fed
    link_wrenches; one case together with a random ENVP row (the oracle on the correspondingly modified model)."""
    from emu_envp import EmuEnvpEnv
    from emu_extf import EmuExtfEnv
    from oracle_extf import OracleExtf
    from test_env_params import _model_of_row

    lo, hi = action_limits
    rng = np.random.default_rng(7)
    w = _random_wrenches(rng, model)
    e = EmuExtfEnv(model.blob(), contacts=False)
    ref = model
    if envp:
        r = _random_env_row(rng, EmuEnvpEnv(model.blob()).default_env_params())
        e.set_env_params(r)
        ref = _model_of_row(model, r)
    e.set_external_forces(w)
    o = OracleExtf(ref.blob(), contacts=False)
    o.set_external_forces(link_wrenches(ref, w.astype(np.float64)))
    e.reset()
    errs, _ = _oracle_parity(model, e, o, ref, rng, lo, hi, 20, 5)
    assert errs.max() < 2e-5, errs.max()


def test_random_wrenches_with_contacts_match_the_oracle(model, action_limits):
    """Check 5 (contacts): single substeps against the oracle, p50 < 2e-5 and p99 < 2e-3 (the env-params bounds)."""
    from emu_extf import EmuExtfEnv
    from oracle_extf import OracleExtf

    lo, hi = action_limits
    rng = np.random.default_rng(8)
    sub = with_params(model, time_step=0.002, solver_iterations=60)
    w = _random_wrenches(rng, model, scale=0.1)
    e = EmuExtfEnv(sub.blob(), num_substeps=1, deferred=1)
    e.set_external_forces(w)
    o = OracleExtf(sub.blob(), num_substeps=1)
    o.set_external_forces(link_wrenches(sub, w.astype(np.float64)))
    e.reset()
    errs, n_contact = _oracle_parity(model, e, o, sub, rng, lo, hi, 220, 1)
    assert n_contact > 60
    assert np.percentile(errs, 50) < 2e-5 and np.percentile(errs, 99) < 2e-3, (np.percentile(errs, [50, 99]), errs.max())


# ---- push schedule -------------------------------------------------------------------------------------------------
def push_directions():
    return np.array([[math.cos(2 * math.pi * k / 32), math.sin(2 * math.pi * k / 32)] for k in range(32)]).astype(np.float32)


def reference_push(seed, gid, episode, step, interval, duration, probability, fmin, fmax, first_step):
    """The schedule in numpy (include/trex_b200.h trex_set_push_schedule): (fx, fy) or None."""
    from test_emulator_parity import _philox4x32_10

    t = int(step)
    if t < first_step:
        return None
    w = t // interval
    u0, u1, u2, u3 = _philox4x32_10([gid & 0xFFFFFFFF, gid >> 32, int(episode), w], [seed, PUSH_KEY])
    if not u0 < np.float32(probability):
        return None
    span = interval - duration
    o = min(int(np.float32(u1) * np.float32(span + 1)), span)
    r = t - w * interval
    if r < o or r >= o + duration:
        return None
    # force_min + u2 (force_max - force_min) as one fused multiply-add: exact in double for the forces used here
    # (force_max - force_min a power of two), then rounded once
    mag = np.float32(np.float64(u2) * np.float64(np.float32(np.float32(fmax) - np.float32(fmin))) + np.float64(np.float32(fmin)))
    d = push_directions()[int(np.float32(u3) * np.float32(32))]
    return np.float32(mag * d[0]), np.float32(mag * d[1])


SCHED = dict(interval=7, duration=3, probability=0.75, force=(3000.0, 3000.0 + 4096.0), first_step=2)


def _schedule_kw():
    return dict(interval=SCHED["interval"], duration=SCHED["duration"], probability=SCHED["probability"],
                fmin=SCHED["force"][0], fmax=SCHED["force"][1], first_step=SCHED["first_step"])


def test_schedule_equals_the_record_set_to_the_reference_pushes(model):
    """Check 6: record zero + schedule on == schedule off + record set to the numpy reference's push every step, byte for
    byte, over episodes that end (auto-reset) inside push windows and start before first_step."""
    from emu_extf import EmuExtfWarp4

    seed, env0, n, body = 9, 1000, 4, BASE
    kw = dict(max_episode_steps=9, seed=seed, env_id=env0, contacts=False)
    a = EmuExtfWarp4(model.blob(), n=n, **kw)
    a.env.set_external_forces(np.zeros((n, 26, 6), np.float32))
    a.env.set_push_schedule(body=body, **SCHED)
    b = EmuExtfWarp4(model.blob(), n=n, **kw)
    b.env.set_external_forces(np.zeros((n, 26, 6), np.float32))
    a.reset()
    b.reset()
    rng = np.random.default_rng(1)
    pushed = resets = 0
    for t in range(30):
        act = rng.uniform(-1.0, 1.0, (n, 25)).astype(np.float32)
        w = np.zeros((n, 26, 6), np.float32)
        for e in range(n):
            p = reference_push(seed, env0 + e, b.rec[e, 153], b.rec[e, 152], **_schedule_kw())
            if p is not None:
                w[e, body, 0], w[e, body, 1] = p
                pushed += 1
        b.env.set_external_forces(w)
        oa, ra, da = a.step(act)
        ob, rb, db = b.step(act)
        assert np.array_equal(_bytes(a.rec), _bytes(b.rec)) and np.array_equal(_bytes(oa), _bytes(ob)), t
        resets += int(db.sum())
    assert pushed > 10 and resets >= n  # pushes happened, and episodes ended inside the schedule
    # a reset inside a push window: the reset step takes no wrench (episode 1 starts at step 0 < first_step anyway)
    assert np.array_equal(_bytes(a.rec[:, 152:154]), _bytes(b.rec[:, 152:154]))


def test_schedule_reference_properties():
    """The reference's pushes: magnitude within [lo, hi], one push of `duration` steps per pushing window, none before
    first_step, the probability respected roughly."""
    kw = _schedule_kw()
    windows_with, windows = 0, 0
    for gid in range(200):
        steps = [t for t in range(7 * 10) if reference_push(5, gid, 0, t, **kw) is not None]
        for w in range(10):
            inw = [t for t in steps if t // 7 == w]
            windows += 1
            if inw:
                windows_with += 1
                assert inw == list(range(inw[0], inw[0] + len(inw)))
                assert len(inw) == 3 or (w == 0 and inw[0] == 2)
        assert all(t >= 2 for t in steps)
        for t in steps:
            fx, fy = reference_push(5, gid, 0, t, **kw)
            assert 3000.0 * 0.9999 <= math.hypot(fx, fy) <= 7096.0 * 1.0001
    assert 0.65 < windows_with / windows < 0.85


BAD_SCHEDULES = {
    "body_negative": dict(body=-1),
    "body_26": dict(body=26),
    "interval_0": dict(interval=0),
    "duration_0": dict(duration=0),
    "duration_above_interval": dict(interval=5, duration=6),
    "first_step_negative": dict(first_step=-1),
    "probability_above_1": dict(probability=1.5),
    "probability_nan": dict(probability=float("nan")),
    "force_negative": dict(force=(-1.0, 10.0)),
    "force_lo_above_hi": dict(force=(20.0, 10.0)),
    "force_inf": dict(force=(0.0, float("inf"))),
}


@pytest.mark.parametrize("bad", list(BAD_SCHEDULES))
def test_bad_schedules_are_rejected(model, bad):
    """Check 7: the host validation shared by the library and the emulator (trex_model.h check_push_schedule)."""
    from emu_extf import EmuExtfEnv

    e = EmuExtfEnv(model.blob())
    good = dict(body=BASE, interval=10, duration=2, probability=0.5, force=(0.0, 100.0), first_step=0)
    e.set_push_schedule(**good)
    with pytest.raises(ValueError):
        e.set_push_schedule(**dict(good, **BAD_SCHEDULES[bad]))


def test_calls_without_a_handle_are_invalid():
    """Check 7 (C ABI, no GPU needed): the three calls refuse a NULL handle; the config struct keeps its size."""
    from trex_gym_b200 import _native

    L = _native.lib()
    buf = (ctypes.c_float * (26 * 6))()
    s = _native.TrexPushSchedule(body=25, interval=10, duration=2, probability=0.5, force_min=0.0, force_max=1.0)
    assert L.trex_set_external_forces(None, ctypes.addressof(buf), None, None) == -1
    assert L.trex_get_external_forces(None, ctypes.addressof(buf), None) == -1
    assert L.trex_set_push_schedule(None, ctypes.byref(s)) == -1
    assert ctypes.sizeof(_native.TrexConfig) == 96 and ctypes.sizeof(_native.TrexPushSchedule) == 64


def test_body_com_table(model):
    """The COM table the kernels read is mc / mass of each merged body, in wrench-record order."""
    from emu_extf import EmuExtfEnv

    com = EmuExtfEnv(model.blob()).body_com()
    mc = np.asarray(model["mb_mc"]).reshape(-1, 3)
    m = np.asarray(model["mb_mass"])
    ref = np.concatenate([mc[1:] / m[1:, None], mc[:1] / m[:1, None]]).astype(np.float32)
    assert np.array_equal(com, ref)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _sim(n, **kw):
    from trex_gym_b200.sim import TrexBatchSim

    return TrexBatchSim(n, device=0, **kw)


def _hold_actions(sim):
    import torch

    return torch.tensor(_hold(sim.model), device=sim.device).repeat(sim.num_envs, 1).contiguous()


def _bytes_equal(a, b):
    return np.array_equal(a.cpu().numpy().view(np.uint8), b.cpu().numpy().view(np.uint8))


GPU_CONFIGS = {
    "random": (1024, {}, "random"),
    "warps_per_block_1": (1024, {"warps_per_block": 1}, "random"),
    "warps_per_block_4": (1024, {"warps_per_block": 4}, "random"),
    "front_solve": (512, {"deferred_solve": False}, "random"),
    "free_only": (512, {"defer_contacts": False}, "random"),
    "contact_memory_shared": (1024, {"contact_memory": 1}, "random"),
    "heavy_memory_shared": (512, {"heavy_memory": 1}, "standing"),
    "heavy_memory_tensor": (512, {"heavy_memory": 2}, "standing"),
    "env_params": (1024, {"env_params": True}, "random"),
    "env_params_warps_per_block_4": (512, {"env_params": True, "warps_per_block": 4}, "standing"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", list(GPU_CONFIGS))
def test_gpu_zero_record_matches_external_forces_off(cfg):
    """GPU check 1: external_forces = 1 with a zero record gives the obs, reward, done and state of external_forces = 0
    byte for byte."""
    n, kw, acts = GPU_CONFIGS[cfg]
    a, b = _sim(n, **kw), _sim(n, external_forces=True, **kw)
    assert float(b.get_external_forces().abs().max()) == 0.0
    steps = 16 if acts == "standing" else 6
    for t in range(steps):
        act = _hold_actions(a) if acts == "standing" else a.random_actions(step=t)
        oa, ra, da = [x.clone() for x in a.step(act)]
        ob, rb, db = b.step(act)
        assert _bytes_equal(oa, ob) and _bytes_equal(ra, rb) and _bytes_equal(da, db), (cfg, t)
    assert _bytes_equal(a.get_state(), b.get_state()), cfg


@pytest.mark.gpu
def test_gpu_graph_capture_with_external_forces():
    a, b = _sim(1024), _sim(1024, external_forces=True)
    for t in range(3):
        act = a.random_actions(step=t)
        oa = a.step_graph(act)[0].clone()
        ob = b.step_graph(act)[0]
        assert _bytes_equal(oa, ob), t
    assert _bytes_equal(a.get_state(), b.get_state())


@pytest.mark.gpu
def test_gpu_random_wrenches_match_the_oracle(model):
    """GPU check 2: 4,096 environments with random wrenches, 64 checked per step against the oracle fed link_wrenches."""
    import torch
    from oracle_extf import OracleExtf

    n, rng = 4096, np.random.default_rng(12)
    b = _sim(n, external_forces=True)
    w = _random_wrenches(rng, model, n=n)
    b.set_external_forces(torch.from_numpy(w[:, :, :3]), torch.from_numpy(w[:, :, 3:]))
    assert np.array_equal(b.get_external_forces().cpu().numpy(), w)
    b.reset()
    check = list(range(0, n, n // 64))
    oracles = {}
    for e in check:
        oracles[e] = OracleExtf(model.blob())
        oracles[e].set_external_forces(link_wrenches(model, w[e].astype(np.float64)))
    nc = next(iter(oracles.values())).num_candidates
    free, contact = [], []
    for t in range(16):
        pre = b.get_state().cpu().numpy()
        act = b.random_actions(step=t)
        b.step(act)
        post = b.get_state().cpu().numpy()
        acts = act.cpu().numpy().astype(np.float64)
        for e in check:
            o = oracles[e]
            o.set_state(np.concatenate([pre[e, :88], pre[e, 88:88 + nc]]).astype(np.float64))
            o.step(acts[e])
            so = o.get_state()
            err = max(rel_err(so[sl], post[e, :88 + nc][sl]) for sl in STATE_BLOCKS.values())
            (contact if o.last_num_contacts else free).append(err)
    assert len(free) > 0 and np.percentile(free, 99) < 2e-5 and max(free) < 5e-5, (np.percentile(free, 99), max(free))
    if contact:  # whole env steps (5 substeps) in contact: the bound of the env-params GPU test
        assert np.percentile(contact, 50) < 1e-3 and np.percentile(contact, 99) < 2e-2, np.percentile(contact, [50, 99])


@pytest.mark.gpu
def test_gpu_schedule_equals_reference_pushes_and_shards(model):
    """GPU check 3: schedule on == record set to the reference pushes (the pushes the emulator applies, see the CPU test)
    byte for byte; two shards (env_offset 0 and N/2) equal one handle of N."""
    import torch

    seed, n, body = 21, 256, BASE
    kw = dict(seed=seed, max_episode_steps=9)
    a = _sim(n, external_forces=True, **kw)
    a.set_push_schedule("base", **SCHED)
    b = _sim(n, external_forces=True, **kw)
    shards = [_sim(n // 2, external_forces=True, env_offset=k * n // 2, **kw) for k in range(2)]
    for s in shards:
        s.set_push_schedule("base", **SCHED)
    pushed = 0
    for t in range(24):
        rec = b.get_state().cpu().numpy()
        f = np.zeros((n, 26, 3), np.float32)
        for e in range(n):
            p = reference_push(seed, e, rec[e, 153], rec[e, 152], **_schedule_kw())
            if p is not None:
                f[e, body, 0], f[e, body, 1] = p
                pushed += 1
        b.set_external_forces(torch.from_numpy(f))
        act = a.random_actions(step=t)
        oa = a.step(act)[0].clone()
        ob = b.step(act)[0].clone()
        assert _bytes_equal(oa, ob), t
        os_ = torch.cat([s.step(act[k * n // 2:(k + 1) * n // 2].contiguous())[0].clone() for k, s in enumerate(shards)])
        assert _bytes_equal(oa, os_), t
    assert pushed > 100
    assert _bytes_equal(a.get_state(), b.get_state())
    assert _bytes_equal(a.get_state(), torch.cat([s.get_state() for s in shards]))


@pytest.mark.gpu
def test_gpu_masked_set_get_round_trip(model):
    """GPU check 3: a masked set replaces every wrench of the masked environments and leaves the others untouched; named
    bodies land in their slots; clear zeroes."""
    import torch

    n = 300
    s = _sim(n, external_forces=True)
    rng = np.random.default_rng(5)
    w0 = _random_wrenches(rng, model, n=n)
    s.set_external_forces(torch.from_numpy(w0[:, :, :3]), torch.from_numpy(w0[:, :, 3:]))
    w1 = _random_wrenches(rng, model, n=n)
    mask = torch.zeros(n, dtype=torch.uint8)
    mask[::7] = 1
    s.set_external_forces(torch.from_numpy(w1[:, :, :3]), torch.from_numpy(w1[:, :, 3:]), mask=mask)
    got = s.get_external_forces().cpu().numpy()
    m = mask.numpy().astype(bool)
    assert np.array_equal(got[m], w1[m]) and np.array_equal(got[~m], w0[~m])
    names = s.model.meta["body_joint_names"]
    f = torch.ones(n, 2, 3)
    s.set_external_forces(f, bodies=["base", names[3]])
    got = s.get_external_forces().cpu().numpy()
    assert np.all(got[:, BASE, :3] == 1.0) and np.all(got[:, 2, :3] == 1.0) and np.all(got[:, :, 3:] == 0.0)
    assert np.count_nonzero(got) == n * 6
    s.clear_external_forces()
    assert float(s.get_external_forces().abs().max()) == 0.0
    assert s.body_com().shape == (26, 3)
    with pytest.raises(ValueError):
        s.set_external_forces(torch.ones(n, 25, 3))
    with pytest.raises(ValueError):
        s.set_push_schedule("base", interval=5, duration=6)
    s.set_push_schedule(None)
    off = _sim(8)
    with pytest.raises(ValueError):
        off.set_external_forces(torch.zeros(8, 26, 3))
    from trex_gym_b200 import _native

    buf = torch.zeros(8, 26, 6, device=off.device)
    L = _native.lib()
    assert L.trex_set_external_forces(off._h, ctypes.c_void_p(buf.data_ptr()), None, None) == -1
    assert L.trex_get_external_forces(off._h, ctypes.c_void_p(buf.data_ptr()), None) == -1
    assert L.trex_set_push_schedule(off._h, None) == -1
    cfg = _native.TrexConfig()
    cfg.external_forces = 2
    h = ctypes.c_void_p()
    blob = s.model.blob()
    assert L.trex_create(blob, len(blob), 8, 0, ctypes.byref(cfg), ctypes.byref(h)) == -1


@pytest.mark.gpu
def test_gpu_vec_env_pushes_move_a_standing_batch():
    """GPU check 4: TrexVecEnv(pushes=...) runs with auto-reset; over the same steps a standing batch pushed on the base
    moves its base clearly further horizontally than the same batch unpushed.  The batch first lands and settles (60
    steps, no push before first_step); displacements are measured from there to the last step of the episode, and the run
    continues through the auto-reset at the horizon.  The unpushed batch is not at rest (it sways on its feet), so the
    pushes are also measured against it environment by environment: both runs are deterministic, so every difference
    between them is the pushes' doing."""
    from trex_gym_b200.trex_env import TrexVecEnv

    n, settle, horizon = 256, 60, 150
    pushes = dict(body="base", interval=30, duration=10, probability=1.0, force=(1.0e4, 2.0e4), first_step=settle)
    runs = {}
    for name, p in (("pushed", pushes), ("still", None)):
        env = TrexVecEnv(n, max_episode_steps=horizon, pushes=p)
        env.reset()
        hold = _hold_actions(env.sim)
        dones = 0
        for t in range(horizon + 10):
            obs, rew, done, _ = env.step(hold)
            dones += int(done.sum())
            assert bool(obs.isfinite().all())
            if t == settle - 1:
                x0 = env.sim.get_state()[:, 0:2].clone()
            if t == horizon - 2:  # the last step of the episode before the auto-reset
                x1 = env.sim.get_state()[:, 0:2].clone()
        runs[name] = (x0, x1, dones)
        env.close()
    assert runs["pushed"][2] == n and runs["still"][2] == n  # every environment auto-reset once, at the horizon
    moved = {k: float((v[1] - v[0]).norm(dim=1).median()) for k, v in runs.items()}
    apart = float((runs["pushed"][1] - runs["still"][1]).norm(dim=1).median())
    # (measured on a B200: medians 0.258 m pushed, 0.214 m unpushed, 0.111 m between the two runs of an environment)
    assert moved["pushed"] > moved["still"] and apart > 0.05, (moved, apart)
