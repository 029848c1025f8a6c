"""Per-environment dynamics parameters (trex_config.env_params = 1): mass scales, friction, motor gains and strength per
environment, and the randomizer that draws them at every reset.

CPU (the product kernel source through tests/emu): the ENVP instances against the env_params = 0 path on the same or on a
correspondingly modified model blob, and against the oracle.  GPU (-m gpu): the library's ENVP kernels."""
import ctypes

import numpy as np
import pytest

from conftest import STATE_BLOCKS, rel_err
from trex_gym_b200.model_compiler import with_body_mass_scale, with_params

FEMUR = 0  # row element of joint_femur_right's body (meta["body_joint_names"][1])


def _states(model, n, rng):
    """n perturbed reset states: joints off the crouch (some limits violated), the later ones on / near the floor."""
    from emu import EmuWarp4

    w = EmuWarp4(model.blob(), n=n)
    w.reset()
    qlo, qhi = model["mb_lower"][1:], model["mb_upper"][1:]
    rec = w.rec.copy()
    for e in range(n):
        rec[e, 13:38] = np.clip(rec[e, 13:38] + rng.uniform(-0.3, 0.3, 25), qlo - 0.02, qhi + 0.02)
        rec[e, 2] -= 0.12 * e
    return rec


def _hold(model):
    names = list(model.meta["obs_joint_names"])
    hold = np.zeros(25, np.float32)
    for k, v in model.meta["starting_configuration"].items():
        hold[names.index(k)] = v
    return hold


# scenario: (n envs, emulator flags, EmuEnv kwargs, steps, start); flags as tests/emu/emu_main.cpp emu_set_deferred
SCENARIOS = {
    "contact": (4, 1, {}, 10, "perturbed"),
    "contact_solve4_shared_memory": (4, 1, {}, 8, "perturbed"),
    "contact_solve4_tensor_memory": (4, 1 | 64, {}, 8, "perturbed"),
    "packed_4warp": (4, 1 | 8, {}, 8, "perturbed"),
    "front_solve": (4, 0, {}, 6, "perturbed"),
    "contact_free": (4, 1, {"contacts": False}, 8, "perturbed"),
    "fallen_start": (4, 1, {"reset_mode": 1, "seed": 3, "max_episode_steps": 3}, 8, "reset"),
    "standing_solve2_shared_memory": (3, 1, {}, 50, "standing"),
    "standing_solve2_tensor_memory": (3, 1 | 32, {}, 50, "standing"),
}


def _run(blob, scen, rows=None, steps=None, start=None, model=None, seed=0):
    """Steps one emulated work unit (without rows: the existing emulator, the env_params = 0 path); returns the list of (rec, obs, reward, done) after every step (and the reset)."""
    from emu import EmuWarp4
    from emu_envp import EmuEnvpWarp4

    n, flags, kw, nsteps, how = SCENARIOS[scen]
    w = (EmuWarp4 if rows is None else EmuEnvpWarp4)(blob, n=n, deferred=flags, **kw)
    if rows is not None:
        w.env.set_env_params(rows)
    obs0 = w.reset()
    out = [(w.rec.copy(), obs0)]
    if how == "perturbed":
        w.rec[:] = start
    rng = np.random.default_rng(seed)
    hold = _hold(model)
    lo, hi = model["mb_lower"][1:], model["mb_upper"][1:]
    names = list(model.meta["obs_joint_names"])
    for t in range(steps or nsteps):
        if how == "standing":
            acts = np.stack([hold + rng.uniform(-0.02, 0.02, 25) * (e > 0) for e in range(n)]).astype(np.float32)
        else:
            acts = rng.uniform(-1.0, 1.0, (n, 25)).astype(np.float32)
        obs, rew, done = w.step(acts)
        out.append((w.rec.copy(), obs.copy(), rew.copy(), done.copy(), w.aux.copy()))
    return out, w


def _equal(a, b, envs=None):
    for t, (x, y) in enumerate(zip(a, b)):
        for k, (u, v) in enumerate(zip(x, y)):
            u, v = (u, v) if envs is None else (np.atleast_1d(u[envs]), np.atleast_1d(v[envs]))
            assert np.array_equal(np.ascontiguousarray(u).view(np.uint8), np.ascontiguousarray(v).view(np.uint8)), (t, k)


@pytest.fixture(scope="module")
def starts(model):
    return _states(model, 4, np.random.default_rng(11))


@pytest.mark.parametrize("scen", list(SCENARIOS))
def test_default_rows_reproduce_the_uniform_path_bit_for_bit(model, scen, starts):
    """Check 1: the ENVP instances with the default row give the records, obs, reward and done of the env_params = 0 path
    byte for byte (same operations in the same order; x * 1.0 is exact, also under FMA contraction)."""
    from emu_envp import EmuEnvpEnv

    n = SCENARIOS[scen][0]
    row = EmuEnvpEnv(model.blob()).default_env_params()
    a, wa = _run(model.blob(), scen, start=starts[:n], model=model)
    b, wb = _run(model.blob(), scen, rows=np.tile(row, (n, 1)), start=starts[:n], model=model)
    _equal(a, b)
    if scen.startswith("standing"):
        assert wb.env.heavy_solves() > 0  # solve2 ran
    if scen == "packed_4warp":
        assert wb.env.packed_rounds() > 0


def _rows_and_models(model, default):
    """Four rows (default; float-exact friction / gains / torque; power-of-two mass scales; both) and the blobs that
    the env_params = 0 path must reproduce them with."""
    p = default.copy()
    p[26], p[27], p[29] = 0.5, 0.01, 2.0e5
    m = default.copy()
    m[25], m[FEMUR] = 2.0, 0.5
    pm = p.copy()
    pm[:26] = m[:26]
    pmodel = with_params(model, friction=0.5, motor_kp=0.01, motor_max_torque=2.0e5)
    return [default, p, m, pm], [model, pmodel, with_body_mass_scale(model, m[:26]), with_body_mass_scale(pmodel, m[:26])]


@pytest.mark.parametrize("scen", ["contact", "packed_4warp", "contact_solve4_tensor_memory", "standing_solve2_shared_memory"])
def test_rows_equal_modified_models_bit_for_bit(model, scen, starts):
    """Checks 2 and 3: four environments of one work unit carry four different rows; each equals, byte for byte, the
    env_params = 0 path on the model with those values (friction / kp / torque through with_params, mass scales of 2 and
    0.5 -- exact in FP32 -- through with_body_mass_scale)."""
    from emu_envp import EmuEnvpEnv

    n = SCENARIOS[scen][0]
    rows, models = _rows_and_models(model, EmuEnvpEnv(model.blob()).default_env_params())
    b, _ = _run(model.blob(), scen, rows=np.stack(rows[:n]), start=starts[:n], model=model)
    for e in range(n):
        a, _ = _run(models[e].blob(), scen, start=starts[:n], model=model)
        _equal(a, b, envs=e)
    # and the rows do change the dynamics
    assert not np.array_equal(b[-1][0][0], b[-1][0][2])


def _random_row(rng, default):
    r = default.copy()
    r[:26] = rng.uniform(0.8, 1.25, 26)
    r[26] = rng.uniform(0.15, 0.5)
    r[27] = default[27] * rng.uniform(0.8, 1.25)
    r[28] = default[28] * rng.uniform(0.8, 1.25)
    r[29] = default[29] * rng.uniform(0.7, 1.0)
    return r.astype(np.float32)


def _model_of_row(model, r):
    return with_params(with_body_mass_scale(model, r[:26].astype(np.float64)), friction=float(r[26]), motor_kp=float(r[27]),
                       motor_kd=float(r[28]), motor_max_torque=float(r[29]))


def test_random_rows_contact_free_match_the_oracle(model, action_limits):
    """Check 4 (contact-free): a random row (non-power-of-two mass scales) against the oracle on the modified model,
    per env step < 2e-5."""
    from emu_envp import EmuEnvpEnv
    from oracle.oracle import Oracle

    lo, hi = action_limits
    rng = np.random.default_rng(4)
    e = EmuEnvpEnv(model.blob(), contacts=False)
    r = _random_row(rng, e.default_env_params())
    e.set_env_params(r)
    o = Oracle(_model_of_row(model, r).blob(), contacts=False)
    e.reset()
    worst = 0.0
    for t in range(20):
        a = rng.uniform(lo, hi)
        o.set_state(e.get_state(o.num_candidates))
        o.step(a)
        e.step(a)
        so, se = o.get_state(), e.get_state(o.num_candidates)
        worst = max(worst, max(rel_err(so[sl], se[sl]) for sl in STATE_BLOCKS.values()))
    assert worst < 2e-5, worst


def test_random_rows_with_contacts_match_the_oracle(model, action_limits):
    """Check 4 (contacts): single substeps of a random row against the oracle on the modified model, within the
    percentile bounds of test_per_substep_parity_with_contacts."""
    from emu_envp import EmuEnvpEnv
    from oracle.oracle import Oracle

    lo, hi = action_limits
    rng = np.random.default_rng(5)
    sub = with_params(model, time_step=0.002, solver_iterations=60)
    e = EmuEnvpEnv(sub.blob(), num_substeps=1, deferred=1)
    r = _random_row(rng, e.default_env_params())
    e.set_env_params(r)
    o = Oracle(_model_of_row(sub, r).blob(), num_substeps=1)
    e.reset()
    errs, n_contact = [], 0
    a = rng.uniform(lo, hi)
    for t in range(220):
        if t % 5 == 0:
            a = rng.uniform(lo, hi)
        o.set_state(e.get_state(o.num_candidates))
        o.step(a)
        e.step(a)
        so, se = o.get_state(), e.get_state(o.num_candidates)
        errs.append(max(rel_err(so[sl], se[sl]) for sl in STATE_BLOCKS.values()))
        n_contact += o.last_num_contacts > 0
    errs = np.asarray(errs)
    assert n_contact > 60
    assert np.percentile(errs, 50) < 2e-5 and np.percentile(errs, 99) < 2e-3, (np.percentile(errs, 50), errs.max())


def _ranges(default):
    lo, hi = default.copy(), default.copy()
    lo[:26], hi[:26] = 0.8, 1.25
    lo[26], hi[26] = 0.15, 0.5
    lo[27], hi[27] = default[27] * 0.8, default[27] * 1.25
    lo[29], hi[29] = default[29] * 0.7, default[29]
    lo[30:], hi[30:] = 0.0, 0.0
    return lo.astype(np.float32), hi.astype(np.float32)


def _philox_rows(lo, hi, seed, gid, episode, dt):
    """Reference of the randomizer: Philox4x32-10, key (seed, 0xe9a5), counter (gid lo, gid hi, episode, block)."""
    from test_emulator_parity import _philox4x32_10

    u = np.zeros(32, np.float32)
    for b in range(8):
        c = _philox4x32_10([gid & 0xFFFFFFFF, gid >> 32, episode, b], [seed, 0xE9A5])
        u[4 * b:4 * b + 4] = c  # (the helper returns the four uniforms)
    # lo + u (hi - lo) as one fused multiply-add
    row = np.array([np.float32(np.float64(u[k]) * np.float64(np.float32(hi[k] - lo[k])) + np.float64(lo[k])) for k in range(32)], np.float32)
    row[30] = np.float32(np.float64(row[29]) * dt)
    return row


def test_randomizer_draws(model):
    """Check 5: rows lie in [lo, hi], lo == hi is exact, the same (seed, env id, episode) gives the same row (the
    reference Philox stream), and ranges that pin every value to the default row leave the reset -- pose and physics
    step -- bit-identical to the run without ranges."""
    from emu import EmuWarp4
    from emu_envp import EmuEnvpEnv, EmuEnvpWarp4

    seed, env0 = 7, 5
    e0 = EmuEnvpEnv(model.blob())
    default = e0.default_env_params()
    lo, hi = _ranges(default)
    lo[28] = hi[28] = default[28]  # kd pinned: lo == hi
    w = EmuEnvpWarp4(model.blob(), n=4, reset_mode=1, seed=seed, env_id=env0)
    w.env.set_env_params(np.tile(default, (4, 1)))
    w.env.set_env_param_ranges(lo, hi)
    dt = model.meta["params"]["time_step"] / 5
    for ep in range(3):
        w.reset()
        rows = w.env.get_env_params(4)
        for e in range(4):
            assert np.all(rows[e, :30] >= lo[:30]) and np.all(rows[e, :30] <= hi[:30])
            assert rows[e, 28] == default[28] and rows[e, 31] == 0.0
            assert np.array_equal(rows[e], _philox_rows(lo, hi, seed, env0 + e, ep, dt)), (ep, e)
        assert len({rows[e, 26] for e in range(4)}) == 4
    # pose stream untouched: pinned ranges == no ranges, bit for bit
    a = EmuWarp4(model.blob(), n=4, reset_mode=1, seed=seed, env_id=env0)
    b = EmuEnvpWarp4(model.blob(), n=4, reset_mode=1, seed=seed, env_id=env0)
    b.env.set_env_params(np.tile(default, (4, 1)))
    b.env.set_env_param_ranges(default * np.r_[np.ones(30), 0, 0].astype(np.float32), default * np.r_[np.ones(30), 0, 0].astype(np.float32))
    for ep in range(2):
        assert np.array_equal(a.reset(), b.reset())
        assert np.array_equal(a.rec, b.rec)
    b.env.set_env_param_ranges(None, None)


BAD_RANGES = {
    "lo_above_hi": lambda lo, hi: (lo.__setitem__(26, 0.6), hi.__setitem__(26, 0.5)),
    "not_finite": lambda lo, hi: hi.__setitem__(27, np.inf),
    "nan": lambda lo, hi: lo.__setitem__(3, np.nan),
    "zero_mass_scale": lambda lo, hi: lo.__setitem__(25, 0.0),
    "negative_friction": lambda lo, hi: lo.__setitem__(26, -0.1),
    "negative_kd": lambda lo, hi: lo.__setitem__(28, -1.0),
    "element_30_set": lambda lo, hi: hi.__setitem__(30, 1.0),
    "element_31_set": lambda lo, hi: (lo.__setitem__(31, 1.0), hi.__setitem__(31, 1.0)),
}


@pytest.mark.parametrize("bad", list(BAD_RANGES))
def test_bad_ranges_are_rejected(model, bad):
    """Check 6: the host validation shared by the library and the emulator (trex_model.h check_env_param_ranges)."""
    from emu_envp import EmuEnvpEnv

    e = EmuEnvpEnv(model.blob())
    e.set_env_params(e.default_env_params())
    lo, hi = _ranges(e.default_env_params())
    e.set_env_param_ranges(lo, hi)  # the good ranges pass
    BAD_RANGES[bad](lo, hi)
    with pytest.raises(ValueError):
        e.set_env_param_ranges(lo, hi)


def test_with_body_mass_scale(model):
    """The reference model of a row: every merged and full-model mass table of a body scales with it; the COM stays."""
    s = np.ones(26)
    s[25], s[FEMUR] = 3.0, 0.7
    m = with_body_mass_scale(model, s)
    S0, S1 = model.sections, m.sections
    assert np.allclose(S1["mb_mass"][0], 3.0 * S0["mb_mass"][0]) and np.allclose(S1["mb_mass"][1], 0.7 * S0["mb_mass"][1])
    assert np.allclose(S1["mb_mass"][2:], S0["mb_mass"][2:])
    for b, f in ((0, 3.0), (1, 0.7), (2, 1.0)):
        assert np.allclose(S1["mb_mc"].reshape(-1, 3)[b], f * S0["mb_mc"].reshape(-1, 3)[b])
        assert np.allclose(S1["mb_I"].reshape(-1, 6)[b], f * S0["mb_I"].reshape(-1, 6)[b])
        assert np.allclose(S1["mb_damp_rot"].reshape(-1, 6)[b], f * S0["mb_damp_rot"].reshape(-1, 6)[b])
        tb = S0["mb_task_body"] == b
        assert np.allclose(S1["mb_task_m"][tb], f * S0["mb_task_m"][tb])
        assert np.allclose(S1["full_mass"][tb], f * S0["full_mass"][tb])
    assert np.isclose(S1["full_mass"].sum(), S1["mb_mass"].sum())
    with pytest.raises(ValueError):
        with_body_mass_scale(model, np.zeros(26))


def test_calls_without_a_handle_are_invalid():
    """Check 6 (C ABI, no GPU needed): the three calls refuse a NULL handle."""
    from trex_gym_b200 import _native

    L = _native.lib()
    buf = (ctypes.c_float * 32)()
    assert L.trex_set_env_params(None, ctypes.addressof(buf), None, None) == -1
    assert L.trex_get_env_params(None, ctypes.addressof(buf), None) == -1
    assert L.trex_set_env_param_ranges(None, ctypes.addressof(buf), ctypes.addressof(buf)) == -1
    assert ctypes.sizeof(_native.TrexConfig) == 96  # the field came out of `reserved`: the struct size is unchanged


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
    "no_contacts": (1024, {"contacts": False}, "random"),
    "c2": (4096, {}, "random"),
    "standing": (512, {}, "standing"),
    "fallen": (512, {"reset_mode": 1, "seed": 11, "max_episode_steps": 4}, "random"),
    "warps_per_block_4": (1024, {"warps_per_block": 4}, "random"),
    "chunk_envs": (1024, {"chunk_envs": 256}, "random"),
    "pipelines_3": (1024, {"pipelines": 3}, "random"),
    "contact_memory_shared": (1024, {"contact_memory": 1}, "random"),
    "heavy_memory_shared": (512, {"heavy_memory": 1}, "standing"),
    "heavy_memory_tensor": (512, {"heavy_memory": 2}, "standing"),
    "front_solve": (512, {"deferred_solve": False}, "random"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", list(GPU_CONFIGS))
def test_gpu_default_rows_match_env_params_off(cfg):
    """Check 7: env_params = 1 with default rows gives the obs, reward, done and state of env_params = 0 byte for byte."""
    n, kw, acts = GPU_CONFIGS[cfg]
    a, b = _sim(n, **kw), _sim(n, env_params=True, **kw)
    assert _bytes_equal(a.get_state(), b.get_state())
    assert np.array_equal(b.get_env_params()[0].cpu().numpy(), b.default_env_params().numpy())
    steps = 24 if acts == "standing" else 8
    for t in range(steps):
        act = _hold_actions(a) if acts == "standing" else a.random_actions(step=t)
        oa, ra, da = [x.clone() for x in a.step(act)]
        ob, rb, db = b.step(act)
        assert _bytes_equal(oa, ob) and _bytes_equal(ra, rb) and _bytes_equal(da, db), (cfg, t)
        assert _bytes_equal(a.get_state(), b.get_state()), (cfg, t)


@pytest.mark.gpu
def test_gpu_graph_capture_with_env_params():
    a, b = _sim(1024), _sim(1024, env_params=True)
    for t in range(4):
        act = a.random_actions(step=t)
        oa = a.step_graph(act)[0].clone()
        ob = b.step_graph(act)[0]
        assert _bytes_equal(oa, ob), t
    assert _bytes_equal(a.get_state(), b.get_state())


@pytest.mark.gpu
def test_gpu_rows_match_separate_handles(model):
    """Check 8: one batch whose environments carry different rows equals, environment by environment, separate handles
    built from the corresponding modified blobs."""
    import torch

    n = 512
    b = _sim(n, env_params=True)
    rows, models = _rows_and_models(model, b.default_env_params().numpy())
    which = torch.arange(n) % 4
    b.set_env_params(torch.from_numpy(np.stack(rows))[which].contiguous().to(b.device))
    got = b.get_env_params().cpu().numpy()
    assert np.array_equal(got[1, :30], rows[1][:30]) and np.array_equal(got[2], rows[2])
    assert got[1, 30] == np.float32(2.0e5 * (0.01 / 5))  # the impulse bound follows the row's torque
    refs = [_sim(n, model=m) for m in models]
    for s in refs + [b]:
        s.reset()
    for t in range(10):
        act = b.random_actions(step=t)
        ob = b.step(act)[0].clone()
        for k, s in enumerate(refs):
            o = s.step(act)[0]
            sel = (which == k).nonzero().flatten().to(b.device)
            assert _bytes_equal(o[sel], ob[sel]), (t, k)
    for k, s in enumerate(refs):
        sel = (which == k).nonzero().flatten().to(b.device)
        assert _bytes_equal(s.get_state()[sel], b.get_state()[sel]), k


@pytest.mark.gpu
def test_gpu_random_rows_match_the_oracle(model):
    """Check 9: 4,096 environments with random rows; 64 of them checked against the oracle on their modified models."""
    import torch
    from oracle.oracle import Oracle

    n, rng = 4096, np.random.default_rng(9)
    b = _sim(n, env_params=True)
    default = b.default_env_params().numpy()
    rows = np.stack([_random_row(rng, default) for _ in range(n)])
    b.set_env_params(torch.from_numpy(rows).to(b.device))
    b.reset()
    check = list(range(0, n, n // 64))
    oracles = {e: Oracle(_model_of_row(model, rows[e]).blob()) for e in check}
    nc = next(iter(oracles.values())).num_candidates
    free, contact = [], []
    for t in range(24):
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
    # (per env step; over 64 environments x 24 steps the largest contact-free error measured on a B200 was 2.9e-5)
    assert len(free) > 0 and np.percentile(free, 99) < 2e-5 and max(free) < 5e-5, (np.percentile(free, 99), max(free))
    if contact:  # whole env steps (5 substeps) in contact: the bound of smoke(), not the per-substep one
        assert np.percentile(contact, 50) < 1e-3 and np.percentile(contact, 99) < 2e-2, np.percentile(contact, [50, 99])


@pytest.mark.gpu
def test_gpu_randomizer_equals_emulator_and_shards(model):
    """Check 10 and check 5 on the device: the rows the GPU draws equal the emulator's bit for bit; a shard with an
    env_offset draws the rows of the same environments of one large handle; a masked reset redraws only the masked
    environments."""
    import torch
    from emu_envp import EmuEnvpWarp4

    seed, n = 13, 64
    kw = dict(reset_mode=1, seed=seed)
    big = _sim(n, env_params=True, **kw)
    default = big.default_env_params().numpy()
    lo, hi = _ranges(default)
    big.set_env_param_ranges(lo, hi)
    big.reset()
    rows = big.get_env_params().cpu().numpy()
    w = EmuEnvpWarp4(model.blob(), n=4, reset_mode=1, seed=seed, env_id=8)
    w.env.set_env_params(np.tile(default, (4, 1)))
    w.env.set_env_param_ranges(lo, hi)
    w.reset()  # the emulator's episode 0 reset draws what the GPU drew at its episode 1 reset: step the emulator once more
    w.reset()
    assert np.array_equal(w.env.get_env_params(4).view(np.uint32), rows[8:12].view(np.uint32))
    shard = _sim(16, env_params=True, env_offset=32, **kw)
    shard.set_env_param_ranges(lo, hi)
    shard.reset()
    assert np.array_equal(shard.get_env_params().cpu().numpy(), rows[32:48])
    # masked reset: only the masked rows change
    mask = torch.zeros(n, dtype=torch.uint8, device=big.device)
    mask[::3] = 1
    big.reset(mask)
    rows2 = big.get_env_params().cpu().numpy()
    m = mask.cpu().numpy().astype(bool)
    assert np.array_equal(rows2[~m], rows[~m]) and not np.any(np.all(rows2[m] == rows[m], axis=1))


@pytest.mark.gpu
def test_gpu_validation():
    """Check 6 on the device: env_params outside {0, 1}, and the three calls on a handle without the record."""
    from trex_gym_b200 import _native
    from trex_gym_b200.model_compiler import load_builtin

    L = _native.lib()
    blob = load_builtin().blob()
    cfg = _native.TrexConfig()
    cfg.env_params = 2
    h = ctypes.c_void_p()
    assert L.trex_create(blob, len(blob), 8, 0, ctypes.byref(cfg), ctypes.byref(h)) == -1
    s = _sim(8)
    buf = (ctypes.c_float * 32)()
    assert L.trex_set_env_param_ranges(s._h, ctypes.addressof(buf), ctypes.addressof(buf)) == -1
    assert L.trex_get_env_params(s._h, ctypes.addressof(buf), None) == -1
    assert L.trex_set_env_params(s._h, ctypes.addressof(buf), None, None) == -1
    b = _sim(8, env_params=True)
    with pytest.raises(ValueError):
        b.set_env_param_ranges({"friction": 0.5}, {"friction": 0.4})
    with pytest.raises(ValueError):
        b.set_env_params({"mass_scale": {"no_such_joint": 2.0}})


@pytest.mark.gpu
def test_gpu_vec_env_randomize():
    """TrexVecEnv(randomize=...) draws rows at reset within the ranges, named by parameter."""
    from trex_gym_b200.trex_env import TrexVecEnv

    env = TrexVecEnv(256, randomize={"mass_scale": (0.8, 1.25), "friction": (0.15, 0.5), "max_torque": (2.1e5, 3.0e5)})
    env.reset()
    rows = env.sim.get_env_params().cpu().numpy()
    assert rows[:, :26].min() >= 0.8 and rows[:, :26].max() <= 1.25 and rows[:, 26].min() >= 0.15 and rows[:, 29].max() <= 3.0e5
    assert len(np.unique(rows[:, 26])) > 200
    obs, rew, done, _ = env.step(env.sim.random_actions(step=0))
    assert bool(obs.isfinite().all())
