"""Joint-space mass matrix, bias forces and body Jacobians (trex_get_dynamics, TrexBatchSim.mass_matrix / bias_forces /
jacobians).

CPU (the product kernel source through tests/emu/emu_dyn.py, and the oracle): M against the textbook mass matrix of the full
133-link tree and the oracle's M^-1, the reset-pose anchors, b against a double-precision Newton-Euler sum over the 133 links
(gravity and velocity terms separately), the kinetic energy, J against the body-state query and a double forward kinematics,
M rebuilt from J, mass scales, and NULL outputs.  GPU (-m gpu): the library's kernel against the emulator, the query leaving
the step untouched, graph capture, argument checks, and J tied to the external-wrench path of the step."""
import ctypes

import numpy as np
import pytest
from test_body_states import _fk, _hold, _inertia_com, _order, _random_records
from test_oracle_kat import _APPENDIX_B_MKK, _mass_matrix_by_jacobians, _world_kinematics

BASE, NDOF, NB = 25, 31, 26
G = 9.81


def _u(rec):
    """generalized velocity of a record: base angular velocity | base linear velocity | joint rates (link order)"""
    rec = np.asarray(rec, np.float64)
    return np.concatenate([rec[7:10], rec[10:13], rec[38:63]])


def _bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def _skew(r):
    return np.array([[0.0, -r[2], r[1]], [r[2], 0.0, -r[0]], [-r[1], r[0], 0.0]])


# ---------------------------------------------------------------------------------------------------------------------
# references (double)
# ---------------------------------------------------------------------------------------------------------------------
def _link_jacobians(model, quat_xyzw, pos, q_dof):
    """[(mass, world inertia about the COM, Jv, Jw)] of every link of the full model (base link first), in u coordinates,
    and the link -> merged body index (blob order) of each link"""
    S = model.sections
    com, Rlw, joints, parent = _world_kinematics(model, quat_xyzw, pos, q_dof)
    n = len(com) - 1
    mass, Idiag = S["full_mass"], S["full_inertia"].reshape(n + 1, 3)
    by_link = {link: (k, ax, pt) for k, (ax, pt, link) in joints.items()}
    roots = list(np.asarray(model["mb_link"]))
    out, body = [], []
    for b in range(n + 1):
        Jw, Jv = np.zeros((3, 31)), np.zeros((3, 31))
        Jw[:, 0:3] = np.eye(3)
        Jv[:, 3:6] = np.eye(3)
        Jv[:, 0:3] = -_skew(com[b] - com[0])
        a, owner = b, None
        while a > 0:
            if a in by_link:
                k, ax, pt = by_link[a]
                Jw[:, 6 + k] = ax
                Jv[:, 6 + k] = np.cross(ax, com[b] - pt)
                owner = roots.index(a - 1) if owner is None else owner
            a = parent[a - 1] + 1
        out.append((mass[b], Rlw[b] @ np.diag(Idiag[b]) @ Rlw[b].T, Jv, Jw))
        body.append(0 if owner is None else owner)
    return out, np.asarray(body)


def _bias_reference(model, rec, g=G, h=1e-6):
    """b = sum_links [m Jv^T (dJv/dt u) + Jw^T (I_w dJw/dt u + w x I_w w) - m Jv^T g], dJ/dt u by a central difference of the
    link Jacobians along the motion (base orientation advanced by the world angular velocity)"""
    from scipy.spatial.transform import Rotation
    rec = np.asarray(rec, np.float64)
    u = _u(rec)

    def jac(t):
        quat = (Rotation.from_rotvec(u[0:3] * t) * Rotation.from_quat(rec[3:7])).as_quat()
        return _link_jacobians(model, quat, rec[0:3] + t * u[3:6], rec[13:38] + t * u[6:31])[0]

    gv = np.array([0.0, 0.0, -g])
    b = np.zeros(31)
    for (m, Iw, Jv, Jw), (_, _, Jvp, Jwp), (_, _, Jvm, Jwm) in zip(jac(0.0), jac(h), jac(-h)):
        dv, dw = (Jvp - Jvm) @ u / (2 * h), (Jwp - Jwm) @ u / (2 * h)
        w = Jw @ u
        b += m * Jv.T @ dv + Jw.T @ (Iw @ dw + np.cross(w, Iw @ w)) - m * Jv.T @ gv
    return b


def _body_jacobians_ref(model, rec):
    """[26, 6, 31] body Jacobians (query order) from the double forward kinematics of test_body_states"""
    rec = np.asarray(rec, np.float64)
    P, R, _, _ = _fk(model, rec)
    parent = np.asarray(model["mb_parent"])
    c = np.asarray(model["mb_mc"], np.float64).reshape(-1, 3) / np.asarray(model["mb_mass"], np.float64)[:, None]
    J = np.zeros((26, 6, 31))
    for b in range(26):
        k = _order(b)
        J[k, 0:3, 3:6] = np.eye(3)
        J[k, 3:6, 0:3] = np.eye(3)
        J[k, 0:3, 0:3] = -_skew(P[k] - rec[0:3])
        a = b
        while a > 0:
            j = a - 1
            ax, o = R[j][:, 2], P[j] - R[j] @ c[a]
            J[k, 0:3, 6 + j] = np.cross(ax, P[k] - o)
            J[k, 3:6, 6 + j] = ax
            a = int(parent[a])
    return J


def _norm_err(M, H):
    """largest |M - H| / sqrt(H_ii H_jj)"""
    d = np.sqrt(np.abs(np.diag(H)))
    return float((np.abs(M - H) / np.outer(d, d)).max())


# ---------------------------------------------------------------------------------------------------------------------
# fixtures
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu_env(model):
    import emu_dyn
    return emu_dyn.EmuDynEnv(model.blob())


@pytest.fixture(scope="module")
def records(model):
    """64 random records, 8 standing ones with floor contact, 8 of fallen episodes (reset_mode 1)"""
    import emu_dyn
    rng = np.random.default_rng(11)
    out = [_random_records(model, rng, 64)]
    env = emu_dyn.EmuDynEnv(model.blob())
    env.reset()
    hold = _hold(model)
    stand = []
    for t in range(60):
        env.step(hold)
        if t >= 52:
            stand.append(env.rec.copy())
    out.append(np.stack(stand))
    lo, hi = model["mb_lower"][1:][model["obs_dof"]], model["mb_upper"][1:][model["obs_dof"]]
    fallen = []
    for s in range(8):
        env = emu_dyn.EmuDynEnv(model.blob(), reset_mode=1, seed=11 + s)
        env.reset()
        for t in range(6):
            env.step(rng.uniform(lo, hi).astype(np.float32))
        fallen.append(env.rec.copy())
    out.append(np.stack(fallen))
    return np.concatenate(out)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the emulator
# ---------------------------------------------------------------------------------------------------------------------
# M against the 133-link mass matrix of test_oracle_kat over the 80 records: largest entry error normalised by
# sqrt(M_ii M_jj) seen 1.9e-6 (tolerance 10x); M Minv_oracle - I over every fourth record: largest entry 2.0e-4 (5x).
TOL_M, TOL_MINV = 2e-5, 1e-3


def test_mass_matrix_against_link_jacobians_and_oracle_inverse(model, emu_env, records):
    from oracle.oracle import Oracle
    M, _, _ = emu_env.dynamics(records, outputs="M")
    worst = 0.0
    for i, rec in enumerate(records):
        r = rec.astype(np.float64)
        H = _mass_matrix_by_jacobians(model, r[3:7], r[0:3], r[13:38])
        worst = max(worst, _norm_err(M[i].astype(np.float64), H))
    assert worst < TOL_M, worst
    o = Oracle(model.blob(), contacts=False)
    o.reset()
    nc = o.num_candidates
    worst_inv = 0.0
    for i in range(0, len(records), 10):
        o.set_state(np.concatenate([records[i, :88], np.zeros(nc)]).astype(np.float64))
        Minv = np.stack([o.minv_column(d) for d in range(31)], 1)
        worst_inv = max(worst_inv, np.abs(M[i].astype(np.float64) @ Minv - np.eye(31)).max())
    assert worst_inv < TOL_MINV, worst_inv


def test_reset_pose_anchors_and_exact_symmetry(model, emu_env, records):
    emu_env.reset()
    M, _, _ = emu_env.dynamics(outputs="M")
    names = model.meta["body_joint_names"][1:]
    for k, name in enumerate(names):
        want = _APPENDIX_B_MKK[name.replace("joint_", "", 1)]
        assert abs(M[6 + k, 6 + k] - want) < 2e-6 * max(1.0, want) + 1e-6, (name, M[6 + k, 6 + k], want)
    mass = float(np.sum(model["full_mass"]))
    assert np.allclose(np.diag(M)[3:6], mass, rtol=5e-7) and not np.any(M[3:6, 3:6] - np.diag(np.diag(M)[3:6]))
    Ms, _, _ = emu_env.dynamics(records, outputs="M")
    assert np.array_equal(_bits(Ms), _bits(Ms.transpose(0, 2, 1)))


# b against the 133-link Newton-Euler sum, gravity only (u = 0) and velocity only (gravity 0), 12 records each: largest
# error over max |b_ref| seen 2.2e-7 (gravity) and 1.0e-6 (velocity); tolerance 10x the larger.
TOL_B = 1e-5


@pytest.mark.parametrize("part", ["gravity", "velocity"])
def test_bias_against_newton_euler_on_the_link_tree(model, records, part):
    import emu_dyn
    from trex_gym_b200.model_compiler import with_params
    sel = records[::7][:12].copy()
    if part == "gravity":
        sel[:, 7:13] = 0.0
        sel[:, 38:63] = 0.0
        mdl, g = model, G
    else:
        mdl, g = with_params(model, gravity=0.0), 0.0
    env = emu_dyn.EmuDynEnv(mdl.blob())
    _, b, _ = env.dynamics(sel, outputs="b")
    worst = 0.0
    for i, rec in enumerate(sel):
        ref = _bias_reference(mdl, rec, g)
        worst = max(worst, np.abs(b[i] - ref).max() / np.abs(ref).max())
    assert worst < TOL_B, worst


# kinetic energy 1/2 u^T M u against the oracle: largest relative error seen 2.2e-7 (tolerance 5e-6)
def test_kinetic_energy_and_base_jacobian(model, emu_env, records):
    from oracle.oracle import Oracle
    o = Oracle(model.blob(), contacts=False)
    o.reset()
    nc = o.num_candidates
    M, _, J = emu_env.dynamics(records, outputs="Mj")
    worst = 0.0
    for i in range(0, len(records), 4):
        o.set_state(np.concatenate([records[i, :88], np.zeros(nc)]).astype(np.float64))
        u = _u(records[i])
        ke = 0.5 * u @ M[i].astype(np.float64) @ u
        worst = max(worst, abs(ke - o.momentum()["ke"]) / o.momentum()["ke"])
    assert worst < 5e-6, worst
    # the base body: its angular velocity is u[0:3] exactly, its COM (the merged base's, not the base link's) moves with
    # u[3:6] + u[0:3] x (c - x_base)
    eye = np.eye(3, dtype=np.float32)
    assert np.array_equal(J[:, BASE, 3:6, 0:3], np.broadcast_to(eye, (len(records), 3, 3)))
    assert np.array_equal(J[:, BASE, 0:3, 3:6], np.broadcast_to(eye, (len(records), 3, 3)))
    assert not J[:, BASE, 3:6, 3:].any() and not J[:, BASE, 0:3, 6:].any()


# J against the double forward kinematics (largest entry error seen 6.1e-7 relative to 1 + |base position|), J u against
# the body-state query's [v | w] on the same records (4.9e-7 relative to 1 + the largest speed), and the body's COM
# Jacobian against the mass-weighted link Jacobians of the 133-link tree (5.2e-7); tolerance about 20x
TOL_J, TOL_JU = 1e-5, 1e-5


def test_jacobians_against_body_states_and_double_fk(model, emu_env, records):
    import emu_bodies
    _, _, J = emu_env.dynamics(records, outputs="j")
    states, _ = emu_bodies.EmuBodiesEnv(model.blob()).body_states(records)
    worst = np.zeros(3)
    for i, rec in enumerate(records):
        Jd = J[i].astype(np.float64)
        worst[0] = max(worst[0], np.abs(Jd - _body_jacobians_ref(model, rec)).max() / (1.0 + np.abs(rec[0:3]).max()))
        vw = Jd @ _u(rec)
        worst[1] = max(worst[1], np.abs(vw - states[i, :, 7:13]).max() / (1.0 + np.abs(states[i, :, 7:13]).max()))
        if i % 8 == 0:
            r = rec.astype(np.float64)
            links, body = _link_jacobians(model, r[3:7], r[0:3], r[13:38])
            for b in range(NB):
                m = sum(links[l][0] for l in np.nonzero(body == b)[0])
                Jv = sum(links[l][0] * links[l][2] for l in np.nonzero(body == b)[0]) / m
                worst[2] = max(worst[2], np.abs(Jd[_order(b), 0:3] - Jv).max() / (1.0 + np.abs(r[0:3]).max()))
    assert worst[0] < TOL_J and worst[1] < TOL_JU and worst[2] < TOL_J, worst


# M = sum_k J_k^T diag(m_k 1, I_k,world) J_k from the kernel's own J and the blob's merged-body inertias: 3.8e-7 seen
def test_mass_matrix_from_the_kernels_jacobians(model, emu_env, records):
    M, _, J = emu_env.dynamics(records, outputs="Mj")
    m = np.concatenate([np.asarray(model["mb_mass"], np.float64)[1:], np.asarray(model["mb_mass"], np.float64)[:1]])
    Ic = _inertia_com(model)
    worst = 0.0
    for i, rec in enumerate(records):
        _, R, _, _ = _fk(model, rec)
        H = np.zeros((31, 31))
        for k in range(NB):
            Jk = J[i, k].astype(np.float64)
            D = np.zeros((6, 6))
            D[0:3, 0:3] = m[k] * np.eye(3)
            D[3:6, 3:6] = R[k] @ Ic[k] @ R[k].T
            H += Jk.T @ D @ Jk
        worst = max(worst, _norm_err(M[i].astype(np.float64), H))
    assert worst < TOL_M, worst


def test_mass_scales(model, emu_env, records):
    from trex_gym_b200.model_compiler import with_body_mass_scale
    full = emu_env.dynamics(records)
    ones = emu_env.dynamics(records, envp=np.ones(32, np.float32))
    for x, y in zip(full, ones):
        assert np.array_equal(_bits(x), _bits(y))
    two = emu_env.dynamics(records, envp=np.full(32, 2.0, np.float32))
    assert np.array_equal(_bits(two[0]), _bits(2.0 * full[0])) and np.array_equal(_bits(two[1]), _bits(2.0 * full[1]))
    assert np.array_equal(_bits(two[2]), _bits(full[2]))
    # a random row against the references built from the scaled model (seen: 1.5e-6 for M, 3.7e-7 for b; same tolerances)
    rng = np.random.default_rng(4)
    row = np.ones(32, np.float32)
    row[:26] = rng.uniform(0.5, 1.5, 26)
    scaled = with_body_mass_scale(model, row[:26])
    sel = records[::10]
    M, b, _ = emu_env.dynamics(sel, envp=row, outputs="Mb")
    for i, rec in enumerate(sel):
        r = rec.astype(np.float64)
        assert _norm_err(M[i].astype(np.float64), _mass_matrix_by_jacobians(scaled, r[3:7], r[0:3], r[13:38])) < TOL_M, i
        ref = _bias_reference(scaled, rec)
        assert np.abs(b[i] - ref).max() / np.abs(ref).max() < TOL_B, i


def test_each_output_alone_equals_the_full_query(emu_env, records):
    full = emu_env.dynamics(records)
    for k, letter in enumerate("Mbj"):
        alone = emu_env.dynamics(records, outputs=letter)
        assert all(alone[j] is None for j in range(3) if j != k)
        assert np.array_equal(_bits(alone[k]), _bits(full[k])), letter


def test_null_arguments_are_rejected():
    from trex_gym_b200 import _native
    L = _native.lib()
    buf = (ctypes.c_float * 64)()
    assert L.trex_get_dynamics(None, None, None, None, None) == -1
    assert L.trex_get_dynamics(None, ctypes.addressof(buf), None, None, None) == -1


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
# Device against emulator on the same records: sinf / cosf and the contracted multiply-adds differ by ulps between the two.
# Largest errors seen on one B200 over the four workloads and the mass-scale test: M 4.0e-6 (entry error over
# sqrt(M_ii M_jj)), b 1.8e-6 (over max |b|), J 2.9e-7 (over 1 + |base position|); tolerance 5x to 10x.
GPU_TOL = {"M": 2e-5, "b": 2e-5, "J": 3e-6}


def _query(sim):
    import torch
    n = sim.num_envs
    out = (torch.empty(n, NDOF, NDOF, device=sim.device), torch.empty(n, NDOF, device=sim.device),
           torch.empty(n, NB, 6, NDOF, device=sim.device))
    sim._dynamics_query(*out)
    return out


def _compare_gpu_emulator(sim, emu_env, idx, envp=None):
    import torch
    M, b, J = (x.cpu().numpy()[idx] for x in _query(sim))
    rec = sim.get_state().cpu().numpy()[idx]
    torch.cuda.synchronize()
    eM, eb, eJ = emu_env.dynamics(rec, envp=envp)
    assert np.array_equal(_bits(M), _bits(M.transpose(0, 2, 1)))
    err = {"M": max(_norm_err(M[i].astype(np.float64), eM[i].astype(np.float64)) for i in range(len(idx))),
           "b": max(np.abs(b[i] - eb[i]).max() / np.abs(eb[i]).max() for i in range(len(idx))),
           "J": float(np.abs(J - eJ).max() / (1.0 + np.abs(rec[:, 0:3]).max()))}
    assert all(err[k] < GPU_TOL[k] for k in err), err


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["random", "standing", "fallen", "primitives"])
def test_gpu_matches_emulator(model, workload):
    import emu_dyn
    import torch
    from trex_gym_b200.model_compiler import load_builtin
    from trex_gym_b200.sim import TrexBatchSim
    n, steps, kw, mdl = 4096, 60, {}, model
    if workload == "random":
        n, steps = 65536, 100  # the bench pre-roll
    elif workload == "fallen":
        kw = dict(reset_mode=1, max_episode_steps=64, seed=11)
    elif workload == "primitives":
        mdl = load_builtin("primitives")
    sim = TrexBatchSim(n, device=0, model=mdl, **kw)
    sim.reset()
    hold = torch.tensor(_hold(mdl), device=sim.device).repeat(n, 1).contiguous()
    for t in range(steps):
        sim.step(hold if workload == "standing" else sim.random_actions(step=t % 16))
    idx = np.random.default_rng(1).choice(n, 256, replace=False)
    _compare_gpu_emulator(sim, emu_dyn.EmuDynEnv(mdl.blob(), **kw), idx)


@pytest.mark.gpu
def test_gpu_mass_scales_match_emulator(model):
    import emu_dyn
    from trex_gym_b200.sim import TrexBatchSim
    n = 1024
    sim = TrexBatchSim(n, device=0, env_params=True)
    sim.set_env_param_ranges({"mass_scale": 0.5}, {"mass_scale": 1.5})
    sim.reset()
    for t in range(20):
        sim.step(sim.random_actions(step=t))
    idx = np.random.default_rng(2).choice(n, 64, replace=False)
    rows = sim.get_env_params().cpu().numpy()[idx]
    _compare_gpu_emulator(sim, emu_dyn.EmuDynEnv(model.blob()), idx, envp=rows)


@pytest.mark.gpu
@pytest.mark.parametrize("env_params,external_forces", [(False, False), (True, True)])
def test_gpu_query_is_read_only(model, env_params, external_forces):
    import torch
    from trex_gym_b200.sim import TrexBatchSim

    def run(query):
        sim = TrexBatchSim(512, device=0, env_params=env_params, external_forces=external_forces)
        sim.reset()
        if external_forces:
            f = torch.zeros(512, 26, 3, device=sim.device)
            f[:, BASE, 0] = 2000.0
            sim.set_external_forces(f)
            sim.set_push_schedule("base", interval=16, duration=4, probability=0.5, force=(1000.0, 5000.0))
        if env_params:
            sim.set_env_param_ranges({"mass_scale": 0.9, "friction": 0.2}, {"mass_scale": 1.1, "friction": 0.3})
            sim.reset()
        out = []
        for t in range(64):
            o, r, d = sim.step(sim.random_actions(step=t))
            out.append((o.clone(), r.clone(), d.clone(), sim.get_state()))
            if query:
                _query(sim)
        torch.cuda.synchronize()
        return [[x.cpu().numpy() for x in o] for o in out]

    a, b = run(False), run(True)
    for t, (x, y) in enumerate(zip(a, b)):
        for u, v in zip(x, y):
            assert np.array_equal(u.view(np.uint8), v.view(np.uint8)), t


@pytest.mark.gpu
def test_gpu_graph_of_step_and_query(model):
    import torch
    from trex_gym_b200.sim import TrexBatchSim
    n = 1024
    sim = TrexBatchSim(n, device=0)
    sim.reset()
    act = torch.tensor(_hold(model), device=sim.device).repeat(n, 1).contiguous()
    M, b, J = (torch.empty(n, NDOF, NDOF, device=sim.device), torch.empty(n, NDOF, device=sim.device),
               torch.empty(n, NB, 6, NDOF, device=sim.device))
    for t in range(20):
        sim.step(act)
    start = sim.get_state().clone()
    torch.cuda.synchronize()
    side = torch.cuda.Stream(device=sim.device)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        sim.step(act)
        sim.mass_matrix(out=M)
        sim.bias_forces(out=b)
        sim.jacobians(out=J)
        side.synchronize()
        sim.set_state(start)
        side.synchronize()
        with torch.cuda.graph(g, stream=side):
            sim.step(act)
            sim.mass_matrix(out=M)
            sim.bias_forces(out=b)
            sim.jacobians(out=J)
    torch.cuda.synchronize()
    sim.set_state(start)
    ref = []
    for t in range(4):
        sim.step(act)
        ref.append((sim.mass_matrix().clone(), sim.bias_forces().clone(), sim.jacobians().clone(), sim.get_state()))
    torch.cuda.synchronize()
    sim.set_state(start)
    for t in range(4):
        g.replay()
        torch.cuda.synchronize()
        for u, v in zip(ref[t], (M, b, J, sim.get_state())):
            assert torch.equal(u.view(torch.int32), v.view(torch.int32)), t


@pytest.mark.gpu
def test_gpu_arguments(model):
    import torch
    from trex_gym_b200.sim import TrexBatchSim
    sim = TrexBatchSim(8, device=0)
    assert sim._L.trex_get_dynamics(sim._h, None, None, None, None) == -1
    assert sim.dof_names()[6:] == list(model.meta["body_joint_names"][1:]) and len(sim.dof_names()) == NDOF
    dev = sim.device
    for bad in (torch.empty(8, 31, 30, device=dev), torch.empty(8, 31, 31, device=dev, dtype=torch.float64),
                torch.empty(8, 31, 31), torch.empty(8, 31, 31, device=dev).transpose(1, 2)):
        with pytest.raises(ValueError):
            sim.mass_matrix(out=bad)
    for bad in (torch.empty(8, 30, device=dev), torch.empty(8, 31, device=dev, dtype=torch.float16), torch.empty(8, 31)):
        with pytest.raises(ValueError):
            sim.bias_forces(out=bad)
    for bad in (torch.empty(8, 26, 31, 6, device=dev), torch.empty(8, 26, 6, 31, device=dev, dtype=torch.int32),
                torch.empty(8, 26, 6, 31)):
        with pytest.raises(ValueError):
            sim.jacobians(out=bad)
    assert sim.mass_matrix().shape == (8, 31, 31) and sim.bias_forces().shape == (8, 31)
    assert sim.jacobians().shape == (8, 26, 6, 31)


# One contact-free step (the batch lifted 20 m, motors inert) from the same record, with and without a wrench [F; T] on a
# leg body: the change of M u (M of the starting record) is dt_step J_k^T [F; T] to first order in the step.  Largest error
# seen on one B200, relative to max |dt J_k^T [F; T]|: 3.9e-4 (second-order terms: damping, the change of M over the step);
# tolerance 4e-3.
@pytest.mark.gpu
def test_gpu_jacobian_transpose_is_the_generalized_impulse_of_a_wrench(model):
    import torch
    from trex_gym_b200.sim import TrexBatchSim
    n = 64
    body = "joint_tibia_left"
    k = model.meta["body_joint_names"].index(body) - 1
    F, T = torch.tensor([3000.0, -2000.0, 4000.0]), torch.tensor([500.0, 800.0, -300.0])
    outs = []
    for push in (False, True):
        sim = TrexBatchSim(n, device=0, env_params=True, external_forces=True, contacts=False)
        sim.reset()
        sim.set_env_params({"kp": 0.0, "kd": 0.0, "max_torque": 0.0})
        s = sim.get_state()
        s[:, 2] += 20.0
        sim.set_state(s)
        if push:
            f = torch.zeros(n, 26, 3, device=sim.device)
            t = torch.zeros(n, 26, 3, device=sim.device)
            f[:, k], t[:, k] = F.to(sim.device), T.to(sim.device)
            sim.set_external_forces(f, t)
        M0, J0 = sim.mass_matrix().double(), sim.jacobians().double()
        sim.step(torch.tensor(_hold(model), device=sim.device).repeat(n, 1).contiguous())
        rec = sim.get_state().double()
        u = torch.cat([rec[:, 7:13], rec[:, 38:63]], 1)
        outs.append((M0, J0, u))
    (M0, J0, ua), (_, _, ub) = outs
    dt = 0.01
    wrench = torch.cat([F, T]).double().to(M0.device)
    want = dt * J0[:, k].transpose(1, 2) @ wrench
    got = (M0 @ (ub - ua)[..., None])[..., 0]
    rel = ((got - want).abs().max(1).values / want.abs().max(1).values).max().item()
    assert rel < 4e-3, rel
