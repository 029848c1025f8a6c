"""GPU tests of the drop-in boundary (SURVEY.md section 8b): the gym surface mirrors the reference's call pattern,
configuration goes through named trex_config fields, the host-buffer entry points and CUDA-graph capture."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _sim(model, n, **kw):
    from trex_gym_b200.sim import TrexBatchSim

    return TrexBatchSim(n, device=0, model=model, **kw)


def test_set_actions_takes_effect_like_the_reference_loop(model):
    """trex_env.py:147-150: `clipped = np.clip(action); for _ in range(action_repeat): model.set_actions(clipped);
    stepSimulation()`.  TrexRobot.set_actions writes the persistent motor targets and TrexBulletEnv.step consumes them:
    driving the robot through set_actions + sim.step() gives bit-identical results to env.step(action)."""
    import torch

    from trex_gym_b200 import TrexBulletEnv

    env_a = TrexBulletEnv(urdf_path=None, model=model)
    env_b = TrexBulletEnv(urdf_path=None, model=model)
    rng = np.random.default_rng(0)
    for t in range(4):
        a = env_a.action_space.sample() * 1.2  # partly outside the limits: the clip matters
        obs_a, rew_a, done_a, info_a = env_a.step(a)
        # the reference's inner loop spelled out on the robot adapter
        clipped = np.clip(a, env_b.action_space.low, env_b.action_space.high)
        env_b.model.set_actions(clipped)
        env_b._sim.step()
        assert env_b.model.get_observations() == obs_a
        assert float(env_b._sim.reward[0].item()) == rew_a
        assert info_a == {} and done_a is False
    # targets persist (pybullet motor state): stepping again without a new set_actions keeps servoing to the same targets
    tgt = env_b._sim.targets.clone()
    env_b._sim.step()
    assert torch.equal(tgt, env_b._sim.targets)
    # and they do steer the robot: a different target gives a different trajectory from the same state
    env_a._sim.set_state(env_b._sim.get_state())
    env_a.model.set_actions(np.zeros(25))
    env_b.model.apply_action(np.full(25, 0.3))  # north-star alias
    env_a._sim.step()
    env_b._sim.step()
    assert np.abs(np.asarray(env_a.model.get_observation()) - np.asarray(env_b.model.get_observations())).max() > 1e-3
    with pytest.raises(ValueError):
        env_a.model.set_actions(np.zeros(7))


def test_vecenv_infos_and_sharded_exploration_noise(model):
    """baselines VecEnv: one info dict per environment.  Exploration noise and random actions are keyed by the GLOBAL
    environment id: two shards of 32 reproduce one batch of 64 bit for bit (and differ from each other)."""
    import torch

    from trex_gym_b200 import TrexVecEnv
    from trex_gym_b200.rollout import MlpPolicy, RolloutBuffer

    venv = TrexVecEnv(8, model=model)
    venv.reset()
    _, _, _, infos = venv.step(np.zeros((8, 25), np.float32))
    assert infos == [{}] * 8 and len({id(i) for i in infos}) == 8

    T = 3
    whole = _sim(model, 64, seed=3)
    shards = [_sim(model, 32, seed=3, env_offset=32 * r) for r in range(2)]
    assert shards[1].env_offset == 32
    dev = whole.device
    pol = MlpPolicy(dev, seed=1)
    pol.view("logstd").fill_(-0.5)
    for policy in (None, pol):
        bw = RolloutBuffer(whole, T).collect(policy=policy, seed=9)
        bs = [RolloutBuffer(s, T).collect(policy=policy, seed=9) for s in shards]
        assert torch.equal(bw.actions[:, :32], bs[0].actions) and torch.equal(bw.actions[:, 32:], bs[1].actions)
        assert not torch.equal(bs[0].actions, bs[1].actions)
        assert torch.equal(bw.obs[:, 32:], bs[1].obs) and torch.equal(bw.rewards[:, :32], bs[0].rewards)
        whole.reset()
        for s in shards:
            s.reset()


def test_named_config_fields_are_validated(model):
    from trex_gym_b200 import _native

    L = _native.lib()
    blob = model.blob()

    def create(**kw):
        cfg = _native.TrexConfig()
        cfg.num_substeps, cfg.enable_contacts = 5, 1
        cfg.distance_weight, cfg.energy_weight, cfg.drift_weight = 1.0, 0.005, 0.002
        for k, v in kw.items():
            if k == "reserved0":
                cfg.reserved[0] = v
            else:
                setattr(cfg, k, v)
        h = ctypes.c_void_p()
        rc = L.trex_create(blob, len(blob), 4, 0, ctypes.byref(cfg), ctypes.byref(h))
        if rc == 0:
            L.trex_destroy(h)
        return rc, L.trex_last_error().decode()

    assert create()[0] == 0
    assert create(warps_per_block=4, solver_placement=_native.SOLVE_NO_HEAVY, env_offset=1 << 40)[0] == 0
    for bad in (dict(warps_per_block=3), dict(solver_placement=7), dict(heavy_share_div=-1), dict(pipelines=9), dict(heavy_memory=3), dict(chunk_envs=6), dict(contact_memory=2),
                dict(reserved0=1)):
        rc, msg = create(**bad)
        assert rc == -1 and list(bad)[0].rstrip("0") in msg, (bad, rc, msg)


def test_step_host_async_double_buffered(model):
    """trex_step_host_async: depth-1 pipeline over two sets of pinned host arrays (copies of step k under step k+1);
    results equal the synchronous call's."""
    import torch

    n = 512
    s_sync, s_async = _sim(model, n), _sim(model, n)
    acts = [s_sync.random_actions(step=t).cpu().pin_memory() for t in range(6)]
    ref = [tuple(np.copy(x) for x in s_sync.step_host(a)) for a in acts]
    bufs = [(torch.empty(n, 75).pin_memory(), torch.empty(n).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory())
            for _ in range(2)]
    got = []
    for t, a in enumerate(acts):
        s_async.step_host_async(a, *bufs[t & 1])
        if t >= 1:  # contract: on return the previous call's outputs are complete
            got.append(tuple(x.numpy().copy() for x in bufs[(t - 1) & 1]))
    s_async.host_wait()
    got.append(tuple(x.numpy().copy() for x in bufs[(len(acts) - 1) & 1]))
    for (ro, rr, rd), (go, gr, gd) in zip(ref, got):
        assert np.array_equal(ro, go) and np.array_equal(rr, gr) and np.array_equal(rd, gd)
    assert torch.equal(s_sync.get_state(), s_async.get_state())


def test_cuda_graph_capture_of_a_step(model):
    """include/trex_b200.h: all launches go to the caller's stream (the heavy-contact kernel forks to a side stream and
    joins back with events), so one trex_step can be captured into a CUDA graph and replayed."""
    import torch

    n = 2048
    eager, graphed = _sim(model, n), _sim(model, n)
    # a batch with every solver class in play: standing (many contacts) and random-action environments
    names = list(model.meta["obs_joint_names"])
    hold = torch.zeros(25, device=eager.device)
    for k, v in model.meta["starting_configuration"].items():
        hold[names.index(k)] = v
    for t in range(30):
        a = eager.random_actions(step=t, seed=5)
        a[: n // 2] = hold
        eager.step(a)
    graphed.set_state(eager.get_state())
    a = eager.random_actions(step=99, seed=5)
    a[: n // 2] = hold
    obs_g = torch.empty(n, 75, device=eager.device)
    rew_g = torch.empty(n, device=eager.device)
    done_g = torch.empty(n, dtype=torch.uint8, device=eager.device)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        pre = graphed.get_state().clone()
        graphed.step_into(a, obs_g, rew_g, done_g)  # warm-up on the side stream (kernel attributes configured)
        graphed.set_state(pre)
        side.synchronize()
        with torch.cuda.graph(g, stream=side):
            graphed.step_into(a, obs_g, rew_g, done_g)
    torch.cuda.synchronize()
    graphed.set_state(pre)
    torch.cuda.synchronize()
    for k in range(3):
        g.replay()
        obs_e, rew_e, _ = eager.step(a)
        torch.cuda.synchronize()
        assert torch.equal(obs_e, obs_g) and torch.equal(rew_e, rew_g), k
    assert torch.equal(eager.get_state()[:, :152], graphed.get_state()[:, :152])
    assert eager.stats()["mean_contacts"] > 4.0  # half the batch stands on both feet


def test_step_graph_replays_the_step(model):
    """TrexBatchSim.capture_graph / step_graph: the whole env step (kernels, fork / join events, counter resets of the persistent
    solvers) captured once into a CUDA graph with simulator-owned buffers and replayed per step -- bit-identical to ``step``."""
    import torch

    n = 4096
    a, b = _sim(model, n, seed=1), _sim(model, n, seed=1)
    for t in range(30):
        act = a.random_actions(step=t)
        o1, r1, d1 = a.step(act)
        o2, r2, d2 = b.step_graph(act)
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(d1, d2), t
    assert torch.equal(a.get_state()[:, :152], b.get_state()[:, :152]) and a.stats()["mean_contacts"] > 0.05


def test_replay_frames_recorded_on_hardware(model, tmp_path):
    """SURVEY.md section 8f row 4 on the GPU: record 20 real frames of two environments while the batch is stepped, then
    recompute the head position on the HOST from each exported frame (base pose + joint angles only) and compare it with
    the head position the kernels reported for that step (aux[:, 0:3], the point the reward is computed from)."""
    import json

    from trex_gym_b200.replay import ReplayRecorder, link_world_position

    sim = _sim(model, 64)
    sim.reset()
    rec = ReplayRecorder(sim, env_indices=(3, 40))
    heads = []
    for t in range(20):
        sim.step(sim.random_actions(step=t, seed=8))
        rec.capture()
        heads.append(sim.aux()[[3, 40], 0:3].cpu().numpy())
    for which in (0, 1):
        path = rec.save(str(tmp_path / ("replay_%d.json" % which)), which=which)
        d = json.load(open(path))
        assert len(d["joint_positions"]) == 20 and d["dt"] == 0.01 and len(d["joint_names"]) == 25
        for t in range(20):
            p = link_world_position(model, d["base_position"][t], d["base_orientation_xyzw"][t], d["joint_positions"][t])
            assert np.abs(p - heads[t][which]).max() < 2e-5, (which, t, p, heads[t][which])
    # the two environments were driven differently: the frames are really per environment
    a, b = rec.as_dict(0), rec.as_dict(1)
    assert np.abs(np.asarray(a["joint_positions"][-1]) - np.asarray(b["joint_positions"][-1])).max() > 1e-3


def test_literal_reference_configuration(model):
    """ADVICE round 1: the default configuration (URDF inertia, derived floor contact) is not what the literal reference
    simulates; ``literal_reference=True`` is -- default-flag inertia and no contact geometry -- and matches the oracle on the
    same blob.  Both configurations ship and are tested."""
    from oracle.oracle import Oracle
    from trex_gym_b200 import TrexBulletEnv
    from trex_gym_b200.model_compiler import load_builtin

    env = TrexBulletEnv(literal_reference=True)
    assert env._sim.model.meta["inertia_source"] == "bullet_default"
    o = Oracle(load_builtin("literal").blob(), contacts=False)
    assert np.abs(np.asarray(env.reset()) - o.reset()).max() < 1e-6
    rng = np.random.default_rng(1)
    for t in range(60):
        a = rng.uniform(env.action_space.low, env.action_space.high).astype(np.float32)
        obs, rew, done, info = env.step(a)
        oobs, orew = o.step(a.astype(np.float64))
    # free running for 60 steps, contact free: still close (1e-4 of the block magnitudes), and falling through the floor plane
    assert np.abs(np.asarray(obs)[:25] - oobs[:25]).max() < 1e-3
    assert env.model.get_base_position()[2] < 1.5 and not done
    env.close()
    std = TrexBulletEnv()
    assert std._sim.model.meta["inertia_source"] == "urdf" and len(std._sim.model["mb_cand_body"]) == 48
    std.close()


def test_pipelined_groups_do_not_change_results(model):
    """trex_config.pipelines: the batch stepped as 1, 2, 3 or 4 independent groups of environments on separate streams
    (group boundaries on multiples of four; the last group may be short) gives bit-identical records, observations, rewards
    and done flags -- also with fallen starts, whose sampler is keyed by the global environment id, and through auto-resets."""
    import torch

    n = 9998  # not a multiple of anything convenient
    sims = [_sim(model, n, pipelines=p, reset_mode=1, max_episode_steps=7, seed=4, env_offset=123) for p in (1, 2, 3, 4)]
    # ... and walked chunk by chunk (trex_config.chunk_envs: all substeps of a chunk before the next one, every chunk of a group in
    # the same work-record slots, so that the records stay in L2), with the last chunk short
    sims += [_sim(model, n, pipelines=p, chunk_envs=c, reset_mode=1, max_episode_steps=7, seed=4, env_offset=123)
             for p, c in ((1, 4096), (2, 1024), (3, 2500))]
    ref = sims[0]
    for t in range(16):
        a = ref.random_actions(step=t, seed=2, env_offset=123)
        outs = [tuple(x.clone() for x in s.step(a)) for s in sims]
        for o in outs[1:]:
            assert all(torch.equal(x, y) for x, y in zip(outs[0], o)), t
    st = [s.get_state() for s in sims]
    assert all(torch.equal(st[0], x) for x in st[1:])
    assert all(s.stats() == ref.stats() for s in sims[1:])
    assert ref.stats()["episodes"] == n * 3 and ref.stats()["mean_contacts"] > 0.3
    # masked reset through the groups
    mask = torch.zeros(n, dtype=torch.uint8, device=ref.device)
    mask[::3] = 1
    obs = [s.reset(mask).clone() for s in sims]
    assert all(torch.equal(obs[0], x) for x in obs[1:])


@pytest.mark.parametrize("workload,envs,rows", [("c2", 0, 4096), ("rollout", 256, 256)])
def test_bench_dump_outputs_end_to_end(tmp_path, workload, envs, rows):
    """bench.py --dump-outputs: the timed loop runs exactly --steps steps, the last one's outputs land in DIR as float32
    with one row per environment, and two runs with the same arguments write the same arrays."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for d in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", workload, "--envs-per-gpu", str(envs),
                              "--steps", "3", "--warmup", "3", "--preroll", "5", "--no-cpu-baseline", "--spread-steps", "0",
                              "--dump-outputs", str(tmp_path / d)], capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
    names = sorted(os.listdir(tmp_path / "a"))
    assert {"obs.npy", "reward.npy", "done.npy"} <= set(names) and names == sorted(os.listdir(tmp_path / "b"))
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and a.shape[0] == rows and np.isfinite(a).all(), f
        assert np.array_equal(a, b), f
    assert np.load(tmp_path / "a" / "obs.npy").shape == (rows, 75)
