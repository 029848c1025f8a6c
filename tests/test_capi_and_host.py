"""No-GPU checks of the drop-in boundary: the shared library loads, exports every symbol declared in
include/trex_b200.h, refuses to run without a GPU, and the host-side logic (spaces shim, sharding,
bench contract) behaves."""
import ctypes
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    src = open(os.path.join(ROOT, "include", "trex_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(trex_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from trex_gym_b200 import _native

    _native.build()
    L = ctypes.CDLL(_native.LIB_PATH)
    names = _declared_functions()
    assert len(names) >= 16
    for n in names:
        assert hasattr(L, n), n
    assert set(names) == set(_native.EXPORTED_SYMBOLS)
    L.trex_version.restype = ctypes.c_char_p
    assert b"sm_100a" in L.trex_version()


_NO_CPU_FALLBACK = """
import ctypes
import pytest
from trex_gym_b200 import _native
from trex_gym_b200.model_compiler import load_builtin
from trex_gym_b200.sim import TrexBatchSim

with pytest.raises(RuntimeError):
    TrexBatchSim(4)
# the C entry point itself also fails loudly instead of computing on the host
L = _native.lib()
blob = load_builtin().blob()
h = ctypes.c_void_p()
rc = L.trex_create(blob, len(blob), 4, 0, None, ctypes.byref(h))
assert rc != 0 and not h.value
assert b"CUDA" in L.trex_last_error() or b"cuda" in L.trex_last_error()
"""


def test_no_cpu_fallback():
    """Without a visible GPU, both the Python class and the C entry point refuse to run.  The check runs in a child
    process with every GPU hidden, so it also runs on a machine that has one."""
    out = subprocess.run([sys.executable, "-c", _NO_CPU_FALLBACK], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]


def test_product_never_imports_oracle():
    """The oracle and the host emulator are test infrastructure: nothing under trex_gym_b200/ may
    import, include, link or load them."""
    pkg = os.path.join(ROOT, "trex_gym_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            path = os.path.join(dirpath, f)
            if f.endswith(".py"):
                text = open(path).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", text, flags=re.M), f
                assert "libtrex_oracle" not in text and "libtrex_emu" not in text, f
            elif f.endswith((".cu", ".h")):
                for inc in re.findall(r'#include\s+"([^"]+)"', open(path).read()):
                    assert "oracle" not in inc and "emu" not in inc and "tests/" not in inc, (f, inc)


def test_box_shim():
    from trex_gym_b200 import spaces

    b = spaces.Box(low=np.array([-1.0, 0.0]), high=np.array([1.0, 2.0]), dtype=np.float32)
    assert b.shape == (2,) and b.low.dtype == np.float32
    b.seed(0)
    for _ in range(10):
        assert b.contains(b.sample())
    rng, seed = spaces.np_random(123)
    assert seed == 123 and 0.0 <= rng.uniform() < 1.0


def test_shard_range():
    from trex_gym_b200.sharding import shard_range

    assert shard_range(0, 8, 65536) == (0, 65536)
    assert shard_range(7, 8, 65536) == (7 * 65536, 8 * 65536)
    with pytest.raises(ValueError):
        shard_range(8, 8, 1)


def _gloo_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from trex_gym_b200.sharding import allreduce_episode_stats, max_over_ranks, shard_range

    lo, hi = shard_range(rank, world, 1024)
    local = {"env_steps": hi - lo, "episodes": rank + 1, "sum_reward": -1.5 * (rank + 1)}
    tot = allreduce_episode_stats(local)
    tmax = max_over_ranks(0.1 * (rank + 1))
    q.put((rank, lo, hi, tot, tmax))
    dist.destroy_process_group()


def test_world_size_2_gloo_sharding_and_stats():
    """N > 1 path on CPU: disjoint shards, no step-path exchange, stats all-reduce, max-over-ranks timing."""
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    ps = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    out = sorted(q.get(timeout=120) for _ in range(2))
    for p in ps:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, lo0, hi0, t0, m0), (r1, lo1, hi1, t1, m1) = out
    assert (lo0, hi0, lo1, hi1) == (0, 1024, 1024, 2048)
    assert t0 == t1 and t0["env_steps"] == 2048 and t0["episodes"] == 3 and abs(t0["sum_reward"] + 4.5) < 1e-12
    assert abs(m0 - 0.2) < 1e-12 and abs(m1 - 0.2) < 1e-12


def test_f_alg_formula():
    sys.path.insert(0, ROOT)
    import bench

    # SURVEY.md section 8d reference points
    assert abs(bench.f_alg(5, 60, 0) - 0.98e6) < 0.02e6
    assert abs(bench.f_alg(5, 60, 8) - 1.85e6) < 0.03e6
    assert abs(bench.f_alg(5, 10, 0) - 0.42e6) < 0.02e6


def test_dump_outputs_writes_float32_and_samples_past_the_limit(tmp_path, monkeypatch):
    import torch

    sys.path.insert(0, ROOT)
    import bench

    obs = torch.arange(40 * 75, dtype=torch.float32).reshape(40, 75)
    done = torch.arange(40, dtype=torch.uint8) % 2
    bench.dump_outputs(str(tmp_path / "all"), {"obs": obs, "done": done})
    assert sorted(os.listdir(tmp_path / "all")) == ["done.npy", "obs.npy"]
    got = np.load(tmp_path / "all" / "done.npy")
    assert got.dtype == np.float32 and np.array_equal(got, done.numpy())
    # past the limit: the same seeded rows of every array, the same ones on every call
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 10 * 76 * 4 + 80)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"obs": obs, "done": done})
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 10 and len(set(idx)) == 10
    assert np.array_equal(np.load(tmp_path / "a" / "obs.npy"), obs.numpy()[idx.astype(int)])
    assert np.array_equal(np.load(tmp_path / "a" / "done.npy"), done.numpy()[idx.astype(int)])
    for name in ("env_index", "obs", "done"):
        assert np.array_equal(np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy")))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_BYTES


def test_bench_step_count_and_dump_arguments():
    """--steps is the number of timed steps: for the rollout workload it is the rollout horizon, a second, different count
    is refused; --steps 0 and a dump from the reference arm (which returns no arrays) are refused."""
    def run(*a):
        return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(a), capture_output=True, text=True, timeout=120)

    for a, msg in ((["--workload", "rollout", "--steps", "4", "--rollout-horizon", "8"], "--rollout-horizon"),
                   (["--steps", "0"], "--steps must be at least 1"),
                   (["--impl", "reference", "--steps", "1", "--dump-outputs", "x"], "--dump-outputs applies to --impl ours")):
        out = run(*a)
        assert out.returncode == 2 and msg in out.stderr, (a, out.stderr[-500:])


def test_reference_arm_prints_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3",
                          "--preroll", "5"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "env-steps/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["higher_is_better"] is True


def test_replay_export_layout():
    """SURVEY section 8f row 4: frames carry the base COM-frame pose and the joint angles by URDF joint name, in the
    record's joint order (pybullet link order of the revolute joints), so the reference side can play them back."""
    import numpy as np

    from trex_gym_b200.model_compiler import load_builtin
    from trex_gym_b200.replay import ReplayRecorder, joint_names_in_state_order

    model = load_builtin()
    names = joint_names_in_state_order(model)
    assert len(names) == 25 and names[0] == "joint_femur_right" and len(set(names)) == 25
    assert sorted(names) == list(model.meta["obs_joint_names"])  # the observation order is the name-sorted one
    # the recorder's frame dictionary, without a simulator: fill frames by hand
    rec = ReplayRecorder.__new__(ReplayRecorder)
    rec.names, rec.dt, rec.frames = names, 0.01, []
    f = np.zeros((1, 160), np.float32)
    f[0, 0:3] = [0.0, 0.0, 3.0]
    f[0, 3:7] = [0.0, 0.0, 0.0, 1.0]
    f[0, 13:38] = np.arange(25) * 0.01
    rec.frames = [f, f]
    d = rec.as_dict()
    assert d["joint_names"] == names and len(d["joint_positions"]) == 2 and len(d["joint_positions"][0]) == 25
    assert d["base_position"][0] == [0.0, 0.0, 3.0] and d["base_orientation_xyzw"][1] == [0.0, 0.0, 0.0, 1.0]
    assert abs(d["joint_positions"][0][3] - 0.03) < 1e-7


def test_replay_host_fk_and_playback_with_a_fake_pybullet(tmp_path):
    """The replay file is self-sufficient: host-side FK of a frame (replay.link_world_position) reproduces the golden head
    position of the reset pose (SURVEY.md section 7.1: (0.000, 3.100, 3.208)) and the oracle's head position at a bent
    pose; play_in_pybullet drives a (fake) pybullet through the frames with the calls the reference side needs."""
    import numpy as np

    from oracle.oracle import Oracle
    from trex_gym_b200.model_compiler import load_builtin
    from trex_gym_b200.replay import ReplayRecorder, joint_names_in_state_order, link_world_position, play_in_pybullet

    model = load_builtin()
    names = joint_names_in_state_order(model)
    q0 = np.zeros(25)
    for k, v in model.meta["starting_configuration"].items():
        q0[names.index(k)] = v
    assert np.allclose(link_world_position(model, [0, 0, 3.0], [0, 0, 0, 1.0], q0), model.meta["golden"]["reset_head_position"], atol=1e-9)
    o = Oracle(model.blob())
    o.reset()
    rng = np.random.default_rng(2)
    for _ in range(12):
        o.step(rng.uniform(-0.5, 0.5, 25))
    s = o.get_state()
    assert np.abs(link_world_position(model, s[0:3], s[3:7], s[13:38]) - o.head_position()).max() < 1e-9
    # playback
    rec = ReplayRecorder.__new__(ReplayRecorder)
    rec.names, rec.dt = names, 0.01
    f = np.zeros((1, 160), np.float32)
    f[0, 0:3], f[0, 3:7], f[0, 13:38] = s[0:3], s[3:7], s[13:38]
    rec.frames = [f, f, f]
    path = rec.save(str(tmp_path / "replay.json"))

    class FakePB:
        GUI, DIRECT, URDF_USE_INERTIA_FROM_FILE = 1, 2, 2

        def __init__(self):
            self.calls = []
            self.joint_names = list(model.meta["joint_names"])

        def connect(self, mode):
            self.calls.append(("connect", mode))

        def loadURDF(self, path, flags=0):
            self.calls.append(("loadURDF", path, flags))
            return 7

        def getNumJoints(self, body):
            return len(self.joint_names)

        def getJointInfo(self, body, i):
            return (i, self.joint_names[i].encode())

        def resetBasePositionAndOrientation(self, body, p, q):
            self.calls.append(("base", tuple(p), tuple(q)))

        def resetJointState(self, body, i, a):
            self.calls.append(("joint", i, a))

    pb = FakePB()
    assert play_in_pybullet(path, "/ref/assets/trex.urdf", realtime=False, pb=pb, gui=False) == 3
    assert pb.calls[0] == ("connect", FakePB.DIRECT) and pb.calls[1] == ("loadURDF", "/ref/assets/trex.urdf", 2)
    joints = [c for c in pb.calls if c[0] == "joint"]
    assert len(joints) == 3 * 25
    # joint k of the record goes to the pybullet joint index of its URDF name (pybullet link order)
    assert [c[1] for c in joints[:25]] == [model.meta["joint_names"].index(n) for n in names]
    assert np.allclose([c[2] for c in joints[:25]], s[13:38], atol=1e-6)
    assert len([c for c in pb.calls if c[0] == "base"]) == 3
