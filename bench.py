#!/usr/bin/env python
"""bench.py -- env-steps/s of the trex-gym hot path at 65,536 envs/GPU (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores

One "step" = one TrexBulletEnv.step (5 fused physics substeps + obs + reward + done) over the whole
batch of synthetic random actions.  One process per GPU (torchrun for N > 1); environments shard
across ranks with NO step-path communication (weak scaling); NCCL is used only for the barrier and
the max-over-ranks of the device time.  Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ENVS_PER_GPU = 65536
B_ALG = 909.0  # algorithmic HBM bytes per env-step (SURVEY.md section 8d)
# algorithmic FLOPs per env-step (SURVEY.md section 8d, frozen planning constants)
C_ABA, C_RESP, C_ROW, C_INT, C_OBS, N_B = 500.0, 1900.0, 90.0, 200.0, 150.0, 26.0


def f_alg(n_sub, mean_iters, mean_contacts, mean_limit_rows=0.0):
    R = 25.0 + mean_limit_rows + 3.0 * mean_contacts
    return n_sub * (N_B * C_ABA + R * C_RESP + mean_iters * R * C_ROW + C_INT) + C_OBS


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu_index = gpu_index
        self.samples = []
        self.source = "nvidia-smi"
        self._halt = threading.Event()

    def _nvml_loop(self):
        """Fast path: NVML in-process (a sample every 20 ms); returns False if NVML is not usable."""
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu_index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            bits = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)]
        except Exception:  # noqa: BLE001
            return False
        self.source = "nvml (same fields as the nvidia-smi clocks query, sampled every 20 ms)"
        while not self._halt.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = int(get_reasons(h))
                self.samples.append([str(self.gpu_index), str(sm), str(mx), "", hex(r)] + ["Active" if r & b else "Not Active" for _, b in bits])
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.02)
        return True

    def run(self):
        if self._nvml_loop():
            return
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    p = [x.strip() for x in line.split(",")]
                    if len(p) >= 9:
                        self.samples.append(p)
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for p in self.samples:
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": self.source}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def oracle_workers(n_threads, steps_per_worker, warmup, seed=0, preroll=0):
    """The reference algorithm (oracle port of pybullet's pipeline) on host cores: one double-precision
    environment per worker thread (the reference is one env per process), same action distribution."""
    from oracle.oracle import Oracle
    from trex_gym_b200.model_compiler import load_builtin

    model = load_builtin()
    blob = model.blob()
    lo = model["mb_lower"][1:][model["obs_dof"]]
    hi = model["mb_upper"][1:][model["obs_dof"]]
    orcs = [Oracle(blob) for _ in range(n_threads)]
    acts = []
    for w in range(n_threads):
        rng = np.random.Generator(np.random.Philox(key=seed + w))
        acts.append(rng.uniform(lo, hi, size=(warmup + steps_per_worker, 25)))
        orcs[w].reset()
    times = [0.0] * n_threads

    def work(w):
        if preroll:
            rng = np.random.Generator(np.random.Philox(key=10_000 + seed + w))
            orcs[w].run(rng.uniform(lo, hi, size=(preroll, 25)), want_obs=False)
        orcs[w].run(acts[w][:warmup], want_obs=False)
        t0 = time.perf_counter()
        orcs[w].run(acts[w][warmup:], want_obs=False)
        times[w] = time.perf_counter() - t0

    ths = [threading.Thread(target=work, args=(w,)) for w in range(n_threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    wall = time.perf_counter() - t0
    mean_iters = float(np.mean([o.total_iterations / max(1, o.total_substeps) for o in orcs]))
    return n_threads * steps_per_worker / max(times), max(times), wall, mean_iters


def pybullet_available():
    """(module, reference checkout) when the real reference path can run here, else (None, reason)."""
    try:
        import pybullet as pb
    except ImportError as e:
        return None, "pybullet not importable (%s)" % e
    for cand in (os.environ.get("TREX_GYM_REFERENCE"), os.path.join(ROOT, "baseline", "_ref"), "/root/reference"):
        if cand and os.path.isfile(os.path.join(cand, "assets", "trex.urdf")):
            return pb, cand
    return None, "pybullet importable but no trex-gym checkout with assets/trex.urdf (set TREX_GYM_REFERENCE)"


def _pybullet_worker(args):
    """One process = one TrexBulletEnv-equivalent pybullet DIRECT client (the reference is one env per process)."""
    ref_dir, n_steps, warmup, seed = args
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import pybullet as pb
    import record_pybullet_golden as rec

    os.environ.setdefault("TREX_GYM_REFERENCE", ref_dir)
    from trex_gym_b200.model_compiler import emit_derived_urdf, load_builtin

    out = os.path.join("/tmp", "trex_bench_derived_%d" % os.getpid())
    os.makedirs(out, exist_ok=True)
    urdf = emit_derived_urdf(os.path.join(ref_dir, "assets", "trex.urdf"), os.path.join(out, "trex_contacts.urdf"), model=load_builtin())
    loop = rec.ReferenceLoop(pb, os.path.join(ref_dir, "assets", "floor.urdf"), urdf, inertia_from_file=True)
    rng = np.random.Generator(np.random.Philox(key=seed))
    acts = rng.uniform(loop.low, loop.high, size=(warmup + n_steps, 25))
    for t in range(warmup):
        loop.step(acts[t])
    t0 = time.perf_counter()
    for t in range(warmup, warmup + n_steps):
        loop.step(acts[t])
    return time.perf_counter() - t0


def pybullet_workers(ref_dir, n_procs, steps_per_worker, warmup):
    import multiprocessing as mp

    with mp.get_context("spawn").Pool(n_procs) as pool:
        times = pool.map(_pybullet_worker, [(ref_dir, steps_per_worker, warmup, w) for w in range(n_procs)])
    return n_procs * steps_per_worker / max(times), max(times)


def cpu_reference(cores, steps_per_worker, warmup, preroll):
    """The reference's CPU path on `cores` host cores: real pybullet when this box has one (BASELINE.md section 3), else the
    double-precision port (oracle/).  Returns (value, seconds, kind, note, mean_iters)."""
    pb, where = pybullet_available()
    if pb is not None:
        v, tmax = pybullet_workers(where, cores, steps_per_worker, warmup + preroll)
        return v, tmax, "pybullet", "pybullet DIRECT, one process per core, derived <collision> URDF, inertia from file (%s)" % where, None
    v, tmax, wall, mi = oracle_workers(cores, steps_per_worker, warmup, preroll=preroll)
    return v, tmax, "port", "CPU restatement of pybullet's algorithm (oracle/trex_oracle.c), not pybullet: %s" % where, mi


def run_reference(args):
    rank, world, local = dist_setup(args.gpus)
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    per_step = 16  # env-steps per worker per bench "step": a bounded sample of the 65,536-env batch
    total_steps = per_step * args.steps
    value, tmax, kind, note, mean_iters = cpu_reference(cores, total_steps, per_step * args.warmup, args.preroll)
    sample = "%d workers x %d env-steps each (one double-precision env per worker, random actions after %d untimed pre-roll steps)" % (cores, total_steps, args.preroll)
    line = {
        "impl": "reference", "metric": "env-steps/sec at 65,536 envs/GPU", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tmax / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "65,536 envs/GPU, random actions (configs[2]); reference arm = bounded sample of %d env-steps per step on host cores" % (cores * per_step),
                   "num_substeps": 5, "solver_iterations": 60, "mean_solver_iterations": mean_iters},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample, "note": note},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
# Workloads (BASELINE.json configs; one command each, see profiles/README.md)
# ---------------------------------------------------------------------------------------------------------------
WORKLOADS = {
    # name: (default envs/GPU, description)
    "random": (65536, "random actions U(low,high) Philox-keyed by (seed,global env,step), pre-rolled into the steady regime (BASELINE.json configs[2])"),
    "c2": (4096, "4,096 envs, random actions (BASELINE.json configs[1]: the parity-test batch)"),
    "standing": (65536, "every env holds the reset pose and stands on both feet (12-16 contacts each): the regime a trained policy produces"),
    "fallen": (65536, "fallen starts (reset_mode 1: base z U(0.3,3), uniform SO(3), joints U(limits)), horizon 64 with auto-reset, random actions (BASELINE.json configs[4])"),
    "rollout": (16384, "PPO rollout loop on the device: MlpPolicy.act_into + step_into per step, trex_gae at the end (BASELINE.json configs[3])"),
}
ACTION_SETS = 16  # pre-generated action sets cycled through the timed steps
DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this much


def dump_outputs(out_dir, arrays):
    """Write the arrays one step returns (one row per environment) as ``out_dir/<name>.npy`` in float32, so that two builds
    can be compared output for output.  When they exceed DUMP_BYTES together, every array keeps the same fixed, seeded
    sample of environments, whose indices go to ``env_index.npy``."""
    host = {k: v.detach().cpu().numpy().astype(np.float32) for k, v in arrays.items()}
    n = len(next(iter(host.values())))
    row_bytes = sum(a[0].nbytes for a in host.values())
    if n * row_bytes > DUMP_BYTES:
        keep = (DUMP_BYTES - 4096) // (row_bytes + 8)
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        host = {k: a[idx] for k, a in host.items()}
        host["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def source_hash():
    """sha256 over the kernel sources: keys the ncu-derived DRAM traffic figure to the build it was measured on."""
    import hashlib

    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "trex_gym_b200", "csrc")
    for name in sorted(os.listdir(csrc)):
        if name.endswith((".h", ".cu")):
            with open(os.path.join(csrc, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def lookup_traffic(workload, n, n_sub):
    """DRAM bytes per env step of `workload` from profiles/traffic.json (written by profiles/measure_traffic.py from an
    `ncu --set full` capture); None -- with the reason -- when the capture belongs to another build or configuration."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tr = json.load(f)
    except Exception:  # noqa: BLE001
        return None, "no profiles/traffic.json"
    if tr.get("source_hash") != source_hash():
        return None, "profiles/traffic.json was measured on kernel sources %s, this build is %s: re-run profiles/measure_traffic.py" % (tr.get("source_hash"), source_hash())
    e = tr.get("workloads", {}).get(workload)
    if not e or e.get("envs") != n or e.get("num_substeps") != n_sub:
        return None, "profiles/traffic.json has no entry for this workload / batch size"
    return int(e["bytes_per_env_step_batch"]), "ncu dram__bytes_read.sum + dram__bytes_write.sum over the kernels of one env step (%s)" % e.get("capture", "")


def make_batch(workload, n, local, rank, args):
    """Simulator + per-step action source of a workload, pre-rolled into its steady regime."""
    import torch

    from trex_gym_b200.sim import TrexBatchSim

    env_offset = rank * n
    kw = dict(device=local, contacts=not args.no_contacts, num_substeps=args.substeps, warps_per_block=args.warps_per_block,
              env_offset=env_offset, max_episode_steps=args.horizon)
    if workload == "fallen":
        kw.update(reset_mode=1, max_episode_steps=args.horizon or 64, seed=11)
    if workload == "rollout":
        kw.update(distance_weight=200.0, energy_weight=1e-6, drift_weight=1.0)  # trex_train.py:66
    sim = TrexBatchSim(n, **kw)
    if workload == "standing":
        names = list(sim.model.meta["obs_joint_names"])
        hold = np.zeros(25, np.float32)
        for k, v in sim.model.meta["starting_configuration"].items():
            hold[names.index(k)] = v
        acts = [torch.tensor(hold, device=sim.device).repeat(n, 1).contiguous()]
        for _ in range(args.preroll):
            sim.step(acts[0])
    else:
        acts = [sim.random_actions(step=t, seed=0, env_offset=env_offset) for t in range(ACTION_SETS)]
        # untimed pre-roll: bring the batch from the reset pose (0.25 m above the floor) to the steady regime of THIS action
        # process (the 16 sets cycling: pre-rolling with other actions leaves a transient of ~50 steps in the timed region)
        for t in range(args.preroll):
            sim.step(acts[t % ACTION_SETS])
    return sim, acts


def run_rollout(args, rank, world, local, dev, use_dist, barrier):
    """configs[3]: the PPO rollout loop of trex_train.py:44-61 on the device -- policy forward (fused kernel), env step into
    the time-major buffers, GAE(0.95, 0.99) at the end.  A 'step' is one env step of the loop; value = N*T / loop time."""
    import torch

    from trex_gym_b200.rollout import MlpPolicy, RolloutBuffer, RunningMeanStd

    n, T = args.envs_per_gpu, args.rollout_horizon
    sim, _ = make_batch("rollout", n, local, rank, args)
    rms = RunningMeanStd(75, sim.device)
    pol = MlpPolicy(sim.device, seed=1, rms=rms)
    buf = RolloutBuffer(sim, T)
    rms.update(buf.obs[0])
    last_v = torch.zeros(n, device=dev)
    warm = RolloutBuffer(sim, max(3, args.warmup))
    warm.collect(policy=pol, seed=3)
    buf.obs[0].copy_(warm.obs[-1])
    del warm
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = sim.kernel_launches
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    buf.collect(policy=pol, seed=4)
    e1.record()
    pol.act_into(buf.obs[T], torch.empty(n, 25, device=dev), last_v, None, step=T, seed=4, env_offset=sim.env_offset)
    buf.compute_gae(last_v)
    e2.record()
    barrier()
    sampler.stop()
    loop_ms, gae_ms = e0.elapsed_time(e1), e1.elapsed_time(e2)
    t_ms = torch.tensor([loop_ms + gae_ms], device=dev, dtype=torch.float64)
    if use_dist:
        import torch.distributed as dist

        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    total_ms = float(t_ms.item())
    st = sim.stats()
    if args.dump_outputs and rank == 0:  # the rows of the loop's last env step
        dump_outputs(args.dump_outputs, {"obs": buf.obs[T], "action": buf.actions[T - 1], "reward": buf.rewards[T - 1], "done": buf.dones[T],
                                         "value": buf.values[T - 1], "neglogp": buf.neglogp[T - 1],
                                         "advantage": buf.advantages[T - 1], "return": buf.returns[T - 1]})
    if rank == 0:
        launches = sim.kernel_launches - l0 + T + 2  # + one policy kernel per step, the bootstrap value, the GAE scan
        line = {
            "metric": "env-steps/sec at 65,536 envs/GPU", "value": world * n * T / (total_ms * 1e-3), "unit": "env-steps/s", "n_gpus": world,
            "steps": T, "warmup": max(3, args.warmup), "ms_per_step": total_ms / T, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "rollout: %d envs/GPU x %d-step horizon, %s" % (n, T, WORKLOADS["rollout"][1]), "envs_per_gpu": n,
                       "rollout_horizon": T, "num_substeps": sim.num_substeps, "policy": "MlpPolicy 75-64-64-25 + value head, random init, obs filter on",
                       "buffers_gb": round((buf.obs.numel() + buf.actions.numel() + 6 * buf.rewards.numel()) * 4 / 1e9, 2),
                       "gae_ms": gae_ms, "mean_contacts_per_env": st["mean_contacts"], "mean_solver_iterations": st["mean_solver_iterations"],
                       "l2": "working set (obs/action rows of the step, %.0f MB of work records) exceeds L2; no flush" % (n * 11392 / 1e6)},
            "e2e": {"value": world * n * T / (total_ms * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "the rollout loop is device-resident by design (no per-step host traffic): e2e = value"},
            "gpu_launches": int(launches), "clocks": sampler.summary(),
        }
        print(json.dumps(line), flush=True)


def run_ours(args):
    import torch

    from trex_gym_b200 import _native

    rank, world, local = dist_setup(args.gpus)
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if args.gpus > 1 and world == 1:
        raise SystemExit("launch with torchrun for --gpus > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    workload = args.workload
    if args.envs_per_gpu <= 0:
        args.envs_per_gpu = WORKLOADS[workload][0]
    if workload == "rollout":
        run_rollout(args, rank, world, local, dev, use_dist, barrier)
        if use_dist:
            dist.barrier()
            dist.destroy_process_group()
        return
    n = args.envs_per_gpu
    sim, acts = make_batch(workload, n, local, rank, args)
    ring = len(acts)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev, dtype=torch.float32)

    # ---- device-resident throughput ("value") -------------------------------------------------
    phase0 = args.preroll if workload != "standing" else 0  # keep cycling where the pre-roll stopped
    step_fn = sim.step
    if getattr(args, "graph", False):
        sim.capture_graph()
        step_fn = sim.step_graph
    for t in range(args.warmup):
        step_fn(acts[(phase0 + t) % ring])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = sim.kernel_launches
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for k in range(args.steps):
        flush.fill_(float(k))  # L2 flush between timed steps (not timed)
        evs[k][0].record()
        out = step_fn(acts[(phase0 + args.warmup + k) % ring])
        evs[k][1].record()
    barrier()
    if args.dump_outputs and rank == 0:  # before the spread and e2e steps overwrite the simulator-owned buffers
        dump_outputs(args.dump_outputs, dict(zip(("obs", "reward", "done"), out)))
    launches = sim.kernel_launches - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    st = sim.stats()
    it_sum, ct_sum = st["mean_solver_iterations"], st["mean_contacts"]
    t_ms = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
    if use_dist:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t_ms.item())
    value = world * n * args.steps / (dev_ms_max * 1e-3)

    # ---- spread of the step time over a longer window (the regime drifts with the action sequence) -------------
    spread = None
    if args.spread_steps > 0:
        sevs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.spread_steps)]
        for k in range(args.spread_steps):
            flush.fill_(float(k))
            sevs[k][0].record()
            step_fn(acts[(phase0 + args.warmup + args.steps + k) % ring])
            sevs[k][1].record()
        barrier()
        ms = np.asarray([a.elapsed_time(b) for a, b in sevs])
        s2 = sim.stats()
        spread = {"steps": int(args.spread_steps), "action_sets": ring, "ms_first10_mean": float(ms[:10].mean()), "ms_last10_mean": float(ms[-10:].mean()), "ms_p10": float(np.percentile(ms, 10)), "ms_p50": float(np.percentile(ms, 50)),
                  "ms_p90": float(np.percentile(ms, 90)), "ms_mean": float(ms.mean()), "ms_max": float(ms.max()),
                  "mean_contacts_per_env_at_end": s2["mean_contacts"], "nan_resets": s2["nan_resets"]}

    # ---- end to end through the host-buffer entry point ("e2e") ----------------------------------
    h_act = [a.cpu().pin_memory() for a in acts]
    h_obs = torch.empty(n, 75, dtype=torch.float32).pin_memory()
    h_rew = torch.empty(n, dtype=torch.float32).pin_memory()
    h_done = torch.empty(n, dtype=torch.uint8).pin_memory()
    for t in range(max(1, args.warmup)):
        sim.step_host(h_act[t % ring], h_obs, h_rew, h_done)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        sim.step_host(h_act[k % ring], h_obs, h_rew, h_done)  # H2D actions, step, D2H obs/reward/done, sync
    barrier()
    e2e_s = time.perf_counter() - t0
    t_e = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if use_dist:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * n * args.steps / float(t_e.item())
    # the same through the depth-1 pipelined entry point (copies of step k under step k+1), two sets of pinned arrays
    h_set = [(h_obs, h_rew, h_done), (torch.empty_like(h_obs).pin_memory(), torch.empty_like(h_rew).pin_memory(), torch.empty_like(h_done).pin_memory())]
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        sim.step_host_async(h_act[k % ring], *h_set[k & 1])
    sim.host_wait()
    barrier()
    t_p = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if use_dist:
        dist.all_reduce(t_p, op=dist.ReduceOp.MAX)
    e2e_pipelined = world * n * args.steps / float(t_p.item())
    sampler.stop()
    clocks = sampler.summary()

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:  # noqa: BLE001
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        tf = _native.ctypes.c_double(0.0)
        _native.check(_native.lib().trex_measure_fp32_peak(local, _native.ctypes.byref(tf)), "trex_measure_fp32_peak")
        fp32_peak = float(tf.value)
        kernel_ms = dev_ms / args.steps  # all kernels of one env step (rank 0's own device time)
        traffic, traffic_note = (lookup_traffic(workload, n, sim.num_substeps) if not args.no_contacts and not os.environ.get("TREX_CHUNK")
                                 else (None, "profiles/traffic.json has no entry for this configuration"))
        flops = f_alg(sim.num_substeps, it_sum, ct_sum) * n
        achieved_tf = flops / (kernel_ms * 1e-3) / 1e12
        hbm_gbs = B_ALG * n / (kernel_ms * 1e-3) / 1e9
        cfg = {"workload": "%s: %d envs/GPU, %s%s" % (workload, n, WORKLOADS[workload][1], "" if not args.no_contacts else "; literal collision-less URDF (free fall)"),
               "envs_per_gpu": n, "num_substeps": sim.num_substeps, "solver_iterations": int(300 / sim.num_substeps),
               "mean_solver_iterations": it_sum, "mean_contacts_per_env": ct_sum, "horizon": args.horizon or (64 if workload == "fallen" else 0),
               "preroll_steps": args.preroll, "action_sets": ring, "ms_timed_first": float(evs[0][0].elapsed_time(evs[0][1])), "ms_timed_last": float(evs[-1][0].elapsed_time(evs[-1][1])),
               "l2": "flushed between timed steps (256 MiB fill, untimed); steps timed individually with CUDA events",
               "parallelism": "envs sharded over %d GPU(s), no step-path collective" % world}
        if spread:
            cfg["spread"] = spread
        line = {
            "metric": "env-steps/sec at 65,536 envs/GPU", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": n * 25 * 4, "d2h_bytes_per_step": n * (75 * 4 + 4 + 1),
                    "pipelined_value": e2e_pipelined,
                    "note": "value: synchronous trex_step_host (numpy in / numpy out, what a gym caller sees); pipelined_value: trex_step_host_async, the same copies overlapped with the neighbouring steps"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "fp32", "achieved": achieved_tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved_tf / fp32_peak if fp32_peak else None,
                         "traffic": traffic, "traffic_source": traffic_note,
                         "kernel": "one env step = %d x (trex_front_kernel; then concurrently trex_solve_tm_kernel (1-8 contacts, contact stash in tensor memory), trex_solve_kernel<0> (contact free), trex_heavy_kernel x 2 (9-16 contacts: tensor-memory and shared-memory instance)) + trex_tail_kernel, per group of environments; shares of the device time in profiles/r2t_launches_random.txt" % sim.num_substeps,
                         "kernel_ms": kernel_ms,
                         "peak_source": "measured in this run: register-resident FFMA microbenchmark (trex_measure_fp32_peak); MEASURED_PEAKS.json has no FP32 figure",
                         "flops_per_env_step": f_alg(sim.num_substeps, it_sum, ct_sum),
                         "hbm": {"achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak, "bytes_per_env_step": B_ALG, "peak_source": hbm_src}},
        }
        if world == 1 and not args.no_cpu_baseline:
            cores = len(os.sched_getaffinity(0))
            steps_pw = 400
            t0 = time.perf_counter()
            v, tmax, kind, note, mi = cpu_reference(cores, steps_pw, 20, args.preroll)
            line["cpu_baseline"] = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": kind,
                                    "sample": "%d workers x %d env-steps (one f64 env each, random actions after %d pre-roll steps), %.1f s" % (cores, steps_pw, args.preroll, time.perf_counter() - t0),
                                    "mean_solver_iterations": mi, "note": note}
        print(json.dumps(line), flush=True)
    if use_dist:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed env steps of the loop that gives the value and --dump-outputs (default 20; with --workload rollout the rollout "
                         "horizon, default 2048).  After it, the e2e figures time 2 x K more steps through the host entry points, and "
                         "--spread-steps more are timed for the spread")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="random", choices=sorted(WORKLOADS), help="default: BASELINE.json configs[2], the headline")
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="0 = the workload's own batch size (65,536 for the headline)")
    ap.add_argument("--spread-steps", type=int, default=-1, help="extra individually timed steps for the step-time spread (default: 200 for the headline at N=1, else 0)")
    ap.add_argument("--rollout-horizon", type=int, default=None, help="env steps of the timed rollout loop (default: --steps if given, else 2048)")
    ap.add_argument("--substeps", type=int, default=5)
    ap.add_argument("--horizon", type=int, default=0, help="max episode steps (0 = reference behaviour: never terminate)")
    ap.add_argument("--no-contacts", action="store_true", help="literal reference URDF (no collision shapes)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--warps-per-block", type=int, default=0)
    ap.add_argument("--graph", action="store_true", help="device-resident value through the CUDA-graph replay of the step (TrexBatchSim.step_graph)")
    ap.add_argument("--preroll", type=int, default=300, help="untimed env-steps from the reset state before warm-up, so the batch is in its steady regime (on the floor, in contact)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (rank 0's environments) as "
                    "DIR/<name>.npy in float32; past 64 MB, a fixed seeded sample of the environments")
    args = ap.parse_args()
    if args.impl == "ours" and args.workload == "rollout":
        # the rollout loop is the timed window: its horizon is the number of timed steps
        if args.steps is not None and args.rollout_horizon is not None and args.steps != args.rollout_horizon:
            ap.error("--steps and --rollout-horizon both set the timed steps of the rollout loop; give one of them")
        given = [v for v in (args.rollout_horizon, args.steps) if v is not None]
        args.steps = args.rollout_horizon = given[0] if given else 2048
    elif args.steps is None:
        args.steps = 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours: the reference arm times host workers and returns no arrays")
    if args.warmup < 3:
        args.warmup = 3
    if args.spread_steps < 0:
        args.spread_steps = 200 if (args.workload == "random" and args.gpus == 1) else 0
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
