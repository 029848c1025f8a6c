"""Cost of joint torque control (trex_config.actuation = TREX_ACTUATION_TORQUE), one process on one GPU.

    python profiles/actuation_bench.py [--envs 65536] [--steps 30] [--rounds 3] [--out profiles/actuation_bench.json]

Two measurements, position mode against torque mode, alternated round by round:
  front       the front kernel's time per launch (torch.profiler, CUDA activities), both handles stepped once from the SAME
              starting records (a position-mode trajectory of 200 random-action steps on the benchmark's default model):
              position mode with the benchmark's random targets, torque mode with random torques U(-2, 2) kN m
  step        the end-to-end env step, each mode on its own trajectory (random targets / random torques, 200 steps of
              pre-roll), each step timed alone with CUDA events and the 126 MB L2 flushed (256 MiB fill, untimed) between
              steps, as bench.py does.  The two modes reach different contact states, so this difference is not the cost of
              the torque term alone.
Prints one JSON line per measurement and mode with the median and spread over rounds, and the device name and power limit
it ran on.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TORQUE_SCALE = 2000.0  # N m: moves the joints without throwing the animal around (the model's bound is 3e5 N m)


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return q


def actions(sim, mode, n_sets=16):
    import torch

    if mode == "position":
        return [sim.random_actions(step=t) for t in range(n_sets)]
    g = torch.Generator(device=sim.device).manual_seed(0)
    return [(torch.rand(sim.num_envs, 25, device=sim.device, generator=g) * 2.0 - 1.0) * TORQUE_SCALE for _ in range(n_sets)]


def front_us_per_launch(sim, act, start):
    """Front-kernel time per launch (us) of one env step of `sim` from the records `start`."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    sim.set_state(start)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sim.step(act)
        torch.cuda.synchronize()
    total, count = 0.0, 0
    for ev in prof.events():
        if "trex_front_kernel" in ev.name and ev.device_type.name == "CUDA":
            total += ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
            count += 1
    if count == 0:
        raise RuntimeError("no trex_front_kernel launch in the profile")
    return total / count, count


def time_steps(sim, acts, steps, flush):
    import torch

    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        flush.fill_(float(k))
        evs[k][0].record()
        sim.step(acts[k % len(acts)])
        evs[k][1].record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in evs]))


def main():
    import torch

    from trex_gym_b200.sim import TrexBatchSim

    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--preroll", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("actuation_bench needs a GPU")
    info = device_info()
    modes = ("position", "torque")
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda:0", dtype=torch.float32)
    sims = {m: TrexBatchSim(args.envs, device=0, actuation=m) for m in modes}
    acts = {m: actions(sims[m], m) for m in modes}
    for t in range(args.preroll):
        for m in modes:
            sims[m].step(acts[m][t % len(acts[m])])
    torch.cuda.synchronize()
    start = sims["position"].get_state().clone()  # the shared starting records of the front-kernel measurement
    ends = {m: sims[m].get_state().clone() for m in modes}  # each mode's own trajectory, for the step measurement
    lines = []
    front = {m: [] for m in modes}
    launches = {}
    for m in modes:
        front_us_per_launch(sims[m], acts[m][0], start)  # warm-up (profiler and kernels)
    for r in range(args.rounds):
        for m in modes:
            us, launches[m] = front_us_per_launch(sims[m], acts[m][r % len(acts[m])], start)
            front[m].append(us)
    for m in modes:
        sims[m].set_state(ends[m])
        time_steps(sims[m], acts[m], 3, flush)  # warm-up
    step = {m: [] for m in modes}
    for r in range(args.rounds):
        for m in modes:
            step[m].append(time_steps(sims[m], acts[m], args.steps, flush))
    for what, data, unit in (("front", front, "us_per_launch"), ("step", step, "ms_per_step")):
        base = float(np.median(data["position"]))
        for m in modes:
            med = float(np.median(data[m]))
            line = {"measurement": what, "actuation": m, "envs": args.envs, unit + "_median": med, unit + "_per_round": data[m],
                    "vs_position": med / base - 1.0, "device": info, "rounds": args.rounds}
            if what == "front":
                line["launches_per_step"] = launches[m]
                line["start"] = "the same records for both modes (position-mode trajectory, %d steps)" % args.preroll
            else:
                line["steps_per_round"] = args.steps
                line["l2"] = "flushed between timed steps (256 MiB fill, untimed); steps timed individually with CUDA events"
                line["note"] = "each mode on its own trajectory: different contact states, not the torque term's cost alone"
            print(json.dumps(line), flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
