"""Cost of the external-wrench path (trex_config.external_forces = 1), one process on one GPU.

    python profiles/external_forces_bench.py [--envs 65536] [--steps 30] [--rounds 3] [--out profiles/external_forces_bench.json]

For the `random` and `standing` workloads of bench.py it alternates three configurations, round by round:
  off         external_forces = 0: the kernels without the wrench record
  zero        external_forces = 1, every wrench zero (results identical to `off`)
  pushed      external_forces = 1 with the push schedule on the base: a window of 50 env steps (0.5 s) holds one push of
              10 steps with probability 1, magnitude uniform in [10, 20] kN -- 0.2 to 0.4 of the animal's weight
              (5,180 kg): an impulse of 1,000-2,000 N s per push, which visibly moves a standing T-rex -- from step 0 of every
              episode
Each step is timed alone with CUDA events, the 126 MB L2 flushed (256 MiB fill, untimed) between steps, as bench.py does.
Prints one JSON line per workload and configuration with the median and spread over rounds, and the device name and power
limit it ran on.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return q


PUSHES = dict(interval=50, duration=10, probability=1.0, force=(1.0e4, 2.0e4), first_step=0)


def make(workload, config, n, preroll):
    import torch

    from trex_gym_b200.sim import TrexBatchSim

    sim = TrexBatchSim(n, device=0, external_forces=config != "off")
    if config == "pushed":
        sim.set_push_schedule("base", **PUSHES)
    if workload == "standing":
        names = list(sim.model.meta["obs_joint_names"])
        hold = np.zeros(25, np.float32)
        for k, v in sim.model.meta["starting_configuration"].items():
            hold[names.index(k)] = v
        acts = [torch.tensor(hold, device=sim.device).repeat(n, 1).contiguous()]
    else:
        acts = [sim.random_actions(step=t) for t in range(16)]
    for t in range(preroll):
        sim.step(acts[t % len(acts)])
    torch.cuda.synchronize()
    return sim, acts


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

    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--preroll", type=int, default=200)
    ap.add_argument("--workloads", default="random,standing")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("external_forces_bench needs a GPU")
    info = device_info()
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda:0", dtype=torch.float32)
    configs = ("off", "zero", "pushed")
    lines = []
    for wl in args.workloads.split(","):
        sims = {c: make(wl, c, args.envs, args.preroll) for c in configs}
        for c in configs:
            time_steps(*sims[c], 3, flush)  # warm-up
        ms = {c: [] for c in configs}
        for r in range(args.rounds):  # alternate the configurations round by round
            for c in configs:
                ms[c].append(time_steps(*sims[c], args.steps, flush))
        base = float(np.median(ms["off"]))
        for c in configs:
            med = float(np.median(ms[c]))
            line = {"workload": wl, "config": c, "envs": args.envs, "ms_per_step_median": med, "ms_per_round": ms[c],
                    "vs_off": med / base - 1.0, "device": info, "steps_per_round": args.steps, "rounds": args.rounds,
                    "l2": "flushed between timed steps (256 MiB fill, untimed); steps timed individually with CUDA events"}
            print(json.dumps(line), flush=True)
            lines.append(line)
        del sims
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
