"""Cost of the dynamics query (trex_get_dynamics), one process on one GPU.

    python profiles/dynamics_bench.py [--envs 65536] [--launches 200] [--steps 30] [--rounds 3] [--out profiles/dynamics_bench.json]

On the `random` workload of bench.py after its pre-roll:
  query       the query for each output alone (M, b, J) and for all three in one launch, timed with CUDA events over
              `--launches` back-to-back launches, the 126 MB L2 flushed (256 MiB fill, untimed) before each window.  Bytes: the
              record, 640 B read per environment (plus the 128 B parameter row with env_params, not used here), and 3,844 B
              (M), 124 B (b) and 19,344 B (J) written per environment; achieved bandwidth against the data sheet's 7.7 TB/s of
              HBM3e (the kernel moves nothing else, so those bytes over that bandwidth are its lower bound)
  step        env step time without and with one full query (M, b and J) after every step, alternated round by round, each
              step timed alone with CUDA events and the L2 flushed between steps, as bench.py does
Prints one JSON line per measurement with the device name and power limit it ran on.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NDOF, NB = 31, 26
READ_B = 160 * 4  # per environment
WRITE_B = {"M": NDOF * NDOF * 4, "b": NDOF * 4, "J": NB * 6 * NDOF * 4}
HBM_TBS = 7.7


def device_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return q


def main():
    import torch

    from trex_gym_b200.sim import TrexBatchSim

    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--preroll", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dynamics_bench needs a GPU")
    info = device_info()
    n = args.envs
    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda:0", dtype=torch.float32)
    sim = TrexBatchSim(n, device=0)
    acts = [sim.random_actions(step=t) for t in range(16)]
    for t in range(args.preroll):
        sim.step(acts[t % 16])
    out = {"M": torch.empty(n, NDOF, NDOF, device=sim.device), "b": torch.empty(n, NDOF, device=sim.device),
           "J": torch.empty(n, NB, 6, NDOF, device=sim.device)}

    def query(which):
        sim._dynamics_query(*(out[k] if k in which else None for k in ("M", "b", "J")))

    lines = []
    for which in ("M", "b", "J", "MbJ"):  # each output alone, then all three in one launch
        for _ in range(10):
            query(which)
        flush.fill_(1.0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.launches):
            query(which)
        b.record()
        torch.cuda.synchronize()
        us = a.elapsed_time(b) * 1e3 / args.launches
        written = sum(WRITE_B[k] for k in which)
        bytes_total = n * (READ_B + written)
        lines.append({"measure": "query", "outputs": which, "envs": n, "us_per_launch": us, "launches": args.launches,
                      "bytes_read_per_env": READ_B, "bytes_written_per_env": written, "bytes_total": bytes_total,
                      "achieved_tb_s": bytes_total / (us * 1e-6) / 1e12, "bound": "HBM bandwidth (7.7 TB/s data sheet)",
                      "share_of_hbm_peak": bytes_total / (us * 1e-6) / 1e12 / HBM_TBS,
                      "floor_us": bytes_total / (HBM_TBS * 1e12) * 1e6, "device": info,
                      "l2": "flushed once before the window"})

    # env step without / with one full query per step
    def time_steps(with_query):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for k in range(args.steps):
            flush.fill_(float(k))
            evs[k][0].record()
            sim.step(acts[k % 16])
            if with_query:
                query("MbJ")
            evs[k][1].record()
        torch.cuda.synchronize()
        return float(np.median([x.elapsed_time(y) for x, y in evs]))

    time_steps(False)
    time_steps(True)
    ms = {False: [], True: []}
    for r in range(args.rounds):
        for q in (False, True):
            ms[q].append(time_steps(q))
    base = float(np.median(ms[False]))
    for q in (False, True):
        med = float(np.median(ms[q]))
        lines.append({"measure": "step_with_query" if q else "step", "workload": "random", "envs": n, "ms_per_step_median": med,
                      "ms_per_round": ms[q], "vs_step": med / base - 1.0, "steps_per_round": args.steps, "rounds": args.rounds,
                      "device": info, "l2": "flushed between timed steps (256 MiB fill, untimed); steps timed individually with CUDA events"})
    for line in lines:
        print(json.dumps(line), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
