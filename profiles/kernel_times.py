"""Device time per kernel of one bench.py run, from torch.profiler (CUDA activities).

    python profiles/kernel_times.py [bench.py arguments]

Prints one line per trex_* kernel: launches, mean and total device time.  The default arguments time the headline
workload after a 300-step pre-roll.  Run it from the repository root; set TREX_LIB to time another build of the library.
"""
import os
import runpy
import sys

from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
args = sys.argv[1:] or ["--no-cpu-baseline", "--steps", "10", "--warmup", "3", "--preroll", "300", "--spread-steps", "0"]
sys.argv = ["bench.py"] + args
sys.path.insert(0, ROOT)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    try:
        runpy.run_path(os.path.join(ROOT, "bench.py"), run_name="__main__")
    except SystemExit:
        pass
for e in sorted(prof.key_averages(), key=lambda e: -e.device_time_total):
    if "trex_" not in e.key:
        continue
    name = e.key[e.key.find("trex_"):].split("(")[0]
    print("%-40s launches %7d  mean %9.2f us  total %9.1f ms" % (name, e.count, e.device_time_total / max(1, e.count),
                                                              e.device_time_total / 1e3), flush=True)
