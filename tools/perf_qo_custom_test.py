"""QOPeriods.find_periods with a custom test_function: the batched driver against a loop of 1-D calls, both bases.

    python tools/perf_qo_custom_test.py [--windows B] [--loop-windows L] [--repeats R] [--out FILE]

Config 5's shape: B = 4096 device-resident windows of N = 4096 samples (seeded `synth` batch), num = 4, the default
stop rule written out as the test (rms(reconstruction) > 0.05 rms(data)).  The batched call is timed with a host clock
around a call that ends in a synchronise (the driver synchronises every round), after a warm-up call; the median of
R calls (default 5) is reported with the fastest and slowest.  The loop of 1-D calls runs over the first L windows
(default 256) and is reported per window.  A further, profiled run of the batched call (torch.profiler, CUDA activities) splits its wall time into kernel time, copy time, time inside the
test function and the rest (host calls, Python bookkeeping, launch gaps).  The card's name and power limit are read
in the same run and printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyperiod_b200 import QOPeriods, synth  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, check=True)
        return q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError, IndexError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


class Test:
    """The default stop rule as a host callable; accumulates the time spent inside it."""

    def __init__(self):
        self.s, self.calls = 0.0, 0

    def __call__(self, _self, a, y):
        t0 = time.perf_counter()
        go = np.sqrt(np.sum(y * y) / len(y)) > np.sqrt(np.sum(a * a) / len(a)) * 0.05
        self.s += time.perf_counter() - t0
        self.calls += 1
        return go


def wall(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def busy_us(intervals):
    """Length of the union of [start, end) intervals (us)."""
    total, end = 0.0, -1e300
    for a, b in sorted(intervals):
        if b <= end:
            continue
        total += b - max(a, end)
        end = b
    return total


def profiled(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        t = wall(fn)
    kern, copy = [], []
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        iv = (e.time_range.start, e.time_range.end)
        (copy if e.name.startswith("Memcpy") else kern).append(iv)
    return t, busy_us(kern) / 1e6, busy_us(copy) / 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=4096)
    ap.add_argument("--loop-windows", type=int, default=256)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    n, num = 4096, 4
    x = synth.synth_batch_device(args.windows, n, 5, "cuda")
    rows = []
    for basis in ("natural", "ramanujan"):
        q = QOPeriods(basis_type=basis)
        run = lambda t: q.find_periods(x, num=num, thresh=None, test_function=t)   # noqa: E731
        run(Test())                                    # warm-up: module loads, workspaces, tables
        times = sorted(wall(lambda: run(Test())) for _ in range(args.repeats))
        t_batch = times[len(times) // 2]
        m = min(args.loop_windows, args.windows)
        q.find_periods(x[0], num=num, thresh=None, test_function=Test())
        t_loop = wall(lambda: [q.find_periods(x[b], num=num, thresh=None, test_function=Test()) for b in range(m)])
        tf = Test()
        t_prof, t_kern, t_copy = profiled(lambda: run(tf))
        row = {"basis": basis, "B": args.windows, "N": n, "num": num,
               "batched_s": t_batch, "batched_s_min_max": [times[0], times[-1]],
               "batched_windows_per_s": args.windows / t_batch,
               "loop_windows": m, "loop_s_per_window": t_loop / m, "loop_windows_per_s": m / t_loop,
               "speedup": (t_loop / m) / (t_batch / args.windows),
               "profiled_wall_s": t_prof, "kernel_s": t_kern, "memcpy_s": t_copy, "test_function_s": tf.s,
               "test_calls": tf.calls, "host_rest_s": max(t_prof - t_kern - t_copy - tf.s, 0.0)}
        rows.append(row)
        print(json.dumps(row), flush=True)
    meta = {"card": card(), "rows": rows}
    print(json.dumps({"card": meta["card"]}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(meta, f, indent=1)


if __name__ == "__main__":
    main()
