"""Throughput of the global-memory ("long") path of QOPeriods: find_periods(num=4, thresh=0.05), CUDA events.

    python tools/perf_long_qo.py [--out FILE]

Each batch is a seeded `synth` batch, device-resident, timed after a warm-up call.  N = 16 384 and 65 536 run on the
long path at the default max_length (N // 3) and 2 048 (65 536: the default would make every round a sweep of
21 845 candidates over 64 K samples).  The last line compares the forced long path with the on-chip path at
N = 8 192.  The card's name and power limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyperiod_b200 import QOPeriods, synth  # noqa: E402


def timed(fn, reps=2):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, check=True)
        return q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError, IndexError):
        return torch.cuda.get_device_name(0) + ", power limit unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rows = []
    for n, b, ml in ((16384, 64, None), (65536, 16, 2048)):
        x = synth.synth_batch_device(b, n, 1, "cuda")
        t = timed(lambda: QOPeriods(staging="auto").find_periods(x, num=4, thresh=0.05, max_length=ml))
        rows.append({"N": n, "B": b, "max_length": ml or n // 3, "s": t, "windows_per_s": b / t})
        print(json.dumps(rows[-1]), flush=True)
    x = synth.synth_batch_device(256, 8192, 2, "cuda")
    t_on = timed(lambda: QOPeriods(staging="shared").find_periods(x, num=4, thresh=0.05))
    t_lg = timed(lambda: QOPeriods(staging="global").find_periods(x, num=4, thresh=0.05))
    rows.append({"N": 8192, "B": 256, "on_chip_windows_per_s": 256 / t_on, "long_windows_per_s": 256 / t_lg})
    print(json.dumps(rows[-1]), flush=True)
    meta = {"card": card(), "rows": rows}
    print(json.dumps({"card": meta["card"]}))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(meta, fh, indent=1)


if __name__ == "__main__":
    main()
