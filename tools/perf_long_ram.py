"""Throughput of the global-memory ("long") fp64 Ramanujan periodogram (csrc/pp_long_ram.cu), CUDA events.

    python tools/perf_long_ram.py [--out FILE]

Each batch is a seeded `synth` batch, device-resident, timed after a warm-up call, periods 2 .. N // 3.  Reported per
size: windows/s, TFLOP/s on the canonical count of the dense contraction (2 sum q^2 flop per window, DESIGN.md 5.5)
and that rate over the DMMA peak pp_microbench measures in the same run.  N = 9 600 (max_length 3 200, the largest
on-chip plan) runs both paths; N = 16 384 with B = 1 is the shift form (a lone window).  The card's name and power
limit are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyperiod_b200 import RamanujanPeriods, _lib, synth  # noqa: E402
from pyperiod_b200._device import stage_windows  # noqa: E402


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


def flop_per_window(qmin, qmax):
    return 2.0 * sum(q * q for q in range(qmin, qmax + 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    peak = _lib.microbench(2)["per_s"]
    print(json.dumps({"dmma_peak_tflops": peak / 1e12}), flush=True)
    r = RamanujanPeriods()
    rows = []

    def row(n, b, ml, path, t):
        fl = flop_per_window(2, ml) * b
        rows.append({"N": n, "B": b, "max_length": ml, "path": path, "s": t, "windows_per_s": b / t,
                     "tflops": fl / t / 1e12, "of_dmma_peak": fl / t / peak})
        print(json.dumps(rows[-1]), flush=True)

    x = synth.synth_batch_device(256, 9600, 1, "cuda")
    w = stage_windows(x, r._device)
    for path, long in (("on_chip", False), ("long", True)):
        row(9600, 256, 3200, path, timed(lambda: r._norms_device(w, 2, 3200, _long=long)))
    for n, b in ((16384, 64), (16384, 1), (32768, 8), (65536, 1)):
        x = synth.synth_batch_device(b, n, 2, "cuda")
        row(n, b, n // 3, "long", timed(lambda: r.find_periods(x)))
    meta = {"card": card(), "dmma_peak_tflops": peak / 1e12, "rows": rows}
    print(json.dumps({"card": meta["card"]}))
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(meta, fh, indent=1)


if __name__ == "__main__":
    main()
