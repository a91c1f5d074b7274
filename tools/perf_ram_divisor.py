"""Throughput of the divisor-form fp64 Ramanujan periodogram (RamanujanPeriods(method="divisor"),
csrc/pp_ram_divisor.cu) against the dense fp64 path, CUDA events.

    python tools/perf_ram_divisor.py [--out FILE] [--budget-s 20]

Every batch is a seeded `synth` batch, device-resident.  Each timed call is preceded by a warm-up call of the same
shape; where both methods are timed they alternate in this process (dense, divisor, dense, divisor, ...).  Reported
per case: seconds per call, windows/s and, for the on-chip divisor kernel, the fold's share of the shared-memory bound
(every period reads the N staged samples once: B * Q * N * 8 bytes over the shared-memory peak pp_microbench measures
in this run).  Cases: config 5 (65 536 x 4 096, q = 2 .. 1 365, find_periods and find_periods_with_weights(thresh=0.2));
N = 16 384, B = 64 (dense: the global-memory path); N = 131 072, B = 8 and 1; N = 2^20, B = 1 (divisor only).  At
N = 2^20 the top 2 048 periods are timed first; the full range (2 .. 349 525) runs only when that slice projects it
under --budget-s, and is reported as not measured otherwise.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyperiod_b200 import RamanujanPeriods, _lib, synth  # noqa: E402


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


def alternate(fns, rounds=2):
    """Seconds per call of each of fns, timed in alternation (one warm-up of each first)."""
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    acc = {k: 0.0 for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            acc[k] += _once(f)
    return {k: v / rounds for k, v in acc.items()}


def _once(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3


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
    ap.add_argument("--budget-s", type=float, default=20.0)
    args = ap.parse_args()
    smem_peak = _lib.microbench(0)["per_s"]
    print(json.dumps({"card": card(), "smem_peak_TBps": smem_peak / 1e12}), flush=True)
    dense, div = RamanujanPeriods(), RamanujanPeriods(method="divisor")
    rows = []

    def row(case, n, b, qmin, qmax, method, t, fold_share=None):
        rows.append({"case": case, "N": n, "B": b, "qmin": qmin, "qmax": qmax, "method": method, "s": t,
                     "windows_per_s": b / t})
        if fold_share is not None:
            rows[-1]["fold_share_of_smem_bound"] = fold_share
        print(json.dumps(rows[-1]), flush=True)

    # config 5
    n, b, ml = 4096, 65536, 1365
    x = synth.synth_batch_device(b, n, 1, "cuda")
    fold_bound = b * (ml - 1) * n * 8 / smem_peak
    ts = alternate({"dense": lambda: dense.find_periods(x), "divisor": lambda: div.find_periods(x)})
    row("config5 find_periods", n, b, 2, ml, "dense", ts["dense"])
    row("config5 find_periods", n, b, 2, ml, "divisor", ts["divisor"], fold_bound / ts["divisor"])
    ts = alternate({"dense": lambda: dense.find_periods_with_weights(x, thresh=0.2),
                    "divisor": lambda: div.find_periods_with_weights(x, thresh=0.2)})
    row("config5 find_periods_with_weights(0.2)", n, b, 2, ml, "dense", ts["dense"])
    row("config5 find_periods_with_weights(0.2)", n, b, 2, ml, "divisor", ts["divisor"])
    del x

    # N = 16 384: dense global-memory path against the divisor form
    n, b = 16384, 64
    x = synth.synth_batch_device(b, n, 2, "cuda")
    ts = alternate({"dense": lambda: dense.find_periods(x), "divisor": lambda: div.find_periods(x)})
    for m in ("dense", "divisor"):
        row("N=16384", n, b, 2, n // 3, m, ts[m])

    # N = 131 072: divisor only
    n = 131072
    for b in (8, 1):
        x = synth.synth_batch_device(b, n, 3, "cuda")
        row("N=131072", n, b, 2, n // 3, "divisor", timed(lambda: div.find_periods(x)))

    # N = 2^20, B = 1: divisor only; the top 2 048 periods first
    n, b = 1 << 20, 1
    ml = n // 3
    x = synth.synth_batch_device(b, n, 4, "cuda")
    t_top = timed(lambda: div.find_periods(x, ml - 2047, ml))
    row("N=2^20 top 2048 periods", n, b, ml - 2047, ml, "divisor", t_top)
    projected = t_top * (ml - 1) / 2048
    if projected <= args.budget_s:
        row("N=2^20", n, b, 2, ml, "divisor", timed(lambda: div.find_periods(x)))
    else:
        print(json.dumps({"case": "N=2^20", "qmin": 2, "qmax": ml, "method": "divisor",
                          "s": "not measured (the top slice projects it over --budget-s)"}), flush=True)
    meta = {"card": card(), "smem_peak_TBps": smem_peak / 1e12, "rows": rows}
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(meta, fh, indent=1)


if __name__ == "__main__":
    main()
