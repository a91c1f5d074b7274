"""Throughput of the divisor-form fp64 Ramanujan periodogram (RamanujanPeriods(method="divisor"),
csrc/pp_ram_divisor.cu) against the dense fp64 path, CUDA events.

    python tools/perf_ram_divisor.py [--out FILE] [--budget-s 20]

Every batch is a seeded `synth` batch, device-resident.  Each timed call is preceded by a warm-up call of the same
shape; where both methods are timed they alternate in this process (dense, divisor, dense, divisor, ...).  Reported
per case: seconds per call, windows/s and, for the on-chip divisor kernel, the fold's share of the shared-memory bound
(every period reads the N staged samples once: B * Q * N * 8 bytes over the shared-memory peak pp_microbench measures
in this run).  Cases: config 5 (65 536 x 4 096, q = 2 .. 1 365, find_periods and find_periods_with_weights(thresh=0.2));
the shapes of ABOVE_THE_LIMIT, whose periodograms do not fit the fused on-chip kernel (both methods, ROUNDS alternating
rounds each with every round's time and the spread, after a check that the two methods' norms agree to AGREE; the
default method now runs the divisor form there as well, so both columns time the same kernel, and DESIGN.md 6.5 keeps
the numbers of the dense global-memory path that ran there before);
N = 131 072, B = 8 and 1; N = 2^20, B = 1 (divisor only).  At
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

ROUNDS = 4      # alternating rounds of the cases above the on-chip limit
AGREE = 2e-11   # norms of the two methods: each within 1e-11 of the exact value


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


def rounds(fns, n=ROUNDS):
    """Seconds per call of each of fns in each of n alternating rounds (one warm-up of each first)."""
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    for _ in range(n):
        for k, f in fns.items():
            out[k].append(_once(f))
    return out


def max_rel(a, b):
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    nz = b != 0
    return float(((a - b).abs()[nz] / b.abs()[nz]).max()) if bool(nz.any()) else float((a - b).abs().max())


# (label, N, B, qmin, qmax or None for N // 3, with weights): every case is above the fused kernel's limit (qmax 3 200)
ABOVE_THE_LIMIT = [
    ("just above the limit", 9603, 256, 2, 3201, False),
    ("full range, group form", 16384, 64, 2, None, False),
    ("full range, shift form", 16384, 1, 2, None, False),
    ("full range", 32768, 8, 2, None, False),
    ("full range", 65536, 1, 2, None, False),
    ("narrow band of large periods", 131072, 9, 43680, 43690, False),
    ("find_periods_with_weights(thresh=0.2)", 16384, 64, 2, None, True),
]


def above_the_limit(dense, div, row):
    """Each case: how far apart the two methods' norms are (reported with whether that is within AGREE), then ROUNDS
    alternating rounds; per method every round's time, their mean and the spread (slowest - fastest) / fastest."""
    for i, (label, n, b, qmin, qmax, weights) in enumerate(ABOVE_THE_LIMIT):
        qmax = qmax or n // 3
        x = synth.synth_batch_device(b, n, 10 + i, "cuda")
        if weights:
            got = {m: r.find_periods_with_weights(x, qmin, qmax, thresh=0.2) for m, r in
                   (("dense", dense), ("divisor", div))}
            err = max_rel(got["divisor"].norms, got["dense"].norms)
            if not torch.equal(torch.as_tensor(got["dense"].periods), torch.as_tensor(got["divisor"].periods)):
                err = float("inf")   # different periods selected
            fns = {m: (lambda r=r: r.find_periods_with_weights(x, qmin, qmax, thresh=0.2)) for m, r in
                   (("dense", dense), ("divisor", div))}
        else:
            err = max_rel(div.find_periods(x, qmin, qmax), dense.find_periods(x, qmin, qmax))
            fns = {m: (lambda r=r: r.find_periods(x, qmin, qmax)) for m, r in (("dense", dense), ("divisor", div))}
        ts = rounds(fns)
        for m in ("dense", "divisor"):
            row(f"N={n} {label}", n, b, qmin, qmax, m, sum(ts[m]) / len(ts[m]),
                extra={"rounds_s": ts[m], "spread": (max(ts[m]) - min(ts[m])) / min(ts[m]), "max_rel_diff": err,
                       "agree": err <= AGREE})
        del x


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

    def row(case, n, b, qmin, qmax, method, t, fold_share=None, extra=None):
        rows.append({"case": case, "N": n, "B": b, "qmin": qmin, "qmax": qmax, "method": method, "s": t,
                     "windows_per_s": b / t})
        if fold_share is not None:
            rows[-1]["fold_share_of_smem_bound"] = fold_share
        rows[-1].update(extra or {})
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

    # above the on-chip limit of the fused kernel: the default (dense) method against the divisor form, alternated
    above_the_limit(dense, div, row)

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
