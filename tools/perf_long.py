"""Throughput of the global-memory ("long") path of Periods: one ranking sweep per window, timed with CUDA events.

    python tools/perf_long.py [--max-candidates K] [--out FILE]

For each N the batch is device-resident and one `sweep(metric="norm")` (every candidate p in [2, max_length], one
warp per (window, p) over the whole GPU) is timed after a warm-up.  A sweep reads 8 * N bytes per candidate, almost
all of it from L2 (the residuals of a piece are sized to stay there), so bytes / time is the read rate the sweep
achieves.  max_length is the default N // 3, capped at --max-candidates (a default-length sweep at N = 2^20 reads
2.9 TB).  The last line compares the forced long path with the on-chip path at N = 12 288 (M-best, num = 5).
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyperiod_b200 import Periods, synth  # noqa: E402


def timed(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--max-candidates", type=int, default=8192)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    props = torch.cuda.get_device_properties(0)
    rows = []
    for n, b in ((16384, 256), (65536, 64), (262144, 16), (1048576, 4)):
        pmax = min(n // 3, args.max_candidates)
        x = synth.synth_batch_device(b, n, 1, "cuda")
        inst = Periods(staging="auto")
        t = timed(lambda: inst.sweep(x, metric="norm", max_length=pmax))
        nbytes = 8.0 * n * (pmax - 1) * b
        rows.append({"N": n, "B": b, "max_length": pmax, "s": t, "windows_per_s": b / t, "samples_per_s": b * n / t,
                     "sweep_read_GBps": nbytes / t / 1e9})
        print(json.dumps(rows[-1]), flush=True)
    x = synth.synth_batch_device(512, 12288, 2, "cuda")
    t_on = timed(lambda: Periods(staging="shared").m_best(x, num=5))
    t_lg = timed(lambda: Periods(staging="global").m_best(x, num=5))
    rows.append({"N": 12288, "B": 512, "call": "m_best(num=5)", "on_chip_windows_per_s": 512 / t_on,
                 "long_windows_per_s": 512 / t_lg})
    print(json.dumps(rows[-1]), flush=True)
    meta = {"gpu": props.name, "sm_count": props.multi_processor_count, "rows": rows}
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(meta, fh, indent=1)


if __name__ == "__main__":
    main()
