#!/usr/bin/env python
"""Benchmark of the north-star metric: windows/sec, M-best, N=4096, Pmax=1024, num=10 (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--windows B_PER_GPU]
                    [--secondary all|none|2,3g,4,5qo,5ram] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* is one pass of Periods.m_best(num=10, max_length=1024) over one batch of synthetic
hop-512 windows cut from a multi-tone stream (SURVEY.md 8d, config 3).  Each GPU owns its own
stream shard (windows are independent: no data-path collective; weak scaling, and at N=8 the job is
exactly config 3's 1,048,576 windows).  Rank 0 prints ONE JSON line.

  value     device-resident: the stream is already in HBM, results stay in HBM; CUDA events, max over ranks
  e2e       through the public API with PINNED HOST buffers: H2D of the stream + kernel + D2H of
            periods/powers/status inside the timed region; median of --e2e-steps steps
  roofline  the M-best kernel against the shared-memory roofline it is bound by (8 B of on-chip operand
            per accumulate-add; SURVEY.md 8d), denominators measured live by pp_microbench; the FP64-pipe
            and HBM views of the same launch ride along
  cpu_baseline  the oracle (numpy port of the reference) on the box's host cores, bounded sample, rank 0, N=1
  secondary the other BASELINE.json configs at their FULL batch sizes (2: 16,384 x 2048 small_to_large;
            3g: m_best_gamma on the headline stream; 4: 262,144 x 8192 Muresan-Parks best_correlation;
            5qo / 5ram: 65,536 x 4096 QOPeriods.find_periods and RamanujanPeriods.find_periods_with_weights),
            sharded over the N GPUs (strong scaling: the batch size is the config's), each entry with its own
            value / e2e / roofline / cpu_baseline / in-run parity sample.  The headline keys are unchanged.
  --impl reference   the same oracle port timed as the reference arm (the reference itself is pure Python,
            does not import at HEAD and cannot travel to the GPU box; see DESIGN.md)
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import sys
import threading
import time

os.environ.setdefault("OMP_NUM_THREADS", "1")
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
os.environ.setdefault("MKL_NUM_THREADS", "1")

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_WIN, HOP, PMAX, NUM = 4096, 512, 1024, 10
METRIC = "windows/sec, M-best N=4096 Pmax=1024 num=10"
UNIT = "windows/s"


# ----------------------------------------------------------------------------- CPU side (oracle workers, one window each)
def _oracle_window(x):
    from oracle import periods as op
    st = {}
    per, pw, _ = op.m_best(x, NUM, PMAX, stats=st)
    return per, pw, st["sweeps"]


def _oracle_gamma(x):
    from oracle import periods as op
    st = {}
    per, pw, _ = op.m_best_gamma(x, NUM, PMAX, stats=st)
    return per, pw, st["sweeps"]


def _oracle_s2l(x):
    from oracle import periods as op
    per, pw, _ = op.small_to_large(x, 0.1)
    return np.asarray(per, dtype=np.int64), np.asarray(pw, dtype=np.float64)


def _oracle_bcorr(x):
    from oracle import periods as op
    per, pw, _ = op.best_correlation(x, num=10, trunc=True, orth=True)
    return per, pw


def _oracle_qo(x):
    from oracle import qo as oq
    with contextlib.redirect_stdout(io.StringIO()):   # the reference prints the period list every round (:488)
        d, res = oq.find_periods(x, num=4, thresh=0.05)
    return (np.asarray(d["periods"], dtype=np.int64), list(d["basis_dictionary"].items()),
            np.asarray(d["weights"], dtype=np.float64), np.asarray(res))


def _oracle_ram(x):
    """Config 5 Ramanujan leg for the parity sample: fp64 closed form of the periodogram (the literal reference
    takes ~20 min per window at q <= 1365), then the reference's own select / get_subspaces / solve_quadratic."""
    from oracle import ramanujan as orr
    norms = orr.norms_closed_form_f64(x)
    try:
        d, res = orr.find_periods_with_weights(x, thresh=0.2, norms=norms)
        return norms, np.asarray(d["periods"], dtype=np.int64), np.asarray(d["weights"]), np.asarray(res), None
    except np.linalg.LinAlgError as e:
        per = np.argwhere(norms / np.abs(np.max(norms)) > 0.2).flatten()
        return norms, per, None, None, repr(e)


def _oracle_ram_literal(args):
    from oracle import ramanujan as orr
    x, q = args
    return float(orr.find_periods(x, 2, q)[q])      # literal restatement of RamanujanPeriods.find_periods


def _noop(_):
    return 0


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        return os.cpu_count() or 1


class OraclePool:
    """One spawn pool for every CPU leg of the run (one process per core, one BLAS thread each)."""

    def __init__(self, cores: int):
        import multiprocessing as mp
        self.cores = cores
        self.pool = mp.get_context("spawn").Pool(cores)
        self.pool.map(_oracle_window, [np.sin(np.arange(N_WIN) * 0.1 * (i + 1)) for i in range(cores)][:cores])  # spin up

    def run(self, windows, fn=_oracle_window):
        t0 = time.perf_counter()
        out = self.pool.map(fn, windows, chunksize=1)
        return out, time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()


def sample_windows(stream: np.ndarray, count: int):
    return [np.array(stream[HOP * b: HOP * b + N_WIN]) for b in range(count)]


# under 64 MB in all with the .npy headers
DUMP_BYTES = 60_000_000


def dump_outputs(out_dir: str, arrays: dict):
    """Write each per-window result array (first axis = window) as out_dir/<name>.npy in float64, which holds the int32
    periods and counts exactly.  When the arrays would exceed DUMP_BYTES together, every array keeps the same fixed,
    seeded sample of windows, and their indices are written as rows.npy."""
    import torch
    arrays = {k: v.view(torch.int32) if v.dtype == getattr(torch, "uint32", None) else v for k, v in arrays.items()}
    b = next(iter(arrays.values())).shape[0]
    row_bytes = 8 * sum(v[0].numel() for v in arrays.values())
    rows = None
    if b * row_bytes > DUMP_BYTES:
        keep = DUMP_BYTES // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(0).choice(b, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        if rows is not None:
            v = v[torch.from_numpy(rows).to(v.device)]
        np.save(os.path.join(out_dir, name + ".npy"), v.cpu().numpy().astype(np.float64))
    if rows is not None:
        np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU every 100 ms while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- reference arm
def run_reference(args, rank: int):
    if rank != 0:
        return
    from pyperiod_b200 import synth
    cores = host_cores()
    per_step = 16 * cores
    stream = synth.synth_stream(per_step, N_WIN, HOP, 30_000)
    wins = sample_windows(stream, per_step)
    pool = OraclePool(cores)
    for _ in range(args.warmup):
        pool.run(wins)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pool.run(wins)
    dt = time.perf_counter() - t0
    pool.close()
    val = per_step * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(per_step, 1, "host"),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{per_step} windows per step (16 per core), oracle numpy port of Periods.m_best, "
                                   f"one process per core"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(b_per_gpu: int, n_gpus: int, where: str):
    return {"workload": f"config 3: Periods.m_best(num={NUM}, max_length={PMAX}) on hop-{HOP} windows of N={N_WIN} "
                        f"cut from a synthetic multi-tone stream (3 tones + noise per 65,536-sample segment)",
            "windows_per_gpu_per_step": b_per_gpu, "windows_per_step": b_per_gpu * n_gpus, "N": N_WIN, "hop": HOP,
            "Pmax": PMAX, "num": NUM, "sharding": f"{n_gpus} independent stream shards, no data-path collective; compact results "
                        f"gathered to rank 0 each step" if n_gpus > 1 else "single GPU",
            "l2": "input stream per step (>= 0.5 GB) is larger than the 126 MB L2", "inputs": where}


# ----------------------------------------------------------------------------- secondary configs (BASELINE.json configs 2, 3-gamma, 4, 5)
class Ctx:
    """What every secondary config needs from the run: device, ranks, the CPU pool, measured peaks."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, values):
        import torch
        t = torch.tensor(list(values), dtype=torch.float64, device=self.dev)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def sum_over_ranks(self, values):
        import torch
        t = torch.tensor(list(values), dtype=torch.float64, device=self.dev)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t]


def timed_steps(ctx: Ctx, fn, steps: int, warm):
    """`warm` untimed calls (callables), then `steps` timed calls of fn between barriers; per-step CUDA-event times
    on the launching stream, max over ranks per step.  Returns (ms list, last result)."""
    import torch
    for w in warm:
        w()
    ctx.barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    out = None
    for e0, e1 in evs:
        e0.record()
        out = fn()
        e1.record()
    ctx.barrier()
    return ctx.max_over_ranks(e0.elapsed_time(e1) for e0, e1 in evs), out


def host_copy_for_e2e(x_dev, limit_bytes: int):
    """Pinned host copy of (a prefix of) a device batch for the end-to-end leg; the prefix is bounded by
    `limit_bytes` so a 17 GB batch does not need 17 GB of page-locked host memory."""
    import torch
    b = x_dev.shape[0]
    rows = max(1, min(b, limit_bytes // (x_dev.shape[1] * 8)))
    h = torch.empty((rows, x_dev.shape[1]), dtype=torch.float64, pin_memory=True)
    h.copy_(x_dev[:rows])
    torch.cuda.synchronize()
    return h


def nbytes_of(*arrays) -> int:
    return int(sum(a.nbytes for a in arrays if a is not None))


def rel_err(got, want):
    want = np.asarray(want, dtype=np.float64)
    got = np.asarray(got, dtype=np.float64)
    den = np.maximum(np.abs(want), 1e-300)
    return float(np.max(np.abs(got - want) / den)) if want.size else 0.0


def secondary_entry(ctx: Ctx, key, workload, n, b_total, ms, ms_e2e, e2e_windows, h2d, d2h, steps_note, launches):
    med = float(np.median(ms))
    med_e = float(np.median(ms_e2e))
    return {"config": key, "workload": workload, "metric": "windows/sec", "unit": UNIT, "N": n,
            "windows_per_step": b_total, "n_gpus": ctx.world, "scaling": "strong",
            "value": b_total / (sum(ms) * 1e-3 / len(ms)), "ms_per_step": sum(ms) / len(ms), "ms_per_step_median": med,
            "steps": len(ms), "warmup": steps_note, "gpu_launches_per_step": launches, "data": "synthetic (generated on the device; "
            "3 tones + noise per window, peak-normalised)", "l2": "input batch larger than the 126 MB L2",
            "e2e": {"value": e2e_windows * ctx.world / (med_e * 1e-3), "unit": UNIT, "windows_per_step": e2e_windows * ctx.world,
                    "steps": len(ms_e2e), "ms_per_step_median": med_e, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}}


def sample_rows(b: int, count: int):
    count = min(b, count)
    return np.unique(np.linspace(0, b - 1, count).astype(np.int64))


def gather(ctx: Ctx, periods, powers, status, total):
    if ctx.world > 1:
        from pyperiod_b200 import sharding
        sharding.gather_compact(periods, powers, status, total, dst=0)


def shard(ctx: Ctx, total: int):
    from pyperiod_b200 import sharding
    lo, hi = sharding.shard_bounds(total, ctx.world, ctx.rank)
    return hi - lo


def sec_s2l(ctx: Ctx):
    """config 2: Periods.small_to_large(thresh=0.1), 16,384 windows of N=2048."""
    import torch
    from pyperiod_b200 import Periods, synth
    n, total = 2048, 16_384
    b = shard(ctx, total)
    x = synth.synth_batch_device(b, n, 20_000 + ctx.rank, ctx.dev)
    algo = Periods(device=ctx.dev)

    def step():
        r = algo.small_to_large(x, thresh=0.1)
        gather(ctx, r.periods, r.powers, r.count, total)
        return r
    ms, r = timed_steps(ctx, step, 10, [step] * 3)
    xh = host_copy_for_e2e(x, ctx.pin_limit)
    ms_e, r2 = timed_steps(ctx, lambda: algo.small_to_large(xh, thresh=0.1), 5, [lambda: algo.small_to_large(xh, thresh=0.1)])
    e = secondary_entry(ctx, "2", "config 2: Periods.small_to_large(thresh=0.1) on 16,384 windows of N=2048", n, total,
                        ms, ms_e, xh.shape[0], xh.numel() * 8, nbytes_of(r2.periods, r2.powers, r2.count, r2.status),
                        3, 1)
    canon = 1023 * n * 8.0
    sec = e["ms_per_step"] * 1e-3
    e["mean_periods"] = ctx.sum_over_ranks([float(r.count.sum())])[0] / total
    e["status_nonzero_windows"] = int(ctx.sum_over_ranks([float((r.status != 0).sum())])[0])
    e["roofline"] = {"kernel": "pp::s2l_kernel", "bound": "smem", "achieved": total * canon / sec / 1e9 / ctx.world,
                     "peak": ctx.smem_peak / 1e9, "unit": "GB/s", "frac": total * canon / sec / ctx.smem_peak / ctx.world,
                     "traffic": None,
                     "algorithmic": "ONE canonical pass of 1023 periods x 2048 adds x 8 B of shared-memory operand per "
                                    "window (per GPU); the kernel executes a partial first-hit sweep per accepted period"}
    if ctx.pool is not None:
        rows = sample_rows(b, 16 * ctx.cores)
        wins = [np.array(v) for v in x[torch.from_numpy(rows).to(ctx.dev)].cpu().numpy()]
        want, dt = ctx.pool.run(wins, _oracle_s2l)
        per, pw, cnt = r.periods.cpu().numpy(), r.powers.cpu().numpy(), r.count.cpu().numpy()
        same = sum(int(np.array_equal(per[i, :cnt[i]].astype(np.int64), want[k][0])) for k, i in enumerate(rows))
        err = max([rel_err(pw[i, :cnt[i]], want[k][1]) for k, i in enumerate(rows)
                   if np.array_equal(per[i, :cnt[i]].astype(np.int64), want[k][0])] + [0.0])
        e["parity"] = {"windows": len(rows), "period_lists_equal": same, "max_rel_power_err": err}
        e["cpu_baseline"] = {"value": len(rows) / dt, "unit": UNIT, "cores": ctx.cores, "kind": "port",
                             "sample": f"{len(rows)} windows of the GPU batch (16 per core), oracle small_to_large, {dt:.1f} s wall"}
    return e


def sec_gamma(ctx: Ctx):
    """config 3, second call: Periods.m_best_gamma(num=10, max_length=1024) on the headline's own stream."""
    import torch
    from pyperiod_b200 import Periods, _lib
    b = ctx.dev_windows.shape[0]
    total = b * ctx.world
    algo = Periods(device=ctx.dev)

    def step():
        r = algo.m_best_gamma(ctx.dev_windows, num=NUM, max_length=PMAX)
        gather(ctx, r.periods, r.powers, r.status, total)
        return r
    ms, r = timed_steps(ctx, step, 3, [step] * 3)
    fe = lambda: algo.m_best_gamma(ctx.host_windows, num=NUM, max_length=PMAX)
    ms_e, r2 = timed_steps(ctx, fe, 3, [fe])
    e = secondary_entry(ctx, "3g", f"config 3 (gamma): Periods.m_best_gamma(num={NUM}, max_length={PMAX}) on the headline's "
                        f"hop-{HOP} stream windows of N={N_WIN}", N_WIN, total, ms, ms_e, b, ctx.stream_bytes,
                        nbytes_of(r2.periods, r2.powers, r2.status, r2.sweeps), 3, 2)
    e["scaling"] = "weak"
    sweeps = ctx.sum_over_ranks([float(r.sweeps.sum())])[0]
    sec = e["ms_per_step"] * 1e-3
    canon = sweeps / ctx.world * (PMAX - 1) * N_WIN * 8.0
    passes = _lib.sweep_passes(N_WIN, 2, PMAX)
    e["sweeps_per_window"] = sweeps / total
    e["status_nonzero_windows"] = int(ctx.sum_over_ranks([float((r.status != 0).sum())])[0])
    e["roofline"] = {"kernel": "pp::mbest_kernel (gamma)", "bound": "smem", "achieved": canon / sec / 1e9,
                     "peak": ctx.smem_peak / 1e9, "unit": "GB/s", "frac": canon / sec / ctx.smem_peak, "traffic": None,
                     "algorithmic": "sweeps_executed x 1023 periods x 4096 adds x 8 B per launch (canonical), per GPU",
                     "executed_frac": canon / sec / ctx.smem_peak * passes / (PMAX - 1)}
    if ctx.pool is not None:
        n_s = 8 * ctx.cores
        want, dt = ctx.pool.run(sample_windows(ctx.stream, n_s), _oracle_gamma)
        same = sum(int(np.array_equal(r2.periods[i], want[i][0])) for i in range(n_s))
        err = max([rel_err(r2.powers[i], want[i][1]) for i in range(n_s) if np.array_equal(r2.periods[i], want[i][0])] + [0.0])
        e["parity"] = {"windows": n_s, "period_lists_equal": same, "max_rel_power_err": err,
                       "sweep_counts_equal": sum(int(r2.sweeps[i] == want[i][2]) for i in range(n_s))}
        e["cpu_baseline"] = {"value": n_s / dt, "unit": UNIT, "cores": ctx.cores, "kind": "port",
                             "sample": f"first {n_s} windows of the stream (8 per core), oracle m_best_gamma, {dt:.1f} s wall"}
    return e


def sec_bcorr(ctx: Ctx):
    """config 4: Periods(trunc=True, orth=True).best_correlation(num=10), 262,144 windows of N=8192."""
    import torch
    from pyperiod_b200 import Periods, _lib
    from pyperiod_b200 import synth
    n, total = 8192, 262_144
    b = shard(ctx, total)
    x = synth.synth_batch_device(b, n, 40_000 + ctx.rank, ctx.dev)
    algo = Periods(True, True, device=ctx.dev)
    small = x[: max(1024, b // 32)]

    def step():
        r = algo.best_correlation(x, num=10)
        gather(ctx, r.periods, r.powers, r.status, total)
        return r
    warm = lambda: algo.best_correlation(small, num=10)
    ms, r = timed_steps(ctx, step, 2, [warm] * 3)
    xh = host_copy_for_e2e(x, ctx.pin_limit)
    fe = lambda: algo.best_correlation(xh, num=10)
    ms_e, r2 = timed_steps(ctx, fe, 2 if xh.shape[0] < b else 1, [lambda: algo.best_correlation(xh[:1024], num=10)])
    e = secondary_entry(ctx, "4", "config 4: Periods(trunc_to_integer_multiple=True, orthogonalize=True)"
                        ".best_correlation(num=10) on 262,144 windows of N=8192 (candidates 2..2729)", n, total, ms, ms_e,
                        xh.shape[0], xh.numel() * 8, nbytes_of(r2.periods, r2.powers, r2.status),
                        "3 calls on a 1/32 slice of the batch (same kernels and shapes per window)", 2)
    sec = e["ms_per_step"] * 1e-3
    canon = 10 * 2728 * n * 8.0 * total / ctx.world
    passes = _lib.sweep_passes(n, 2, 2729)
    e["status_nonzero_windows"] = int(ctx.sum_over_ranks([float((r.status != 0).sum())])[0])
    e["roofline"] = {"kernel": "pp::bcorr_kernel", "bound": "smem", "achieved": canon / sec / 1e9, "peak": ctx.smem_peak / 1e9,
                     "unit": "GB/s", "frac": canon / sec / ctx.smem_peak, "traffic": None,
                     "algorithmic": "10 rounds x 2728 periods x 8192 sequential adds x 8 B per window (canonical), per GPU; "
                                    f"executed: hierarchical nomination ({passes} passes per round) + exact sequential "
                                    "folds of the near-maximal candidates",
                     "executed_frac": canon / sec / ctx.smem_peak * passes / 2728}
    if ctx.pool is not None:
        rows = sample_rows(b, 4 * ctx.cores)
        wins = [np.array(v) for v in x[torch.from_numpy(rows).to(ctx.dev)].cpu().numpy()]
        want, dt = ctx.pool.run(wins, _oracle_bcorr)
        per, pw = r.periods.cpu().numpy(), r.powers.cpu().numpy()
        same = sum(int(np.array_equal(per[i].astype(np.int64), np.asarray(want[k][0], dtype=np.int64))) for k, i in enumerate(rows))
        err = max([float(np.max(np.abs(pw[i] - want[k][1]))) for k, i in enumerate(rows)] + [0.0])
        e["parity"] = {"windows": len(rows), "period_lists_equal": same, "max_abs_power_err": err}
        e["cpu_baseline"] = {"value": len(rows) / dt, "unit": UNIT, "cores": ctx.cores, "kind": "port",
                             "sample": f"{len(rows)} windows of the GPU batch (4 per core), oracle best_correlation(num=10, "
                                       f"trunc, orth), {dt:.1f} s wall"}
    return e


def sec_qo(ctx: Ctx):
    """config 5, first call: QOPeriods().find_periods(num=4, thresh=0.05), 65,536 windows of N=4096."""
    import torch
    from pyperiod_b200 import QOPeriods, synth
    n, total = 4096, 65_536
    b = shard(ctx, total)
    x = synth.synth_batch_device(b, n, 50_000 + ctx.rank, ctx.dev)
    algo = QOPeriods(device=ctx.dev)
    small = x[: max(1024, b // 16)]

    def step():
        r = algo.find_periods(x, num=4, thresh=0.05)
        gather(ctx, r.periods, r.norms, r.status, total)
        return r
    warm = lambda: algo.find_periods(small, num=4, thresh=0.05)
    ms, r = timed_steps(ctx, step, 3, [warm] * 3)
    xh = host_copy_for_e2e(x, ctx.pin_limit)
    fe = lambda: algo.find_periods(xh, num=4, thresh=0.05)
    ms_e, r2 = timed_steps(ctx, fe, 3, [lambda: algo.find_periods(xh[:2048], num=4, thresh=0.05)])
    e = secondary_entry(ctx, "5qo", "config 5: QOPeriods().find_periods(num=4, thresh=0.05) on 65,536 windows of N=4096 "
                        "(candidates 2..1365; dict + residual returned)", n, total, ms, ms_e, xh.shape[0], xh.numel() * 8,
                        nbytes_of(r2.periods, r2.norms, r2.n_periods, r2.dict_q, r2.dict_keep, r2.n_dict, r2.weights,
                                  r2.n_weights, r2.res, r2.status),
                        "3 calls on a 1/16 slice of the batch", "1 (+1 for windows whose dictionary outgrows 1024 rows)")
    sec = e["ms_per_step"] * 1e-3
    rows_f = r.n_weights.double()
    rounds = ctx.sum_over_ranks([float(r.n_dict.sum())])[0]
    chol = ctx.sum_over_ranks([float((rows_f ** 3 / 3.0).sum())])[0]
    canon = rounds / ctx.world * 1364 * n * 8.0
    st = r.status
    e["mean_rows"] = ctx.sum_over_ranks([float(rows_f.sum())])[0] / total
    e["rounds_per_window"] = rounds / total
    e["status_histogram"] = {str(k): int(ctx.sum_over_ranks([float((st == k).sum())])[0]) for k in range(7)}
    e["roofline"] = {"kernel": "pp::qo_find_kernel", "bound": "smem", "achieved": canon / sec / 1e9, "peak": ctx.smem_peak / 1e9,
                     "unit": "GB/s", "frac": canon / sec / ctx.smem_peak, "traffic": None,
                     "algorithmic": "gamma sweeps: rounds x 1364 periods x 4096 adds x 8 B (canonical) per GPU; the same "
                                    "kernel also factors the normal equations on the FP64 tensor cores",
                     "tensor": {"bound": "tensor", "achieved": chol / ctx.world / sec / 1e12, "peak": ctx.dmma_peak / 1e12,
                                "unit": "TFLOP/s", "frac": chol / ctx.world / sec / ctx.dmma_peak,
                                "algorithmic": "R^3/3 flop of each window's final dictionary (the factor is extended "
                                               "round by round, never recomputed), against the measured DMMA peak"}}
    if ctx.pool is not None:
        rows = sample_rows(xh.shape[0], 4 * ctx.cores)   # windows of the end-to-end call: its results are on the host
        wins = [np.array(v) for v in xh[torch.from_numpy(rows)].numpy()]
        want, dt = ctx.pool.run(wins, _oracle_qo)
        same = dsame = 0
        werr, rerr = [], []
        for k, i in enumerate(rows):
            d, res = r2.window(int(i))
            ok = np.array_equal(np.asarray(d["periods"], dtype=np.int64), want[k][0])
            same += int(ok)
            dok = [(str(a), int(c)) for a, c in d["basis_dictionary"].items()] == [(str(a), int(c)) for a, c in want[k][1]]
            dsame += int(dok)
            if ok and dok:
                werr.append(float(np.max(np.abs(d["weights"] - want[k][2])) / max(np.max(np.abs(want[k][2])), 1e-300)))
                rerr.append(float(np.max(np.abs(res - want[k][3]))))
        e["parity"] = {"windows": len(rows), "period_lists_equal": same, "dictionaries_equal": dsame,
                       "max_weight_err_rel_to_largest": max(werr + [0.0]), "max_abs_residual_err": max(rerr + [0.0])}
        e["cpu_baseline"] = {"value": len(rows) / dt, "unit": UNIT, "cores": ctx.cores, "kind": "port",
                             "sample": f"{len(rows)} windows of the GPU batch (4 per core), oracle QO find_periods, {dt:.1f} s wall"}
    return e


def sec_ram(ctx: Ctx):
    """config 5, second call: RamanujanPeriods().find_periods_with_weights(thresh=0.2), 65,536 windows of N=4096."""
    import torch
    from pyperiod_b200 import RamanujanPeriods, synth
    n, total, qmax = 4096, 65_536, 1365
    b = shard(ctx, total)
    x = synth.synth_batch_device(b, n, 50_000 + ctx.rank, ctx.dev)   # the same batch as the QO call
    algo = RamanujanPeriods(device=ctx.dev)
    small = x[: max(1024, b // 32)]

    def pad(t, k=64):
        if t.dtype not in (torch.int32, torch.float64):
            t = t.view(torch.int32)
        out = torch.zeros((t.shape[0], k), dtype=t.dtype, device=t.device)
        out[:, : min(k, t.shape[1])] = t[:, :k]
        return out

    def step():
        r = algo.find_periods_with_weights(x, thresh=0.2)
        gather(ctx, pad(r.periods), pad(r.norms), r.status, total)
        return r
    warm = lambda: algo.find_periods_with_weights(small, thresh=0.2)
    ms, r = timed_steps(ctx, step, 2, [warm] * 3)
    ms_n, nrm = timed_steps(ctx, lambda: algo.find_periods(x), 2, [])
    xh = host_copy_for_e2e(x, min(ctx.pin_limit, 16_384 * n * 8))
    fe = lambda: algo.find_periods_with_weights(xh, thresh=0.2)
    ms_e, r2 = timed_steps(ctx, fe, 1, [lambda: algo.find_periods_with_weights(xh[:1024], thresh=0.2)])
    e = secondary_entry(ctx, "5ram", "config 5: RamanujanPeriods().find_periods_with_weights(thresh=0.2) on 65,536 windows "
                        "of N=4096 (periodogram q = 2..1365 on the FP64 tensor cores, then the quadratic program)", n,
                        total, ms, ms_e, xh.shape[0], xh.numel() * 8,
                        nbytes_of(r2.periods, r2.norms, r2.n_periods, r2.dict_q, r2.dict_keep, r2.n_dict, r2.weights,
                                  r2.n_weights, r2.res, r2.status),
                        "3 calls on a 1/32 slice of the batch", "periodogram 2 (dictionary table + fused fold/DMMA kernel for the whole batch); select 1; row count 1; solve 1-2")
    sec_n = sum(ms_n) / len(ms_n) * 1e-3
    flops = 2.0 * sum(q * q for q in range(2, qmax + 1)) * total / ctx.world
    st = r.status
    e["periodogram_only"] = {"value": total / sec_n, "unit": UNIT, "ms_per_step": sec_n * 1e3}
    e["mean_rows"] = ctx.sum_over_ranks([float(r.n_weights.double().sum())])[0] / total
    e["status_histogram"] = {str(k): int(ctx.sum_over_ranks([float((st == k).sum())])[0]) for k in range(7)}
    e["roofline"] = {"kernel": "pp::ram_gemm_kernel", "bound": "tensor", "achieved": flops / sec_n / 1e12,
                     "peak": ctx.dmma_peak / 1e12, "unit": "TFLOP/s", "frac": flops / sec_n / ctx.dmma_peak, "traffic": None,
                     "algorithmic": "2 q^2 flop per period and window (circulant product on the fold sums), q = 2..1365, "
                                    "over the periodogram launches alone; peak = measured DMMA m8n8k4 rate "
                                    "(pp_microbench kind 2); MEASURED_PEAKS.json has no FP64 tensor figure"}
    if ctx.pool is not None:
        rows = sample_rows(b, ctx.cores)
        wins = [np.array(v) for v in x[torch.from_numpy(rows).to(ctx.dev)].cpu().numpy()]
        want, dt = ctx.pool.run(wins, _oracle_ram)
        nh = nrm[torch.from_numpy(rows).to(ctx.dev)].cpu().numpy()
        nerr = max(rel_err(nh[k, 2:], want[k][0][2:]) for k in range(len(rows)))
        same, rerr, lin = 0, [], 0
        for k, i in enumerate(rows):
            per = r.periods[int(i), : int(r.n_periods[int(i)])].cpu().numpy().astype(np.int64)
            same += int(np.array_equal(per, want[k][1]))
            if want[k][4] is not None:
                lin += 1
                continue
            if int(r.status[int(i)]) == 0:
                rerr.append(float(np.max(np.abs(r.res[int(i)].cpu().numpy() - want[k][3]))))
        e["parity"] = {"windows": len(rows), "max_rel_norm_err_vs_fp64_closed_form": nerr, "period_lists_equal": same,
                       "oracle_linalg_errors": lin, "max_abs_residual_diff_vs_oracle_lu": max(rerr + [0.0]),
                       "note": "residuals are compared with the oracle's LU solve, itself only good to ~1e-6 on the "
                               "ill-conditioned dictionaries (cond up to 1e14); tests/test_gpu_ramanujan.py compares both "
                               "with an extended-precision solution"}
        # the literal reference algorithm is O(Q^3.15): ~20 min per window at Q = 1365; time Q = 128 and 256, extrapolate
        _, t128 = ctx.pool.run([(wins[i % len(wins)], 128) for i in range(ctx.cores)], _oracle_ram_literal)
        _, t256 = ctx.pool.run([(wins[i % len(wins)], 256) for i in range(ctx.cores)], _oracle_ram_literal)
        expo = float(np.log(t256 / t128) / np.log(2.0))
        t1365 = t256 * (qmax / 256) ** expo
        e["cpu_baseline"] = {"value": ctx.cores / t1365, "unit": UNIT, "cores": ctx.cores, "kind": "port",
                             "sample": f"EXTRAPOLATED periodogram only: literal oracle at Q=128 ({t128:.1f} s) and Q=256 "
                                       f"({t256:.1f} s), one window per core, measured exponent {expo:.2f}, scaled to "
                                       f"Q=1365; parity sample used the fp64 closed form ({dt:.1f} s for {len(rows)} windows)"}
    return e


SECONDARY = {"2": sec_s2l, "3g": sec_gamma, "4": sec_bcorr, "5qo": sec_qo, "5ram": sec_ram}


def run_secondary(ctx: Ctx, which):
    import torch
    out = []
    for key in which:
        t0 = time.perf_counter()
        try:
            entry = SECONDARY[key](ctx)
        except Exception as exc:  # a failing secondary config never takes the headline line down
            import traceback
            traceback.print_exc(file=sys.stderr)
            entry = {"config": key, "error": repr(exc)}
        entry["bench_wall_s"] = time.perf_counter() - t0
        out.append(entry)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------- B200 arm
def run_b200(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist
    from pyperiod_b200 import Periods, _lib, sharding, synth

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's banner / logs never go to stdout
        dist.init_process_group("nccl", device_id=dev)
    B = args.windows
    assert B % 128 == 0, "--windows must be a multiple of 128 (segment alignment)"

    cpu = None
    oracle_out = None
    pool = None
    cores = host_cores()
    first_seg = rank * (B * HOP // 65_536)
    stream = synth.synth_stream(B, N_WIN, HOP, 30_000, first_segment=first_seg)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        pool = OraclePool(cores)   # workers start before the CUDA context exists; the sample itself runs after the
                                   # GPU measurements, so the host load stays away from the timed GPU steps

    # ---- measured roofline denominators (outside any timed region)
    smem_peak = _lib.microbench(0)
    dadd_peak = _lib.microbench(1)
    dmma_peak = _lib.microbench(2)

    host_stream = torch.from_numpy(stream).pin_memory()
    dev_stream = host_stream.to(dev)
    dev_windows = torch.as_strided(dev_stream, (B, N_WIN), (HOP, 1))
    host_windows = torch.as_strided(host_stream, (B, N_WIN), (HOP, 1))
    algo = Periods(device=dev)

    def step_device():
        r = algo.m_best(dev_windows, num=NUM, max_length=PMAX)
        if world > 1:  # the only collective: compact periods/powers/status to rank 0 (NCCL over NVLink)
            sharding.gather_compact(r.periods, r.powers, r.status, B * world, dst=0)
        return r

    def step_e2e():
        return algo.m_best(host_windows, num=NUM, max_length=PMAX)   # H2D + kernel + D2H to numpy

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        res = step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        res = step_device()
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    sampler.stop_flag = True
    sampler.join()
    sweeps = int(res.sweeps.sum().item())
    status_bad = int((res.status != 0).sum().item())
    near_tie_windows = int((res.near_ties != 0).sum().item())
    if args.dump_outputs and rank == 0:   # the last timed step's results (rank 0's windows when several GPUs run)
        dump_outputs(args.dump_outputs, {"periods": res.periods, "powers": res.powers, "status": res.status,
                                         "sweeps": res.sweeps, "near_ties": res.near_ties})

    # ---- end-to-end through the public API with pinned host buffers: every step timed on its own, median reported
    e2e_steps = max(1, args.e2e_steps)
    step_e2e()
    barrier()
    e2e_ms = []
    for _ in range(e2e_steps):
        ev0.record()
        r2 = step_e2e()
        ev1.record()
        barrier()
        e2e_ms.append(ev0.elapsed_time(ev1))
    h2d = stream.nbytes
    d2h = int(r2.periods.nbytes + r2.powers.nbytes + r2.status.nbytes + r2.sweeps.nbytes + r2.near_ties.nbytes)

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload, after the GPU measurements
    if pool is not None:
        n_s = 64 * cores   # ~10-20 s of CPU work at ~0.16 s per window per core
        oracle_out, dt = pool.run(sample_windows(stream, n_s))
        cpu = {"value": n_s / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"first {n_s} windows of the GPU run's own stream (64 per core), oracle numpy port of "
                         f"Periods.m_best, one process per core, {dt:.1f} s wall"}

    # ---- parity on the sampled windows (period lists must be identical)
    parity = None
    if oracle_out is not None:
        got_p = r2.periods[: len(oracle_out)]
        got_w = r2.powers[: len(oracle_out)]
        same = sum(int(np.array_equal(got_p[i], oracle_out[i][0])) for i in range(len(oracle_out)))
        rel = max(float(np.max(np.abs(got_w[i] - oracle_out[i][1]) / np.abs(oracle_out[i][1])))
                  for i in range(len(oracle_out)))
        sw_same = sum(int(r2.sweeps[i] == oracle_out[i][2]) for i in range(len(oracle_out)))
        parity = {"windows": len(oracle_out), "period_lists_equal": same, "sweep_counts_equal": sw_same,
                  "max_rel_power_err": rel}

    # ---- max over ranks
    t = torch.tensor([ms_total] + e2e_ms, dtype=torch.float64, device=dev)
    cnt = torch.tensor([float(sweeps), float(status_bad), float(near_tie_windows)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    ms_total = float(t[0])
    e2e_ms = [float(v) for v in t[1:]]
    ms_e2e = float(np.median(e2e_ms))
    sweeps_all = float(cnt[0])

    # ---- the other BASELINE configs at full size (extra keys; the headline is complete at this point)
    which = [] if args.secondary == "none" else (list(SECONDARY) if args.secondary == "all" else args.secondary.split(","))
    secondary = None
    if which:
        free_host = 64 << 30
        try:
            import psutil
            free_host = int(psutil.virtual_memory().available)
        except Exception:
            pass
        ctx = Ctx(dev=dev, rank=rank, world=world, pool=pool, cores=cores, smem_peak=smem_peak["per_s"],
                  dadd_peak=dadd_peak["per_s"], dmma_peak=dmma_peak["per_s"], dev_windows=dev_windows,
                  host_windows=host_windows, stream=stream, stream_bytes=stream.nbytes,
                  pin_limit=int(min(20 << 30, free_host // (4 * max(1, world)))))
        secondary = run_secondary(ctx, which)
    if pool is not None:
        pool.close()

    if rank == 0:
        secs = ms_total * 1e-3
        value = B * world * args.steps / secs
        e2e_val = B * world / (ms_e2e * 1e-3)
        # algorithmic work of ONE launch on ONE GPU (SURVEY.md 8d): sweeps executed (counted on device)
        # x (Pmax-1) candidate periods x N accumulate-adds, 8 B of shared-memory operand each.
        # The hierarchical ranking sweep EXECUTES only one pass per top period in (Pmax/2, Pmax] (the rest
        # follow from S_2p), minus the tops that ride on another top's pass, so its executed traffic is
        # passes/(Pmax-1) of the canonical figure; both are reported so the algorithmic saving is visible
        # rather than hidden.
        adds_per_launch = (sweeps_all / world) * (PMAX - 1) * N_WIN
        passes = _lib.sweep_passes(N_WIN, 2, PMAX)   # window passes per sweep actually executed (tops minus riders)
        exec_adds_per_launch = (sweeps_all / world) * passes * N_WIN
        launch_s = secs / args.steps
        smem_bps = adds_per_launch * 8 / launch_s
        hbm_bytes = B * (HOP * 8 + NUM * 12 + 8)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic = None
        traffic_src = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
            traffic = tr["mbest_kernel"]["dram_bytes_per_window"] * B
            traffic_src = "profiles/dram_traffic.json (one ncu --set full capture of this kernel, per window) x windows per launch"
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(B, world, "device-resident stream"),
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": ms_e2e, "ms_per_step_all": e2e_ms, "statistic": "median over steps",
                    "api": "Periods().m_best(pinned host (B,4096) hop-512 view, num=10, max_length=1024) -> numpy"},
            "gpu_launches": 2 * args.steps,  # per step: pp::tops_kernel (descriptor table, ~2 us) + pp::mbest_kernel
            "roofline": {
                "kernel": "pp::mbest_kernel", "bound": "smem",
                "achieved": smem_bps / 1e9, "peak": smem_peak["per_s"] / 1e9, "unit": "GB/s",
                "frac": smem_bps / smem_peak["per_s"], "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "pp_microbench kind 0 (conflict-free LDS.128 streaming), measured in this run; "
                               "MEASURED_PEAKS.json has no shared-memory figure",
                "algorithmic": "sweeps_executed x 1023 periods x 4096 adds x 8 B shared-memory operand per launch "
                               "(canonical direct fold, SURVEY.md 8d)",
                "sweeps_per_window": sweeps_all / (B * world),
                "executed": {"note": f"hierarchical sweep: {passes} passes over the window per sweep (one per top period in "
                                     f"({PMAX // 2}, {PMAX}] minus the tops riding on another top's pass)",
                             "passes_per_sweep": passes,
                             "achieved": exec_adds_per_launch * 8 / launch_s / 1e9, "unit": "GB/s",
                             "frac": exec_adds_per_launch * 8 / launch_s / smem_peak["per_s"]},
                "fp64": {"achieved_gadd_s": adds_per_launch / launch_s / 1e9, "peak_gadd_s": dadd_peak["per_s"] / 1e9,
                         "frac": adds_per_launch / launch_s / dadd_peak["per_s"]},
                "hbm": {"bound": "hbm", "achieved": hbm_bytes / launch_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": hbm_bytes / launch_s / 1e9 / hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"},
            },
            "clocks": sampler.summary(),
            "status_nonzero_windows": int(cnt[1]),
            "near_tie_windows": int(cnt[2]),
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if parity is not None:
            line["parity"] = parity
        if secondary is not None:
            line["secondary"] = secondary
        emit(line)
    if world > 1:
        dist.barrier()
        sharding.Comm.destroy_all()
        dist.destroy_process_group()


class StdoutGuard:
    """Rank 0 prints exactly ONE JSON line: everything any library writes to fd 1 meanwhile (NCCL's version
    banner is a C-level printf) is sent to stderr, and the line goes out through the saved descriptor."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


_LINES = []


def emit(line: dict):
    _LINES.append(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--windows", type=int, default=131_072, help="windows per GPU per step (multiple of 128)")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--secondary", default="all",
                    help="other BASELINE configs appended to the line: all | none | comma list of 2,3g,4,5qo,5ram")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the M-best results of the last timed step as DIR/<name>.npy (float64; a fixed sample of "
                         "windows above 60 MB); the same arguments give the same inputs, so two builds compare output "
                         "for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    with StdoutGuard():
        if args.impl == "reference":
            run_reference(args, rank)
        else:
            run_b200(args, rank, world, local_rank)
    for text in _LINES:
        print(text, flush=True)


if __name__ == "__main__":
    main()
