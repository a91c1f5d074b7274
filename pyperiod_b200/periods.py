"""`Periods` -- drop-in for pyPeriod.Periods (pyPeriod/Periods.py:90-644) on the B200.

Both call shapes of the reference are accepted (SURVEY.md 8b):
  README form   Periods(x, trunc_to_integer_multiple=False, orthogonalize=False); p.m_best(num=10)
  HEAD form     Periods(trunc_to_integer_multiple=False, orthogonalize=False);   p.m_best(x, num=10)
and every method also takes a (B, N) batch of windows.  All arithmetic runs in the CUDA
library (csrc/, through include/pyperiod_b200.h); this file only stages buffers, builds the
integer side tables and shapes the results like the reference does.

1-D input  -> exactly the reference's return types (numpy uint32/float64 arrays; Python
              lists for small_to_large).
(B, N) input -> BatchResult (unpacks as `periods, powers, bases`), bases only when
              return_bases=True (they are 8*num*N bytes per window).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from warnings import warn

import numpy as np
import torch

from . import _lib
from ._device import Windows, call, ptr, stage_windows, stream_ptr, to_host, workspace_for
from .tables import get_tables, orth_chain


@dataclass
class BatchResult:
    """Result of a batched call.  Arrays are numpy for host input, torch (device) otherwise."""
    periods: object          # (B, K) uint32
    powers: object           # (B, K) float64
    bases: object            # (B, K, N) float64 or None
    status: object           # (B,) int32, _lib.STATUS_*
    count: object = None     # (B,) int32 -- small_to_large only: periods accepted
    sweeps: object = None    # (B,) int32 -- M-best only: step-1 sweeps executed
    near_ties: object = None  # (B,) int32 -- M-best only: sweeps decided by the exact re-ranking of near-tied candidates

    def __iter__(self):
        yield self.periods
        yield self.powers
        yield self.bases

    def window(self, b: int):
        """Per-window result in the reference's own form."""
        k = int(self.count[b]) if self.count is not None else self.periods.shape[1]
        per, pw = self.periods[b, :k], self.powers[b, :k]
        bs = None if self.bases is None else self.bases[b, :k]
        if self.count is not None:  # small_to_large returns lists (Periods.py:266-268)
            return (list(map(int, per)), list(map(float, pw)), None if bs is None else [r for r in bs])
        return per, pw, bs


def _is_data(obj) -> bool:
    if isinstance(obj, (bool, np.bool_)) or obj is None:
        return False
    if isinstance(obj, torch.Tensor):
        return obj.dim() >= 1
    return isinstance(obj, (np.ndarray, list, tuple)) and np.ndim(obj) >= 1


STAGINGS = ("auto", "shared", "global")
_smem_optin: dict = {}


def _check_staging(staging):
    if staging not in STAGINGS:
        raise ValueError("staging must be 'auto', 'shared' or 'global'")


def _global_staging(staging, device, algo, n, pmax, num=0, metric=0, trunc=False, orth=False,
                    fold=_lib.FOLD_DIRECT) -> bool:
    """Whether a call runs on the global-memory path: forced by staging="global", never with "shared", and with
    "auto" exactly when the on-chip plan of the call does not fit the device's opt-in shared memory per block."""
    if staging == "global":
        return True
    if staging == "shared":
        return False
    return not _lib.fits_on_chip(algo, n, pmax, num, metric, int(bool(trunc)), int(bool(orth)), fold,
                                 smem_optin(device))


def smem_optin(device) -> int:
    """Opt-in shared memory per block of `device` (cached)."""
    key = str(device)
    if key not in _smem_optin:
        with torch.cuda.device(device):
            _smem_optin[key] = _lib.device_info()["smem_optin_bytes"]
    return _smem_optin[key]


def _u32(t: torch.Tensor):
    return t.view(torch.uint32) if hasattr(torch, "uint32") else t


def _export(w: Windows, t, as_u32=False):
    if t is None:
        return None
    if w.from_host:
        a = to_host(t)
        return a.view(np.uint32) if as_u32 else a
    return _u32(t) if as_u32 else t


class Periods:
    """Sethares-Staley periodicity transforms, B200-native.  See module docstring."""

    def __init__(self, *args, trunc_to_integer_multiple=None, orthogonalize=None, device=None, dtype="fp64",
                 fold_mode=None, devices=None, staging="auto"):
        """device / devices / dtype / fold_mode are not part of the reference API.  devices=[...] (CUDA device indices
        or names) shards a host (B, N) batch over several GPUs from ONE process: contiguous blocks of windows, one
        worker thread and one set of launches per device, results concatenated on the host (windows are independent:
        no collective; the one-process-per-GPU form of the same sharding is pyperiod_b200.sharding).  dtype="fp32" ranks the M-best sweeps in float
        (half the shared-memory traffic) and re-folds every candidate inside the float error bound in fp64, so the
        period lists and norms are those of the fp64 path (the north star's fp32 option).  fold_mode (a
        _lib.FOLD_* value or name) picks how ranking sweeps obtain the residue sums; None = the module default.

        staging picks where a window lives while it is processed.  "shared" stages it in one CTA's shared memory (the
        on-chip kernels; a window whose plan does not fit raises PPError).  "global" runs the global-memory path: the
        residual stays in a device workspace and every sweep is spread over the whole GPU, for windows of any length.
        "auto" (default) takes the on-chip path whenever its plan fits the device and the global path otherwise.  The
        global path ranks with direct fp64 folds: in every fold_mode and with dtype="fp32" it selects the periods and
        powers of the fp64 path (powers can differ from the hierarchical on-chip sweep in the last bits)."""
        args = list(args)
        self._data = None
        if args and _is_data(args[0]):
            self._data = args.pop(0)                      # README form (README.md:71)
        if len(args) > 2:
            raise TypeError("Periods([data,] trunc_to_integer_multiple=False, orthogonalize=False)")
        trunc = args[0] if len(args) >= 1 else False
        orth = args[1] if len(args) >= 2 else False
        if trunc_to_integer_multiple is not None:
            trunc = trunc_to_integer_multiple
        if orthogonalize is not None:
            orth = orthogonalize
        self._trunc_to_integer_multiple = bool(trunc)
        self._orthogonalize = bool(orth)
        self._device = device
        self._devices = None if devices is None else [torch.device("cuda", d) if isinstance(d, int) else torch.device(d)
                                                      for d in devices]
        if self._devices is not None and not self._devices:
            raise ValueError("devices must name at least one CUDA device")
        if dtype not in ("fp64", "fp32"):
            raise ValueError("dtype must be 'fp64' or 'fp32'")
        self._dtype = dtype
        self._fold_mode = fold_mode
        _check_staging(staging)
        self._staging = staging
        _lib.load()  # fail loudly now if the CUDA library is missing

    def _fold(self) -> int:
        """Fold mode of this instance's calls (per-call argument of the C ABI)."""
        if self._fold_mode is None and self._dtype == "fp32":
            return _lib.FOLD_NOMINATE_F32
        return _lib.resolve_fold_mode(self._fold_mode)

    # ------------------------------------------------------------------ single-process multi-device sharding
    def _sharded(self, name, args, kw):
        """Run method `name` on contiguous row blocks of a host (B, N) batch, one block per entry of `devices`, each
        from its own thread (the C calls and the copies release the GIL, so the devices work concurrently), and
        concatenate the per-window results.  Returns None when the call is not a multi-device batch call."""
        if self._devices is None:
            return None
        args = list(args)
        data = args[0] if args and _is_data(args[0]) else self._data
        if data is None or (isinstance(data, torch.Tensor) and data.device.type == "cuda") or np.ndim(data) != 2:
            return None
        rest = args[1:] if args and _is_data(args[0]) else args
        from concurrent.futures import ThreadPoolExecutor
        from .sharding import shard_bounds
        b = data.shape[0]
        devs = self._devices[: max(1, min(len(self._devices), b))]

        def work(i):
            lo, hi = shard_bounds(b, len(devs), i)
            sub = Periods(self._trunc_to_integer_multiple, self._orthogonalize, device=devs[i], dtype=self._dtype,
                          fold_mode=self._fold_mode, staging=self._staging)
            return getattr(sub, name)(data[lo:hi], *rest, **kw)   # row slices keep hop-framed (overlapping) strides

        with ThreadPoolExecutor(len(devs)) as pool:
            parts = [p for p in pool.map(work, range(len(devs))) if p.periods.shape[0]]

        def cat(field):
            vals = [getattr(p, field) for p in parts]
            if any(v is None for v in vals):
                return None
            return np.concatenate([v if isinstance(v, np.ndarray) else v.cpu().numpy() for v in vals])
        k = max(p.periods.shape[1] for p in parts)
        for p in parts:   # small_to_large: per-shard capacity may differ
            if p.periods.shape[1] < k:
                pad = k - p.periods.shape[1]
                p.periods = np.pad(p.periods, ((0, 0), (0, pad)))
                p.powers = np.pad(p.powers, ((0, 0), (0, pad)))
                if p.bases is not None:
                    p.bases = np.pad(p.bases, ((0, 0), (0, pad), (0, 0)))
        return BatchResult(cat("periods"), cat("powers"), cat("bases"), cat("status"), count=cat("count"),
                           sweeps=cat("sweeps"), near_ties=cat("near_ties"))

    # ------------------------------------------------------------------ argument plumbing
    def _split(self, args, names):
        """Peel an optional leading `data` argument off *args (HEAD form) else use the bound data."""
        args = list(args)
        if args and _is_data(args[0]):
            data = args.pop(0)
        elif self._data is not None:
            data = self._data
        else:
            raise TypeError("no data: pass it to the method or to Periods(data)")
        if len(args) > len(names):
            raise TypeError("too many positional arguments")
        return data, dict(zip(names, args))

    # ------------------------------------------------------------------ static operators
    @staticmethod
    def project(data, p=2, trunc_to_integer_multiple=False, orthogonalize=False, return_single_period=False,
                device=None, staging="auto"):
        """Projection onto the p-periodic subspace (Periods.py:142-219); bit-exact with the reference.

        1-D -> (N,) (or (p,) with return_single_period); (B, N) -> (B, N) / (B, p).  staging: see Periods().
        """
        _check_staging(staging)
        lib = _lib.load()
        w = stage_windows(data, device)
        p = int(p)
        if p < 1:
            raise ValueError("need p >= 1")
        out_len = p if return_single_period else w.n
        if p > w.n:
            # The reference pads the window to ONE row of p samples (Periods.py:172-176): without truncation the
            # projection is the data itself (divisor 1; tile(...)[:N], and the "single period" is that length-N
            # vector sliced [0:p]); with truncation the mean runs over zero complete rows: nan (Periods.py:178-184).
            if orthogonalize:
                raise ValueError("orthogonalize with p > len(data) is not supported")
            out = torch.full((w.b, w.n), float("nan"), dtype=torch.float64, device=w.device)
            if not trunc_to_integer_multiple:
                out[:, :] = torch.as_strided(w.tensor, (w.b, w.n), (w.ldx, 1))
            res = _export(w, out)
            return res[0] if w.was_1d else res
        chain = np.asarray(orth_chain(p) if orthogonalize else [], dtype=np.int32)
        out = torch.empty((w.b, out_len), dtype=torch.float64, device=w.device)
        if _global_staging(staging, w.device, _lib.ALGO_PROJECT, w.n, p):
            ws = workspace_for(w.device, lib.pp_long_workspace_bytes, _lib.ALGO_PROJECT, w.b, w.n, p, 0, 0)
            call(lib.pp_long_project, "pp_long_project", w.device, ptr(w.tensor), w.ldx, w.b, w.n, p,
                 int(bool(trunc_to_integer_multiple)), chain.ctypes.data_as(C.c_void_p), len(chain), ptr(out), out_len,
                 out_len, ptr(ws), ws.numel(), stream_ptr(w.device))
        else:
            call(lib.pp_project, "pp_project", w.device, ptr(w.tensor), w.ldx, w.b, w.n, p,
                 int(bool(trunc_to_integer_multiple)), chain.ctypes.data_as(C.c_void_p), len(chain), ptr(out), out_len,
                 out_len, stream_ptr(w.device))
        res = _export(w, out)
        return res[0] if w.was_1d else res

    @staticmethod
    def periodic_norm(x, p=None, device=None):
        """||x|| / sqrt(len) [/ sqrt(p)] (Periods.py:221-241).  1-D -> float, (B, N) -> (B,)."""
        lib = _lib.load()
        w = stage_windows(x, device)
        out = torch.empty((w.b,), dtype=torch.float64, device=w.device)
        call(lib.pp_periodic_norm, "pp_periodic_norm", w.device, ptr(w.tensor), w.ldx, w.b, w.n, int(p) if p else 0,
             ptr(out), stream_ptr(w.device))
        res = _export(w, out)
        return float(res[0]) if w.was_1d else res

    # ------------------------------------------------------------------ one sweep (parity probe)
    def sweep(self, *args, **kw):
        """Metric of every candidate period for each window: returns (metrics[B, pmax+1], best_p[B], best_val[B]).

        metric in {"norm", "gamma", "maxabs", "imposed"}.  Not part of the reference API; it exposes
        the inner loop of Periods.py:501-515 / 324-331 for parity tests and profiling.
        """
        data, pos = self._split(args, ["metric", "min_length", "max_length"])
        kw = {**pos, **kw}
        metric = {"norm": 0, "gamma": 1, "maxabs": 2, "imposed": 3}[kw.get("metric", "norm")]
        lib = _lib.load()
        w = stage_windows(data, self._device)
        pmin = int(kw.get("min_length", 2))
        pmax = kw.get("max_length")
        pmax = math.floor(w.n / 3) if pmax is None else int(pmax)
        trunc = self._trunc_to_integer_multiple and metric != 2
        orth = self._orthogonalize and metric != 2
        tb = get_tables(pmax)
        co, cq, _, _ = tb.device(w.device)
        metrics = torch.zeros((w.b, pmax + 1), dtype=torch.float64, device=w.device)
        best_p = torch.empty((w.b,), dtype=torch.int32, device=w.device)
        best_v = torch.empty((w.b,), dtype=torch.float64, device=w.device)
        if _global_staging(self._staging, w.device, _lib.ALGO_SWEEP, w.n, pmax, 0, metric, trunc, orth, self._fold()):
            ws = workspace_for(w.device, lib.pp_long_workspace_bytes, _lib.ALGO_SWEEP, w.b, w.n, pmax, 0, int(orth))
            call(lib.pp_long_sweep, "pp_long_sweep", w.device, ptr(w.tensor), w.ldx, w.b, w.n, pmin, pmax, metric,
                 int(trunc), int(orth), ptr(co), ptr(cq), tb.pmax, ptr(metrics), ptr(best_p), ptr(best_v), ptr(ws),
                 ws.numel(), stream_ptr(w.device))
            return _export(w, metrics), _export(w, best_p), _export(w, best_v)
        ws = workspace_for(w.device, lib.pp_workspace_bytes, _lib.ALGO_SWEEP, w.n, pmax, 0, int(orth))
        call(lib.pp_sweep, "pp_sweep", w.device, ptr(w.tensor), w.ldx, w.b, w.n, pmin, pmax, metric, int(trunc),
             int(orth), self._fold(), ptr(co), ptr(cq), tb.pmax, ptr(metrics), ptr(best_p), ptr(best_v), ptr(ws),
             ws.numel(), stream_ptr(w.device))
        return _export(w, metrics), _export(w, best_p), _export(w, best_v)

    # ------------------------------------------------------------------ M-best family
    def m_best(self, *args, **kw):
        """M-best (Periods.py:408-430).  m_best([data,] num=5, max_length=None, min_length=2)."""
        return self._m_best_meta(False, args, kw)

    def m_best_gamma(self, *args, **kw):
        """M-best gamma (Periods.py:432-454)."""
        return self._m_best_meta(True, args, kw)

    def _m_best_meta(self, gamma, args, kw):
        multi = self._sharded("m_best_gamma" if gamma else "m_best", args, kw)
        if multi is not None:
            return multi
        data, pos = self._split(args, ["num", "max_length", "min_length"])
        kw = {**pos, **kw}
        return_bases = kw.pop("return_bases", None)
        num = int(kw.pop("num", 5))
        max_length = kw.pop("max_length", None)
        min_length = int(kw.pop("min_length", 2))
        if kw:
            raise TypeError(f"unexpected arguments {sorted(kw)}")
        if self._orthogonalize:
            warn("`Orthogonalize = True` has no effect in M-best.")  # Periods.py:482-483 (HEAD still applies it)
        lib = _lib.load()
        # a large host batch is uploaded in pieces on a side stream; each piece gets its own launch so the
        # PCIe copy overlaps the kernels (the results are compact: one read-back at the end)
        w = stage_windows(data, self._device, pipeline=True)
        if return_bases is None:
            return_bases = w.was_1d
        pmax = math.floor(w.n / 3) if max_length is None else int(max_length)
        tb = get_tables(pmax)
        co, cq, fo, fc = tb.device(w.device)
        orth = int(self._orthogonalize)
        fold = self._fold()
        trunc = int(self._trunc_to_integer_multiple)
        metric = _lib.METRIC_GAMMA if gamma else _lib.METRIC_NORM
        long = _global_staging(self._staging, w.device, _lib.ALGO_MBEST, w.n, pmax, num, metric, trunc, orth, fold)
        if long:
            ws = workspace_for(w.device, lib.pp_long_workspace_bytes, _lib.ALGO_MBEST, w.b, w.n, pmax, num, orth)
        else:
            ws = workspace_for(w.device, lib.pp_workspace_bytes, _lib.ALGO_MBEST, w.n, pmax, num, orth)
        periods = torch.empty((w.b, num), dtype=torch.int32, device=w.device)
        powers = torch.empty((w.b, num), dtype=torch.float64, device=w.device)
        bases = torch.empty((w.b, num, w.n), dtype=torch.float64, device=w.device) if return_bases else None
        sweeps = torch.empty((w.b,), dtype=torch.int32, device=w.device)
        near = torch.empty((w.b,), dtype=torch.int32, device=w.device)
        status = torch.empty((w.b,), dtype=torch.int32, device=w.device)
        cur = torch.cuda.current_stream(w.device)
        for b0, b1, ready in w.launch_plan():
            if ready is not None:
                cur.wait_event(ready)
            if long:
                call(lib.pp_long_mbest, "pp_long_mbest", w.device, C.c_void_p(w.ptr + b0 * w.ldx * 8), w.ldx, b1 - b0,
                     w.n, num, min_length, pmax, int(gamma), trunc, orth, ptr(co), ptr(cq), ptr(fo), ptr(fc), tb.pmax,
                     ptr(periods[b0:b1]), ptr(powers[b0:b1]), ptr(None if bases is None else bases[b0:b1]),
                     ptr(sweeps[b0:b1]), ptr(near[b0:b1]), ptr(status[b0:b1]), ptr(ws), ws.numel(),
                     stream_ptr(w.device))
                continue
            call(lib.pp_mbest, "pp_mbest", w.device, C.c_void_p(w.ptr + b0 * w.ldx * 8), w.ldx, b1 - b0, w.n, num,
                 min_length, pmax, int(gamma), int(self._trunc_to_integer_multiple), orth, fold, ptr(co), ptr(cq),
                 ptr(fo), ptr(fc), tb.pmax, ptr(periods[b0:b1]), ptr(powers[b0:b1]),
                 ptr(None if bases is None else bases[b0:b1]), ptr(sweeps[b0:b1]), ptr(near[b0:b1]),
                 ptr(status[b0:b1]), ptr(ws), ws.numel(), _lib.profile_ptr(), stream_ptr(w.device))
        res = BatchResult(_export(w, periods, True), _export(w, powers), _export(w, bases), _export(w, status),
                          sweeps=_export(w, sweeps), near_ties=_export(w, near))
        if w.was_1d:
            if int(res.status[0]) == _lib.STATUS_NO_PERIOD:
                # the reference dies on `bases[i] = None` when no period has a positive norm
                raise TypeError("no period with a positive norm (all-zero input?)")
            return res.periods[0], res.powers[0], (None if res.bases is None else res.bases[0])
        return res

    # ------------------------------------------------------------------ small-to-large
    def small_to_large(self, *args, **kw):
        """Small-to-large (Periods.py:246-287).  small_to_large([data,] thresh=0.1, n_periods=None).

        Batch extras: kmax (capacity per window, default 32), return_bases.
        """
        multi = self._sharded("small_to_large", args, kw)
        if multi is not None:
            return multi
        data, pos = self._split(args, ["thresh", "n_periods"])
        kw = {**pos, **kw}
        thresh = float(kw.pop("thresh", 0.1))
        n_periods = kw.pop("n_periods", None)
        kmax = int(kw.pop("kmax", 32))
        return_bases = kw.pop("return_bases", None)
        if kw:
            raise TypeError(f"unexpected arguments {sorted(kw)}")
        lib = _lib.load()
        w = stage_windows(data, self._device, pipeline=True)
        if return_bases is None:
            return_bases = w.was_1d
        n_periods = math.floor(w.n / 2) if n_periods is None else int(n_periods)
        tb = get_tables(n_periods)
        co, cq, _, _ = tb.device(w.device)
        orth = int(self._orthogonalize)
        trunc = int(self._trunc_to_integer_multiple)
        long = _global_staging(self._staging, w.device, _lib.ALGO_S2L, w.n, n_periods, 0, _lib.METRIC_IMPOSED, trunc,
                               orth)
        if long:
            ws = workspace_for(w.device, lib.pp_long_workspace_bytes, _lib.ALGO_S2L, w.b, w.n, n_periods, 0, orth)
        else:
            ws = workspace_for(w.device, lib.pp_workspace_bytes, _lib.ALGO_S2L, w.n, n_periods, 0, orth)
        fn, name = (lib.pp_long_small_to_large, "pp_long_small_to_large") if long else \
            (lib.pp_small_to_large, "pp_small_to_large")
        cur = torch.cuda.current_stream(w.device)
        plan = list(w.launch_plan()) if w.plan is None else None   # a pipelined plan issues its copies as it is walked
        while True:
            periods = torch.empty((w.b, kmax), dtype=torch.int32, device=w.device)
            powers = torch.empty((w.b, kmax), dtype=torch.float64, device=w.device)
            bases = torch.empty((w.b, kmax, w.n), dtype=torch.float64, device=w.device) if return_bases else None
            count = torch.empty((w.b,), dtype=torch.int32, device=w.device)
            status = torch.empty((w.b,), dtype=torch.int32, device=w.device)
            for b0, b1, ready in (plan if plan is not None else w.launch_plan()):
                if ready is not None:
                    cur.wait_event(ready)
                call(fn, name, w.device, C.c_void_p(w.ptr + b0 * w.ldx * 8), w.ldx,
                     b1 - b0, w.n, thresh, n_periods, trunc, orth, ptr(co), ptr(cq),
                     tb.pmax, kmax, ptr(periods[b0:b1]), ptr(powers[b0:b1]), ptr(None if bases is None else bases[b0:b1]),
                     ptr(count[b0:b1]), ptr(status[b0:b1]), ptr(ws), ws.numel(), stream_ptr(w.device))
            if not w.was_1d:
                break    # batch: windows over capacity carry PP_STATUS_OVERFLOW (no host synchronisation here)
            need = int(count.max())
            if need <= kmax:
                break
            kmax = need  # 1-D drop-in: rerun with enough room so nothing is truncated
        res = BatchResult(_export(w, periods, True), _export(w, powers), _export(w, bases), _export(w, status),
                          count=_export(w, count))
        return res.window(0) if w.was_1d else res

    # ------------------------------------------------------------------ best correlation
    def best_correlation(self, *args, **kw):
        """Best-correlation (Periods.py:289-349).  best_correlation([data,] num=5, max_length=None, ratio=0.01)."""
        multi = self._sharded("best_correlation", args, kw)
        if multi is not None:
            return multi
        data, pos = self._split(args, ["num", "max_length", "ratio"])
        kw = {**pos, **kw}
        num = int(kw.pop("num", 5))
        max_length = kw.pop("max_length", None)
        ratio = float(kw.pop("ratio", 0.01))
        return_bases = kw.pop("return_bases", None)
        if kw:
            raise TypeError(f"unexpected arguments {sorted(kw)}")
        lib = _lib.load()
        w = stage_windows(data, self._device, pipeline=True)
        if return_bases is None:
            return_bases = w.was_1d
        max_length = math.floor(w.n / 3) if max_length is None else int(max_length)
        tb = get_tables(max_length)
        co, cq, _, _ = tb.device(w.device)
        periods = torch.empty((w.b, num), dtype=torch.int32, device=w.device)
        powers = torch.empty((w.b, num), dtype=torch.float64, device=w.device)
        bases = torch.empty((w.b, num, w.n), dtype=torch.float64, device=w.device) if return_bases else None
        status = torch.empty((w.b,), dtype=torch.int32, device=w.device)
        trunc, orth = int(self._trunc_to_integer_multiple), int(self._orthogonalize)
        long = _global_staging(self._staging, w.device, _lib.ALGO_BCORR, w.n, max_length, num, _lib.METRIC_MAXABS,
                               trunc, orth, self._fold())
        if long:
            ws = workspace_for(w.device, lib.pp_long_workspace_bytes, _lib.ALGO_BCORR, w.b, w.n, max_length, 0, orth)
        else:
            ws = workspace_for(w.device, lib.pp_workspace_bytes, _lib.ALGO_BCORR, w.n, max_length, num, orth)
        cur = torch.cuda.current_stream(w.device)
        for b0, b1, ready in w.launch_plan():
            if ready is not None:
                cur.wait_event(ready)
            if long:
                call(lib.pp_long_best_correlation, "pp_long_best_correlation", w.device,
                     C.c_void_p(w.ptr + b0 * w.ldx * 8), w.ldx, b1 - b0, w.n, num, max_length, ratio, trunc, orth,
                     ptr(co), ptr(cq), tb.pmax, ptr(periods[b0:b1]), ptr(powers[b0:b1]),
                     ptr(None if bases is None else bases[b0:b1]), ptr(status[b0:b1]), ptr(ws), ws.numel(),
                     stream_ptr(w.device))
                continue
            call(lib.pp_best_correlation, "pp_best_correlation", w.device, C.c_void_p(w.ptr + b0 * w.ldx * 8), w.ldx,
                 b1 - b0, w.n, num, max_length, ratio, int(self._trunc_to_integer_multiple), int(self._orthogonalize),
                 self._fold(), ptr(co), ptr(cq), tb.pmax, ptr(periods[b0:b1]), ptr(powers[b0:b1]),
                 ptr(None if bases is None else bases[b0:b1]), ptr(status[b0:b1]), ptr(ws), ws.numel(),
                 stream_ptr(w.device))
        res = BatchResult(_export(w, periods, True), _export(w, powers), _export(w, bases), _export(w, status))
        if w.was_1d:
            if int(res.status[0]) == _lib.STATUS_NO_PERIOD:
                raise TypeError("no period with a non-zero correlation (all-zero input?)")
            return res.periods[0], res.powers[0], (None if res.bases is None else res.bases[0])
        return res

    # ------------------------------------------------------------------ best frequency
    def best_frequency(self, *args, **kw):
        """Best-frequency (Periods.py:351-398).  best_frequency([data,] win_size=None, num=5).

        Per round: the magnitude spectrum of the residual (torch.fft.rfft -- an FFT, cuFFT's), then ONE fused launch
        (pp_best_frequency_round) in which every window finds its own peak bin, derives its own period, projects
        exactly, writes period / norm / basis and updates its residual.  No host synchronisation between rounds.
        Like the reference, a window whose DC bin is the largest has p = round(2*win/0) = round(inf): OverflowError.
        """
        data, pos = self._split(args, ["win_size", "num"])
        kw = {**pos, **kw}
        win_size = kw.pop("win_size", None)
        num = int(kw.pop("num", 5))
        return_bases = kw.pop("return_bases", True)
        if kw:
            raise TypeError(f"unexpected arguments {sorted(kw)}")
        lib = _lib.load()
        w = stage_windows(data, self._device)
        n = w.n
        if win_size is None:
            win_size = n
        elif win_size < n:
            warn("win_size is smaller than the input signal length. It will be truncated and information will be lost.")
        win_size = int(win_size)
        dev = w.device
        work = torch.as_strided(w.tensor, (w.b, n), (w.ldx, 1)).clone()   # data.copy() (Periods.py:381)
        data_norm = torch.empty((w.b,), dtype=torch.float64, device=dev)
        call(lib.pp_periodic_norm, "pp_periodic_norm", dev, ptr(work), n, w.b, n, 0, ptr(data_norm), stream_ptr(dev))
        orth = int(self._orthogonalize)
        tb = get_tables(n if orth else 2)
        co, cq, _, _ = tb.device(dev)
        periods = torch.zeros((w.b, num), dtype=torch.int32, device=dev)
        norms = torch.zeros((w.b, num), dtype=torch.float64, device=dev)
        bases = torch.zeros((w.b, num, n), dtype=torch.float64, device=dev) if return_bases else None
        status = torch.zeros((w.b,), dtype=torch.int32, device=dev)
        long = _global_staging(self._staging, dev, _lib.ALGO_BFREQ, n, n)
        ws = workspace_for(dev, lib.pp_long_workspace_bytes, _lib.ALGO_BFREQ, w.b, n, n, 0, 0) if long else None
        for i in range(num):
            mags = torch.abs(torch.fft.rfft(work, win_size, dim=1)).contiguous()
            args = (ptr(work), w.b, n, ptr(mags), mags.shape[1], win_size, int(self._trunc_to_integer_multiple), orth,
                    ptr(co), ptr(cq), tb.pmax, ptr(periods), ptr(norms), ptr(bases), i, num, ptr(status))
            if long:
                call(lib.pp_long_best_frequency_round, "pp_long_best_frequency_round", dev, *args, ptr(ws), ws.numel(),
                     stream_ptr(dev))
            else:
                call(lib.pp_best_frequency_round, "pp_best_frequency_round", dev, *args, stream_ptr(dev))
        powers = norms / data_norm[:, None]
        res = BatchResult(_export(w, periods, True), _export(w, powers), _export(w, bases), _export(w, status))
        if w.was_1d:
            if int(res.status[0]) != _lib.STATUS_OK:
                raise OverflowError("cannot convert float infinity to integer")   # int(np.round(2*win/0)), Periods.py:386
            return res.periods[0], res.powers[0], (None if res.bases is None else res.bases[0])
        return res

    # ------------------------------------------------------------------ properties (Periods.py:606-644)
    @property
    def trunc_to_integer_multiple(self):
        # the reference's getter returns BOTH flags as a tuple (Periods.py:610-611); kept for fidelity
        return self._trunc_to_integer_multiple, self._orthogonalize

    @trunc_to_integer_multiple.setter
    def trunc_to_integer_multiple(self, value):
        self._trunc_to_integer_multiple, self._orthogonalize = value

    @property
    def orthogonalize(self):
        return self._orthogonalize

    @orthogonalize.setter
    def orthogonalize(self, value):
        self._orthogonalize = value

    @property
    def window(self):
        return self._window

    @window.setter
    def window(self, value):
        self._window = value
