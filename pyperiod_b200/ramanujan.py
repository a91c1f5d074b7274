"""`RamanujanPeriods` -- drop-in for pyPeriod.RamanujanPeriods (pyPeriod/RamanujanPeriods.py:61-169).

`find_periods` is the Ramanujan periodogram: a fold of every period followed by a dense contraction
with the circulant of Ramanujan sums on the FP64 tensor cores (csrc/pp_ramanujan.cu);
`find_periods_with_weights` thresholds it on the device and hands the selected periods to the
QOPeriods solve stage (csrc/pp_qo.cu).  method="divisor" computes the same fp64 periodogram from the divisor form of
the Ramanujan sums instead (csrc/pp_ram_divisor.cu); fp64 periodograms whose fused on-chip plan does not fit in shared
memory take that form too, from global memory, whatever the method.  Values are fp64;
the reference stores its projection in float32 (RamanujanPeriods.py:127), so agreement with it is bounded by ~1e-7 relative on the norms.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._device import Workspace, call, ptr, stage_windows, stream_ptr, workspace_for
from .periods import _export, smem_optin
from .qoperiods import RMAX_FIRST, QOBatchResult, QOPeriods, long_qo_workspace, qo_workspace
from .tables import get_tables

TILE_WINDOWS = 2048      # tf32 / f32_compat: windows whose folds are held at once (7.5 MB per window at qmax = 1365)
RMAX_TWO_CTAS = 1 << 30    # rows above which large dictionaries get a launch of their own (off: one launch, longest first, measured 5 % faster)
L2_GROUP_WINDOWS = 1024  # fp64 (fused kernel): windows kept L2-resident while every period passes over them


class RamanujanPeriods(QOPeriods):
    def __init__(self, basis_type="natural", device=None, precision="fp64", staging="auto", method="dense"):
        """precision (not part of the reference API): "fp64" (FP64 tensor cores, default: the fp64 value of the
        reference's formula), "tf32" (split TF32 contraction on the tcgen05 tensor cores, fp32 accumulation: norms to
        ~1e-5 relative), or "f32_compat" (the reference's own float32 storage and summation order,
        RamanujanPeriods.py:127 and :77-78, reproduced operation by operation: norms equal the reference's to the
        last float32 bit).  staging: see QOPeriods; it applies to the solve stage of find_periods_with_weights.
        method (not part of the reference API): "dense" (default: the fused tensor-core contraction above wherever its
        plan fits in shared memory, max_length <= 3 200 on a B200; above that the divisor form) or "divisor" (the
        same fp64 norms from the divisor form of the Ramanujan sums, csrc/pp_ram_divisor.cu: a fold and a few comb
        sums per period instead of a dense product, O(N + q omega(q)) per period instead of O(q^2); values differ
        from the dense path's by rounding only).  The divisor form runs on chip when its plan fits in shared memory
        and from global memory otherwise.  "divisor" needs precision="fp64"; tf32 and f32_compat run on chip only and
        raise PPError above their limits."""
        if method not in ("dense", "divisor"):
            raise ValueError("method must be 'dense' or 'divisor'")
        if method == "divisor" and precision != "fp64":
            raise ValueError("method='divisor' computes the fp64 periodogram only (precision='fp64'): tf32 and "
                             "f32_compat reproduce the rounding of a dense contraction")
        super().__init__(basis_type, False, False, device=device, staging=staging)
        if precision not in ("fp64", "tf32", "f32_compat"):
            raise ValueError("precision must be 'fp64', 'tf32' or 'f32_compat'")
        self._method = method
        self._precision = precision
        self._verbose = None
        self._k = 0

    # ------------------------------------------------------------------ periodogram
    def _norms_device(self, w, min_length, max_length, _long=None):
        """Norms [B, max_length + 1] on the device.  A dense fp64 periodogram whose fused on-chip plan does not fit runs
        in divisor form.  _long (tests): True forces the divisor form from global memory, False the on-chip kernel of
        the method, None lets the plans decide."""
        lib = _lib.load()
        tb = get_tables(max_length)
        if self._method == "divisor":
            return self._norms_divisor(lib, tb, w, min_length, max_length, _long)
        mode = {"fp64": _lib.RAM_FP64, "tf32": _lib.RAM_TF32, "f32_compat": _lib.RAM_F32COMPAT}[self._precision]
        fits = not _long
        if mode == _lib.RAM_FP64 and _long is None and 1 <= min_length <= max_length <= w.n:
            fits = _lib.ramanujan_fits_on_chip(mode, w.n, min_length, max_length, smem_optin(w.device))
        if mode == _lib.RAM_FP64 and not fits:
            return self._norms_divisor(lib, tb, w, min_length, max_length, _long)
        mu, phi = tb.mu_device(w.device), tb.phi_device(w.device)
        # fp64: the fused kernel needs no fold storage; `tile` is the group of windows kept L2-resident.  The other
        # modes hold the folds (and products) of one tile in the workspace (7.5 MB per window at qmax = 1365).
        tile = {"fp64": L2_GROUP_WINDOWS, "tf32": TILE_WINDOWS, "f32_compat": TILE_WINDOWS // 2}[self._precision]
        if mode != _lib.RAM_FP64:
            tile = min(tile, max(4, w.b))
        ws = workspace_for(w.device, lib.pp_ramanujan_workspace_bytes, w.n, min_length, max_length, tile, mode)
        norms = torch.zeros((w.b, max_length + 1), dtype=torch.float64, device=w.device)
        fn = {"fp64": lib.pp_ramanujan_norms, "tf32": lib.pp_ramanujan_norms_tf32,
              "f32_compat": lib.pp_ramanujan_norms_f32compat}[self._precision]
        call(fn, "pp_ramanujan_norms", w.device, ptr(w.tensor), w.ldx, w.b, w.n, int(min_length), int(max_length),
             ptr(mu), ptr(phi), tb.pmax, tile, ptr(norms), max_length + 1, ptr(ws), ws.numel(), stream_ptr(w.device))
        return norms

    def _norms_divisor(self, lib, tb, w, min_length, max_length, _long):
        """The divisor-form periodogram (pp_ramanujan_norms_divisor): shared-memory staging when its plan fits."""
        spf, phi = tb.spf_device(w.device), tb.phi_device(w.device)
        staging = _lib.STAGING_AUTO
        if _long is not None:
            staging = _lib.STAGING_GLOBAL if _long else _lib.STAGING_SHARED
        elif 1 <= min_length <= max_length <= w.n:
            fits = _lib.ramanujan_divisor_fits_on_chip(w.n, min_length, max_length, smem_optin(w.device))
            staging = _lib.STAGING_SHARED if fits else _lib.STAGING_GLOBAL
        ws = workspace_for(w.device, lib.pp_ramanujan_divisor_workspace_bytes, w.b, w.n, min_length, max_length)
        norms = torch.zeros((w.b, max_length + 1), dtype=torch.float64, device=w.device)
        call(lib.pp_ramanujan_norms_divisor, "pp_ramanujan_norms_divisor", w.device, ptr(w.tensor), w.ldx, w.b, w.n,
             int(min_length), int(max_length), ptr(spf), ptr(phi), tb.pmax, staging, ptr(norms), max_length + 1,
             ptr(ws), ws.numel(), stream_ptr(w.device))
        return norms

    def find_periods(self, x, min_length=2, max_length=None, select_periods=None):
        """Periodogram norms, length max_length+1, zero below min_length (RamanujanPeriods.py:67-86)."""
        w = stage_windows(x, self._device)
        if not max_length:
            max_length = w.n // 3
        norms = _export(w, self._norms_device(w, min_length, max_length))
        norms = norms[0] if w.was_1d else norms
        if select_periods:
            if hasattr(select_periods, "__call__"):
                return select_periods(norms)
            return None  # the reference falls through without a return value here
        return norms

    # ------------------------------------------------------------------ periodogram + quadratic program
    def find_periods_with_weights(self, x, min_length=2, max_length=None, thresh=0.2, kmax=32, rmax=None,
                                  return_res=True, refine=1, **kwargs):
        """RamanujanPeriods.py:88-122: periods over thresh * max norm -> dictionary -> normal equations.

        `test_function(norms) -> periods` replaces the threshold rule as in the reference (:94-101); it is a host
        callable, evaluated between the periodogram kernel and the solve kernel (per window for a batch).
        Every window is solved whatever the size of its dictionary (up to N rows; more is singular by rank): the
        rows are counted first (pp_qo_dictionary_rows), windows above RMAX_FIRST rows go to a second launch sized
        for the largest of them, and the weights come back in a ragged array."""
        test_function = kwargs.pop("test_function", None)
        if kwargs:
            raise TypeError(f"unexpected arguments {sorted(kwargs)}")
        lib = _lib.load()
        w = stage_windows(x, self._device)
        n, dev = w.n, w.device
        if not max_length:
            max_length = n // 3
        norms = self._norms_device(w, min_length, max_length)
        i32 = dict(dtype=torch.int32, device=dev)
        if test_function is not None:
            picked = [np.asarray(test_function(row), dtype=np.int64).flatten() for row in norms.cpu().numpy()]
            kmax = max([len(v) for v in picked] + [1])
            per_h = np.zeros((w.b, kmax), np.int32)
            for b, v in enumerate(picked):
                if len(v) and (v.min() < 1 or v.max() > n):
                    raise ValueError("test_function must return periods in [1, len(x)]")
                per_h[b, : len(v)] = v
            periods = torch.from_numpy(per_h).to(dev)
            nper = torch.tensor([len(v) for v in picked], **i32)
        else:
            while True:
                periods = torch.zeros((w.b, kmax), **i32)
                nper = torch.zeros((w.b,), **i32)
                call(lib.pp_ramanujan_select, "pp_ramanujan_select", dev, ptr(norms), w.b, max_length + 1,
                     max_length + 1, float(thresh), kmax, ptr(periods), ptr(nper), stream_ptr(dev))
                need = int(nper.max()) if w.b else 0
                if need <= kmax:
                    break
                kmax = need
        pmax = int(max(int(periods.max()) if w.b else 2, max_length, 2))
        tb = get_tables(pmax)
        phi = tb.phi_device(dev)
        # rows of every window's dictionary: sizes the factor storage and the ragged weights
        rows = torch.zeros((w.b,), **i32)
        call(lib.pp_qo_dictionary_rows, "pp_qo_dictionary_rows", dev, w.b, kmax, ptr(periods), ptr(nper), pmax, ptr(phi),
             tb.pmax, ptr(rows), stream_ptr(dev))
        solvable = rows <= n                              # more rows than samples: singular by rank, no storage
        kept = torch.where(solvable, rows, torch.zeros_like(rows)).long()
        woff = torch.cumsum(kept, 0) - kept               # exclusive prefix sum
        total = int(kept.sum()) if w.b else 0
        weights = torch.zeros((max(total, 1),), dtype=torch.float64, device=dev)
        dict_q, dict_keep = torch.zeros((w.b, kmax), **i32), torch.zeros((w.b, kmax), **i32)
        n_dict, n_weights, status = (torch.zeros((w.b,), **i32) for _ in range(3))
        res = torch.empty((w.b, n), dtype=torch.float64, device=dev) if return_res else None
        first = RMAX_FIRST if rmax is None else int(rmax)
        small = torch.nonzero(~solvable | (rows <= first)).flatten().int()
        bigw = torch.nonzero(solvable & (rows > first)).flatten()
        launches = [(small, min(first, max(int(kept[small.long()].max()) if small.numel() else 32, 32)))]
        # Large dictionaries: one more launch, longest factorisations first, sized for the largest.  Above ~3300 rows
        # the solve kernel keeps the window in global memory so that two CTAs per SM still fit (the factorisation of
        # one window is a latency-bound chain: a second CTA on the SM nearly doubles the throughput).
        # RMAX_TWO_CTAS splits them into two launches instead (measured 5 % slower: the few largest windows then
        # have no smaller ones to fill the tail of their launch).
        for sel in (bigw[rows[bigw] <= RMAX_TWO_CTAS], bigw[rows[bigw] > RMAX_TWO_CTAS]):
            if sel.numel():
                order = sel[torch.argsort(rows[sel], descending=True)].int()   # longest factorisations first
                launches.append((order, int(rows[sel].max())))
        for order, rmax_l in launches:
            if order.numel() == 0:
                continue
            if self._long(dev, _lib.QO_KIND_SOLVE, n, pmax, kmax, rmax_l):
                ws = long_qo_workspace(lib, dev, _lib.QO_KIND_SOLVE, int(order.numel()), n, pmax, kmax, rmax_l)
                fn, name = lib.pp_long_qo_solve, "pp_long_qo_solve"
            else:
                ws = qo_workspace(lib, dev, n, pmax, kmax, rmax_l)
                fn, name = lib.pp_qo_solve, "pp_qo_solve"
            call(fn, name, dev, ptr(w.tensor), w.ldx, w.b, n, kmax, ptr(periods), ptr(nper), pmax,
                 int(refine), ptr(phi), tb.pmax, int(rmax_l), ptr(order), int(order.numel()), ptr(dict_q), ptr(dict_keep),
                 ptr(n_dict), ptr(n_weights), ptr(weights), 0, ptr(woff), ptr(res), ptr(status), ptr(ws), ws.numel(),
                 stream_ptr(dev))
        sel_norms = torch.gather(norms, 1, periods.long().clamp(max=max_length))  # norms[periods] (:116), padded entries unused
        out = QOBatchResult(_export(w, periods), _export(w, sel_norms), _export(w, nper), _export(w, dict_q),
                            _export(w, dict_keep), _export(w, n_dict), _export(w, weights), _export(w, n_weights),
                            _export(w, res), _export(w, status), n=n, weights_off=_export(w, woff))
        if w.was_1d:
            st = int(out.status[0])
            if st == _lib.STATUS_SINGULAR:
                raise np.linalg.LinAlgError("Singular matrix")  # the reference's np.linalg.solve raises here
            d, r = out.window(0)
            d["periods"] = np.asarray(d["periods"]).astype(np.int64)  # np.argwhere indices (:97-101)
            self._output = d
            return d, r
        return out
