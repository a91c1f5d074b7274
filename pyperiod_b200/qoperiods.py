"""`QOPeriods` -- drop-in for pyPeriod.QOPeriods (pyPeriod/QOPeriods.py:148-1310), default path on the B200.

`find_periods(data, num, thresh, ...)` runs the whole residualisation loop of QOPeriods.py:313-596 in
one persistent kernel per batch (csrc/pp_qo.cu): gamma sweep -> dictionary layout -> Gram + Cholesky
-> reconstruction / residual -> stop test.  1-D input returns the reference's `(dict, res)`; a
(B, N) batch returns a QOBatchResult whose `.window(b)` rebuilds that pair for one window.

Supported: `_orthogonalize=False`, `update_weights=True`, `basis_type` "natural" (default) and "ramanujan"
(QOPeriods.py:970-971, 1005-1052), the default `test_function` on the device and a custom one (a host callable
between batched rounds, 1-D or (B, N), either basis).
`_orthogonalize=True` is dead in the reference (best_base is None) and `update_weights=False` raises OverflowError
there under numpy 2: both raise NotImplementedError here instead of silently doing something else.
Deviation from the reference: the stray `print(nonzero_periods)` at QOPeriods.py:488 is not reproduced.
"""
from __future__ import annotations

import ctypes as C
import itertools
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from ._device import Workspace, call, ptr, stage_windows, stream_ptr, to_host, workspace_for
from ._device import RowDownloader
from .periods import Periods, _check_staging, _export, _u32, smem_optin
from .tables import get_tables

MAX_ROUNDS = 64  # device-side cap on `num` (the reference's default num = len(data) is "way too many", :377)
RMAX_FIRST = 1024      # rows of the dense weights array of a batch call (and of the first solve launch of RamanujanPeriods)
RMAX_FACTOR = 3072     # dictionary rows the first find launch holds Cholesky factors for: windows between RMAX_FIRST
                       # and this many rows write their weights to an overflow pool instead of waiting for a second
                       # launch (which is bound by its single largest window); larger ones are re-run
POOL_FRACTION = 16     # overflow-pool slots = windows / POOL_FRACTION (config 5: 1 % of the windows need one)
POOL_MIN_SLOTS = 64
WORKSPACE_FRACTION = 0.5   # share of the free device memory the Cholesky factors of one launch may take


def qo_workspace(lib, dev, n, pmax, num, rmax, basis=_lib.BASIS_NATURAL):
    """Workspace for the QO kernels: factors for the full persistent grid, or as many CTAs as the memory budget holds
    (the launch shrinks its grid to the workspace it is given; one factor of 4096 rows is 68 MB)."""
    with torch.cuda.device(dev):
        full = int(lib.pp_qo_workspace_bytes(n, pmax, num, rmax, 0, basis))
        one = int(lib.pp_qo_workspace_bytes(n, pmax, num, rmax, 1, basis))
        free, _ = torch.cuda.mem_get_info(dev)
    budget = max(one, int(free * WORKSPACE_FRACTION))
    return Workspace.get(dev, min(full, budget))   # a cached buffer that is already large enough is reused


def long_qo_workspace(lib, dev, kind, b, n, pmax, num, rmax, basis=_lib.BASIS_NATURAL):
    """Workspace of the global-memory QO path: residuals and one Cholesky factor per window of a piece, the factors
    within the same share of the free device memory as the on-chip launches."""
    with torch.cuda.device(dev):
        free, _ = torch.cuda.mem_get_info(dev)
    return workspace_for(dev, lib.pp_long_qo_workspace_bytes, kind, max(int(b), 1), n, pmax, num, rmax, basis,
                         int(free * WORKSPACE_FRACTION))


def indicator_rows(q: int, n: int, keep) -> np.ndarray:
    """Natural-basis rows 1[(m - i) % q == 0], i < keep; keep == 0/None keeps all q rows (QOPeriods.py:940-974)."""
    m = np.arange(int(n))
    rows = ((m[None, :] - np.arange(int(q))[:, None]) % int(q) == 0).astype(np.float64)
    return rows[:keep] if keep else rows


def ramanujan_sum(q: int) -> np.ndarray:
    """c_q(m), m < q, as exact integers: mu(q/g) phi(q) / phi(q/g), g = gcd(m, q) (the reference sums complex
    exponentials, QOPeriods.py:1037-1045, and is 1e-13 away from these)."""
    tb = get_tables(max(int(q), 2))
    g = np.gcd(np.arange(int(q)), int(q))
    g[0] = int(q)
    return (tb.mu[int(q) // g] * (int(tb.phi[int(q)]) // tb.phi[int(q) // g])).astype(np.float64)


def ramanujan_rows(q: int, n: int, keep) -> np.ndarray:
    """Ramanujan-basis rows c_q((m - i) mod q), i < keep; keep == 0/None keeps all q rows (QOPeriods.py:970-974)."""
    c = ramanujan_sum(q)
    m = np.arange(int(n))
    rows = c[(m[None, :] - np.arange(int(q))[:, None]) % int(q)]
    return rows[:keep] if keep else rows


def build_subspaces(dict_q, dict_keep, n: int, basis: str = "natural") -> np.ndarray:
    """The stacked dictionary matrix the reference returns under 'subspaces' (an output structure)."""
    rows = ramanujan_rows if basis == "ramanujan" else indicator_rows
    blocks = [np.zeros((0, n))] + [rows(q, n, k) for q, k in zip(dict_q, dict_keep)]
    return np.vstack(blocks)


@dataclass
class QOBatchResult:
    """Padded batch outputs of find_periods; numpy for host input, torch (device) otherwise."""
    periods: object      # (B, num) uint32, first n_periods[b] valid
    norms: object        # (B, num) float64
    n_periods: object    # (B,)
    dict_q: object       # (B, num) int32: dictionary keys in insertion order
    dict_keep: object    # (B, num) int32: rows kept per key (0 = repeated period)
    n_dict: object       # (B,)
    weights: object      # (B, ldw) float64, first n_weights[b] valid -- or, with weights_off, the flat ragged array
    n_weights: object    # (B,)
    res: object          # (B, N) float64 or None
    status: object       # (B,) int32
    n: int = 0
    weights_off: object = None   # (B,) int64 start of window b in the flat `weights` (ragged layout)
    big: object = None           # {window: 1-D weights} of windows whose dictionary outgrew the first launch
    basis: str = "natural"

    def weights_of(self, b: int) -> np.ndarray:
        g = (lambda t: t.cpu().numpy() if isinstance(t, torch.Tensor) else t)
        nw = int(g(self.n_weights)[b])
        if self.big is not None and b in self.big:
            return np.array(g(self.big[b])[:nw])
        if self.weights_off is not None:
            o = int(g(self.weights_off)[b])
            return np.array(g(self.weights[o:o + nw]))
        return np.array(g(self.weights[b, :nw]))

    def window(self, b: int, data_row=None):
        """(dict, res) of window b in the reference's form."""
        g = (lambda t: t.cpu().numpy() if isinstance(t, torch.Tensor) else t)
        st = int(g(self.status)[b])
        res = None if self.res is None else np.array(g(self.res)[b])
        if st == _lib.STATUS_ZERO_INPUT:  # QOPeriods.py:394-406
            out = {"periods": np.array([1]), "norms": np.array([0]), "subspaces": np.ones((1, self.n)),
                   "weights": np.array([0]), "basis_dictionary": {"1": self.n}}
            return out, np.zeros(self.n)
        nd, nw, npd = int(g(self.n_dict)[b]), int(g(self.n_weights)[b]), int(g(self.n_periods)[b])
        if nd == 0:  # nothing was ever solved: the reference still holds its initial lists (:409-415)
            return ({"periods": [], "norms": [], "subspaces": [], "weights": [], "basis_dictionary": {}}, res)
        dq, dk = g(self.dict_q)[b, :nd], g(self.dict_keep)[b, :nd]
        per = np.array(g(self.periods)[b, :npd]).view(np.uint32) if g(self.periods).dtype != np.uint32 \
            else np.array(g(self.periods)[b, :npd])
        out = {"periods": per, "norms": np.array(g(self.norms)[b, :npd]),
               "subspaces": build_subspaces(dq, dk, self.n, self.basis), "weights": self.weights_of(b),
               "basis_dictionary": {str(int(q)): int(k) for q, k in zip(dq, dk)}}
        return out, res


@dataclass
class PeriodsBatch:
    """Batched QOPeriods.get_periods: `flat[off[b] : off[b] + sum(q_b)]` holds window b's waveforms back to back."""
    flat: object      # (sum over windows of sum(q),) float64 -- numpy for host input, torch otherwise
    off: np.ndarray   # (B + 1,) int64
    dict_q: np.ndarray
    n_dict: np.ndarray
    status: object

    def window(self, b: int):
        seg = self.flat[int(self.off[b]): int(self.off[b + 1])]
        seg = seg.cpu().numpy() if isinstance(seg, torch.Tensor) else seg
        out, pos = [], 0
        for q in self.dict_q[b, : int(self.n_dict[b])].tolist():
            out.append(np.array(seg[pos: pos + q]))
            pos += q
        return tuple(out)


def _extract(dev, dq, dk, nd, dq_h, nd_h, weights_flat, ldw, woff):
    """Launch pp_qo_get_periods for a batch.  dq/dk/nd: device int32; dq_h/nd_h: the same on the host (sizes)."""
    lib = _lib.load()
    bsz, kmax = dq_h.shape
    valid = np.arange(kmax)[None, :] < nd_h[:, None]
    qv = np.where(valid, dq_h, 0).astype(np.int64)
    t = qv.sum(axis=1)
    rows = np.zeros(bsz, np.int64)
    for i in range(kmax):
        for j in range(i + 1, kmax):
            both = valid[:, i] & valid[:, j]
            if both.any():
                rows += np.where(both, np.gcd(np.where(both, qv[:, i], 1), np.where(both, qv[:, j], 1)), 0)
    off = np.zeros(bsz + 1, np.int64)
    np.cumsum(t, out=off[1:])
    out = torch.zeros((max(int(off[-1]), 1),), dtype=torch.float64, device=dev)
    iters = torch.zeros((bsz,), dtype=torch.int32, device=dev)
    status = torch.zeros((bsz,), dtype=torch.int32, device=dev)
    off_d = torch.from_numpy(off[:-1].copy()).to(dev)
    call(lib.pp_qo_get_periods, "pp_qo_get_periods", dev, bsz, kmax, int(max(t.max(), 1)), int(rows.max()), ptr(dq),
         ptr(dk), ptr(nd), ptr(weights_flat), int(ldw), ptr(woff), ptr(out), ptr(off_d), ptr(iters), ptr(status),
         stream_ptr(dev))
    return out, off, status


class QOPeriods(Periods):
    """Quadratic-program periodicity decomposition (default path), B200-native."""

    def __init__(self, basis_type="natural", trunc_to_integer_multiple=False, orthogonalize=False, device=None,
                 staging="auto"):
        """staging (not in the reference): where a window lives while it is processed, as for Periods.  "shared"
        stages it in one CTA's shared memory; "global" runs from global memory (csrc/pp_long_qo.cu) for any length;
        "auto" (default) takes the global-memory path exactly for the launches whose on-chip plan does not fit."""
        super().__init__(trunc_to_integer_multiple, orthogonalize, device=device)
        _check_staging(staging)
        self._staging = staging
        self._output = None
        self._basis_type = basis_type
        self._verbose = False
        self._k = 0
        self._window = False
        self._output_bases = None
        self._container = []

    def _long(self, dev, kind, n, pmax, num, rmax, basis=_lib.BASIS_NATURAL, trunc=False) -> bool:
        """Whether one launch runs on the global-memory path (see `staging`)."""
        if self._staging != "auto":
            return self._staging == "global"
        fold = _lib.FOLD_DIRECT if trunc else self._fold()   # the find kernel folds directly under trunc
        return not _lib.qo_fits_on_chip(kind, n, pmax, num, rmax, basis, fold, smem_optin(dev))

    # ------------------------------------------------------------------ detection
    def find_periods(self, data, num=None, thresh=None, min_length=2, max_length=None, update_weights=True,
                     return_res=True, rmax=None, refine=1, **kwargs):
        """QOPeriods.find_periods (QOPeriods.py:313-596).

        Not in the reference: rmax (dictionary rows the first launch holds factors for; windows that outgrow it are
        re-run with room for N rows, so no window is dropped), refine (steps of iterative refinement of the normal
        equations, default 1), return_res.

        test_function(self, data, reconstruction) (QOPeriods.py:388-391, 418) replaces the default stop test for 1-D
        input and batches alike; it is called with numpy 1-D arrays once per window and round, round-major and in
        ascending window order within a round (a stateful test sees that order)."""
        test_function = kwargs.pop("test_function", None)
        if kwargs:
            raise TypeError(f"unexpected arguments {sorted(kwargs)}")
        if self._orthogonalize or not update_weights:
            raise NotImplementedError("orthogonalize=True is dead code in the reference and update_weights=False "
                                      "raises OverflowError there under numpy 2; neither is implemented")
        if self._basis_type not in ("natural", "ramanujan"):
            raise ValueError("basis_type must be 'natural' or 'ramanujan'")
        if test_function is not None:
            return self._find_periods_custom_test(data, num, min_length, max_length, test_function, rmax, refine,
                                                  return_res)
        basis = _lib.BASIS_RAMANUJAN if self._basis_type == "ramanujan" else _lib.BASIS_NATURAL
        lib = _lib.load()
        w = stage_windows(data, self._device, pipeline=True)
        n = w.n
        if max_length is None:
            max_length = int(np.floor(n / 3))
        num = min(n, MAX_ROUNDS) if num is None else int(num)
        if num > MAX_ROUNDS:
            raise ValueError(f"num > {MAX_ROUNDS} is not supported on the device")
        if thresh is None:
            if num > 1:
                raise TypeError("thresh is None: the reference's default test multiplies it (QOPeriods.py:391)")
            thresh = 0.0
        retry_big = rmax is None
        # natural basis: more rows than samples is singular by rank, so N rows is the most a factor ever holds;
        # Ramanujan basis: rows <= sum of the periods (no factor is stored, rmax is the capacity of `weights`)
        rows_cap = n if basis == _lib.BASIS_NATURAL else num * int(max_length)
        if self._staging != "shared":   # dictionaries the global-memory path can hold
            rows_cap = min(rows_cap, _lib.long_qo_max_rows(smem_optin(w.device)))
        pooled = rmax is None and basis == _lib.BASIS_NATURAL and rows_cap > RMAX_FIRST
        rmax = min(rows_cap, RMAX_FACTOR if pooled else RMAX_FIRST) if rmax is None else int(rmax)
        tb = get_tables(max_length)
        dev = w.device
        phi = tb.phi_device(dev)
        cur = torch.cuda.current_stream(dev)

        trunc = int(self._trunc_to_integer_multiple)

        def launch(x_ptr, ldx, count, rmax_l, plan, pool=False, download=False):
            """One pp_qo_find_periods call per piece of `plan` ((first, end, upload event) triples) into one set of
            batch outputs.  pool: the dense weights array keeps RMAX_FIRST columns, larger dictionaries (up to rmax_l
            rows) put their weights into an overflow pool.  A launch whose on-chip plan does not fit (or any launch
            with staging="global") runs whole on the global-memory path, with dense weights."""
            long = self._long(dev, _lib.QO_KIND_FIND, n, int(max_length), num, rmax_l, basis, trunc)
            if long:
                pool = download = False
            rpad = (rmax_l + 31) // 32 * 32
            ldw = min(rpad, (RMAX_FIRST + 31) // 32 * 32) if pool else rpad
            i32 = dict(dtype=torch.int32, device=dev)
            f64 = dict(dtype=torch.float64, device=dev)
            o = dict(periods=torch.zeros((count, num), **i32), norms=torch.zeros((count, num), **f64),
                     n_periods=torch.zeros((count,), **i32), dict_q=torch.zeros((count, num), **i32),
                     dict_keep=torch.zeros((count, num), **i32), n_dict=torch.zeros((count,), **i32),
                     n_weights=torch.zeros((count,), **i32), weights=torch.zeros((count, ldw), **f64),
                     res=torch.empty((count, n), **f64) if return_res else None, status=torch.zeros((count,), **i32))
            slots = max(POOL_MIN_SLOTS, count // POOL_FRACTION) if pool else 0
            o["pool"] = torch.empty((slots, rpad), **f64) if pool else None
            o["pool_slot"] = torch.full((count,), -1, **i32) if pool else None
            if long:
                for _, _, ready in plan:
                    if ready is not None:
                        cur.wait_event(ready)
                ws = long_qo_workspace(lib, dev, _lib.QO_KIND_FIND, count, n, int(max_length), num, rmax_l, basis)
                call(lib.pp_long_qo_find_periods, "pp_long_qo_find_periods", dev, C.c_void_p(x_ptr), ldx, count, n,
                     num, float(thresh), int(min_length), int(max_length), trunc, int(refine), basis, ptr(phi), tb.pmax,
                     int(rmax_l), ptr(o["periods"]), ptr(o["norms"]), ptr(o["n_periods"]), ptr(o["dict_q"]),
                     ptr(o["dict_keep"]), ptr(o["n_dict"]), ptr(o["n_weights"]), ptr(o["weights"]), ldw, ptr(o["res"]),
                     ptr(o["status"]), ptr(ws), ws.numel(), stream_ptr(dev))
                return o
            ws = qo_workspace(lib, dev, n, int(max_length), num, rmax_l, basis)
            # host input: the two large results (residuals, dense weights) travel to the host piece by piece while the
            # next piece is being computed
            down = None
            if download:
                o["host"] = {"res": np.empty((count, n)) if return_res else None, "weights": np.empty((count, ldw))}
                down = RowDownloader(dev, {"res": (o["res"], o["host"]["res"]), "weights": (o["weights"], o["host"]["weights"])})
            for b0, b1, ready in plan:
                if ready is not None:
                    cur.wait_event(ready)
                sl = lambda t: ptr(None if t is None else t[b0:b1])
                call(lib.pp_qo_find_periods, "pp_qo_find_periods", dev, C.c_void_p(x_ptr + b0 * ldx * 8), ldx, b1 - b0,
                     n, num, float(thresh), int(min_length), int(max_length), trunc,
                     self._fold(), int(refine), basis, ptr(phi), tb.pmax, int(rmax_l), ptr(None), 0, sl(o["periods"]),
                     sl(o["norms"]), sl(o["n_periods"]), sl(o["dict_q"]), sl(o["dict_keep"]), sl(o["n_dict"]),
                     sl(o["n_weights"]), sl(o["weights"]), ldw, sl(o["res"]), sl(o["status"]), ptr(o["pool"]), slots,
                     sl(o["pool_slot"]), ptr(ws), ws.numel(), _lib.profile_ptr(), stream_ptr(dev))
                if down is not None:
                    down.mark(b0, b1)
                    down.drain()
            if down is not None:
                down.finish()
            return o

        if pooled and self._long(dev, _lib.QO_KIND_FIND, n, int(max_length), num, rmax, basis, trunc):
            pooled = False   # the global-memory path keeps dense weights
        o = launch(w.ptr, w.ldx, w.b, rmax, w.launch_plan(), pool=pooled,
                   download=w.from_host and w.plan is not None)
        host = o.get("host")
        big = None
        if pooled:
            # weights that went to the overflow pool (one host round trip for the slot table)
            over = torch.nonzero(o["pool_slot"] >= 0).flatten()
            if over.numel():
                rows_o = o["n_weights"][over].tolist()
                slot_o = o["pool_slot"][over].tolist()
                pool_t = o["pool"] if not w.from_host else o["pool"][: max(slot_o) + 1].cpu()
                big = {int(b): pool_t[s_, :r_] for b, s_, r_ in zip(over.tolist(), slot_o, rows_o)}
        rmax_l = rmax
        reruns = 0
        while retry_big:
            idx = torch.nonzero(o["status"] == _lib.STATUS_TOO_LARGE).flatten()
            if not idx.numel():
                break
            # dictionaries that outgrew the factor storage (or found the overflow pool exhausted): re-run just those
            # windows with room for the rows they reported, at least doubled (a later round may need more: the loop
            # repeats until nothing is left or the cap -- N rows, more is singular by rank -- is reached)
            need = int(o["n_weights"][idx].max())
            grown = min(rows_cap, max(2 * rmax_l, (need + 255) // 256 * 256))
            if grown <= rmax_l and not (pooled and reruns == 0):
                break    # already at the cap: these windows keep PP_STATUS_TOO_LARGE
            rmax_l = max(rmax_l, grown)
            reruns += 1
            xb = torch.as_strided(w.tensor, (w.b, n), (w.ldx, 1))[idx].contiguous()
            o2 = launch(xb.data_ptr(), n, int(idx.numel()), rmax_l, [(0, int(idx.numel()), None)])
            for key in ("periods", "norms", "n_periods", "dict_q", "dict_keep", "n_dict", "n_weights", "status"):
                o[key][idx] = o2[key]
            if return_res:
                if host is not None:
                    host["res"][idx.cpu().numpy()] = o2["res"].cpu().numpy()
                else:
                    o["res"][idx] = o2["res"]
            w2 = o2["weights"] if not w.from_host else o2["weights"].cpu()
            big = big or {}
            big.update({int(b): w2[i] for i, b in enumerate(idx.tolist())})
        out = QOBatchResult(_export(w, o["periods"], True), _export(w, o["norms"]), _export(w, o["n_periods"]),
                            _export(w, o["dict_q"]), _export(w, o["dict_keep"]), _export(w, o["n_dict"]),
                            host["weights"] if host is not None else _export(w, o["weights"]), _export(w, o["n_weights"]),
                            (host["res"] if return_res else None) if host is not None else _export(w, o["res"]),
                            _export(w, o["status"]), n=n, big=big, basis=self._basis_type)
        if w.was_1d:
            if int(out.status[0]) == _lib.STATUS_TOO_LARGE:
                raise ValueError("dictionary has more rows than rmax; pass a larger rmax")
            pair = out.window(0)
            self._output = self._output_bases = pair[0]
            return pair
        return out

    # ------------------------------------------------------------------ custom stop test (QOPeriods.py:388-391, 418)
    def _find_periods_custom_test(self, data, num, min_length, max_length, test_function, rmax, refine, return_res):
        """The loop of QOPeriods.py:417-594 with a caller-supplied `test_function(self, data, reconstruction)` for B >= 1
        windows and both bases.  A host callable decides after every round, so the rounds are separate launches; each
        round serves every window still running:
          1. one gamma sweep of the active residuals (Periods.sweep with this instance's fold mode and staging);
          2. one pp_qo_dictionary_rows of every active window's periods, which sizes step 3;
          3. one solve of those periods against the original data (pp_qo_solve / pp_qo_solve_ramanujan, or their
             global-memory namesakes where the launch does not fit on chip): windows above RMAX_FIRST rows (or all
             of them, with an explicit rmax) go to a second launch sized for the largest one;
          4. one download of the solved windows' residuals, from which the reconstructions data - res are formed;
          5. test_function(self, x_b, recon_b) with numpy 1-D arrays for each solved window, in ascending window
             order (the calls are round-major: every window's test of round i comes before any of round i + 1).
        Per window: zero input gives the reference's canned result (:394-406); a failed solve (status SINGULAR,
        TOO_LARGE or GUARD) ends the window with the previous round's outputs (:552-559); False from the test ends it
        with the weights of all periods found and the last period not reported (:560-594)."""
        lib = _lib.load()
        ram = self._basis_type == "ramanujan"
        basis = _lib.BASIS_RAMANUJAN if ram else _lib.BASIS_NATURAL
        kind = _lib.QO_KIND_SOLVE_RAMANUJAN if ram else _lib.QO_KIND_SOLVE
        solvers = {(False, False): "pp_qo_solve", (False, True): "pp_qo_solve_ramanujan",
                   (True, False): "pp_long_qo_solve", (True, True): "pp_long_qo_solve_ramanujan"}
        w = stage_windows(data, self._device)
        n, bsz, dev = w.n, w.b, w.device
        if max_length is None:
            max_length = int(np.floor(n / 3))
        num = n if num is None else int(num)
        i32 = dict(dtype=torch.int32, device=dev)
        xs = torch.as_strided(w.tensor, (bsz, n), (w.ldx, 1))
        x_host = to_host(xs) if bsz else np.zeros((0, n))
        zero = np.sum(np.abs(x_host), axis=1) <= 1e-16   # QOPeriods.py:394-406
        # per-window outputs: the small ones on the host, residuals and (ragged) weights on the device
        found = np.zeros((bsz, num), np.int32)           # periods in found order
        nfound = np.zeros(bsz, np.int32)
        norms = np.zeros((bsz, num))                     # by round, as the reference indexes them (:476-477)
        periods = np.zeros((bsz, num), np.int32)
        n_periods = np.zeros(bsz, np.int32)
        dict_q, dict_keep = np.zeros((bsz, num), np.int32), np.zeros((bsz, num), np.int32)
        n_dict, n_weights = np.zeros(bsz, np.int32), np.zeros(bsz, np.int32)
        status = np.where(zero, _lib.STATUS_ZERO_INPUT, _lib.STATUS_OK).astype(np.int32)
        woff = np.zeros(bsz, np.int64)
        weights = torch.zeros((1,), dtype=torch.float64, device=dev)
        res = xs.clone()
        res[torch.from_numpy(np.flatnonzero(zero)).to(dev)] = 0.0
        sweeper = Periods(self._trunc_to_integer_multiple, False, device=dev, fold_mode=self._fold_mode,
                          staging=self._staging)
        active = np.flatnonzero(~zero)
        for i in range(num):
            if not active.size:
                break
            act_d = torch.from_numpy(active).to(dev)
            _, bp, bv = sweeper.sweep(res[act_d], metric="gamma", min_length=int(min_length), max_length=int(max_length))
            bp, bv = bp.cpu().numpy(), bv.cpu().numpy()
            norms[active, i] = bv
            got = active[bp > 0]
            found[got, nfound[got]] = bp[bp > 0]
            nfound[got] += 1
            kmax = max(int(nfound[active].max()), 1)
            pmax = max(int(found[active, :kmax].max()), 2)
            tb = get_tables(pmax)
            phi = tb.phi_device(dev)
            nper_h = np.zeros(bsz, np.int32)
            nper_h[active] = nfound[active]
            per_d = torch.from_numpy(np.ascontiguousarray(found[:, :kmax])).to(dev)
            nper_d = torch.from_numpy(nper_h).to(dev)
            rows_d = torch.zeros((bsz,), **i32)
            call(lib.pp_qo_dictionary_rows, "pp_qo_dictionary_rows", dev, bsz, kmax, ptr(per_d), ptr(nper_d), pmax,
                 ptr(phi), tb.pmax, ptr(rows_d), stream_ptr(dev))
            rows = rows_d.cpu().numpy().astype(np.int64)
            # weights storage for the dictionaries that can be solved (natural basis: more rows than samples is
            # singular by rank)
            kept = rows if ram else np.where(rows <= n, rows, 0)
            woff_r = np.cumsum(kept) - kept
            wts_r = torch.zeros((max(int(kept.sum()), 1),), dtype=torch.float64, device=dev)
            dq_r, dk_r = torch.zeros((bsz, kmax), **i32), torch.zeros((bsz, kmax), **i32)
            nd_r, nw_r, st_r = (torch.zeros((bsz,), **i32) for _ in range(3))
            res_r = torch.empty((bsz, n), dtype=torch.float64, device=dev)
            if rmax is not None:
                launches = [(active, int(rmax))]
            else:
                big = kept[active] > RMAX_FIRST
                launches = [(active[~big], min(RMAX_FIRST, max(int(kept[active[~big]].max(initial=0)), 32))),
                            (active[big], int(kept[active[big]].max(initial=0)))]
            for order, rmax_l in launches:
                if not order.size:
                    continue
                long = self._long(dev, kind, n, pmax, kmax, rmax_l, basis)
                ws = long_qo_workspace(lib, dev, kind, order.size, n, pmax, kmax, rmax_l, basis) if long else \
                    qo_workspace(lib, dev, n, pmax, kmax, rmax_l, basis)
                name = solvers[(long, ram)]
                order_d = torch.from_numpy(order.astype(np.int32)).to(dev)
                call(getattr(lib, name), name, dev, ptr(w.tensor), w.ldx, bsz, n, kmax, ptr(per_d), ptr(nper_d), pmax,
                     int(refine), ptr(phi), tb.pmax, rmax_l, ptr(order_d), int(order.size), ptr(dq_r), ptr(dk_r),
                     ptr(nd_r), ptr(nw_r), ptr(wts_r), 0, ptr(torch.from_numpy(woff_r).to(dev)), ptr(res_r), ptr(st_r),
                     ptr(ws), ws.numel(), stream_ptr(dev))
            st = st_r.cpu().numpy()
            ok = active[st[active] == _lib.STATUS_OK]
            failed = active[st[active] != _lib.STATUS_OK]
            status[failed] = st[failed]                 # LinAlgError in the reference: previous outputs stay (:552-559)
            if ok.size:
                periods[ok] = found[ok]
                n_periods[ok] = nfound[ok]
                dict_q[ok, :kmax] = dq_r.cpu().numpy()[ok]
                dict_keep[ok, :kmax] = dk_r.cpu().numpy()[ok]
                n_dict[ok] = nd_r.cpu().numpy()[ok]
                ok_d = torch.from_numpy(ok).to(dev)
                res[ok_d] = res_r[ok_d]
                # ragged weights: this round's for the solved windows, the kept ones for every other window
                nw = n_weights.astype(np.int64)
                nw[ok] = nw_r.cpu().numpy()[ok]
                src = woff.copy()
                src[ok] = weights.numel() + woff_r[ok]
                off = np.cumsum(nw) - nw
                idx = np.repeat(src - off, nw) + np.arange(int(nw.sum()))
                weights = torch.cat([weights, wts_r])[torch.from_numpy(idx).to(dev)]
                n_weights, woff = nw.astype(np.int32), off
            active = ok
            if i + 1 >= num or not ok.size:
                break
            recon = x_host[ok] - to_host(res[ok_d])
            go = np.array([bool(test_function(self, x_host[b], recon[j])) for j, b in enumerate(ok)])
            stop = ok[~go]
            n_periods[stop] = np.maximum(nfound[stop] - 1, 0)   # weights of all periods, the last not reported (:560-594)
            active = ok[go]
        host = w.from_host
        dv = (lambda a: a) if host else (lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev))
        out = QOBatchResult(periods.view(np.uint32) if host else _u32(dv(periods)), dv(norms), dv(n_periods),
                            dv(dict_q), dv(dict_keep), dv(n_dict), to_host(weights) if host else weights, dv(n_weights),
                            (to_host(res) if host else res) if return_res else None, dv(status), n=n,
                            weights_off=dv(woff), basis=self._basis_type)
        if w.was_1d:
            if int(out.status[0]) == _lib.STATUS_TOO_LARGE:
                raise ValueError("dictionary has more rows than rmax; pass a larger rmax")
            pair = out.window(0)
            self._output = self._output_bases = pair[0]
            return pair
        return out

    # ------------------------------------------------------------------ extraction (QOPeriods.py:719-741)
    def get_periods(self, weights, dictionary=None, decomp_type="row reduction"):
        """Redistribute shared-GCD energy between the found periods (QOPeriods.py:719-741).

        Reference form: `get_periods(weights, dictionary, decomp_type)` -> tuple of per-period waveforms.
        Batch form: `get_periods(result)` with the QOBatchResult of find_periods / find_periods_with_weights ->
        PeriodsBatch (`.window(b)` is the reference's tuple).  Every window is one CTA of pp_qo_get_periods: the zero
        padded weights minus their projection onto the row space of the pairwise-GCD matrix, by conjugate gradients
        with implicit rows -- what every `decomp_type` of the reference computes (they differ in how the dependent
        rows are removed; the reference's "lu" / "qr" results are rounding noise when rows are dependent).
        Like the reference, "row reduction" raises LinAlgError when the matrix has rank one (a single period, or two
        coprime periods): reduce_rows returns a 1-D array there and np.linalg.solve rejects it."""
        if isinstance(weights, QOBatchResult):
            return self._get_periods_batch(weights)
        layout = [(int(q), int(c)) for q, c in dictionary.items()]
        dev = torch.device("cuda", torch.cuda.current_device()) if self._device is None else torch.device(self._device)
        k = max(len(layout), 1)
        dq = np.zeros((1, k), np.int32)
        dk = np.zeros((1, k), np.int32)
        for i, (q, c) in enumerate(layout):
            dq[0, i], dk[0, i] = q, c
        qs = [q for q, _ in layout]
        if decomp_type == "row reduction" and (len(qs) == 1 or (len(qs) == 2 and int(np.gcd(qs[0], qs[1])) == 1)):
            raise np.linalg.LinAlgError("0-dimensional array given. Array must be at least two-dimensional")
        wt = torch.as_tensor(np.asarray(weights, dtype=np.float64), device=dev).reshape(1, -1)
        out, off, st = _extract(dev, torch.from_numpy(dq).to(dev), torch.from_numpy(dk).to(dev),
                                torch.tensor([len(layout)], dtype=torch.int32, device=dev), dq, np.array([len(layout)]),
                                wt, wt.shape[1], None)
        if int(st[0]) != _lib.STATUS_OK:
            raise np.linalg.LinAlgError("pairwise-GCD projection did not converge")
        flat = out.cpu().numpy()
        return tuple(np.array(flat[s: s + q]) for s, q in zip(np.cumsum([0] + qs[:-1]), qs))

    def _get_periods_batch(self, r: "QOBatchResult"):
        g = (lambda t: t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t))
        dev = r.dict_q.device if isinstance(r.dict_q, torch.Tensor) else \
            (torch.device("cuda", torch.cuda.current_device()) if self._device is None else torch.device(self._device))
        dq_h, nd_h = g(r.dict_q).astype(np.int32), g(r.n_dict).astype(np.int32)
        to_dev = lambda t, dt: (t if isinstance(t, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(t))).to(dev).to(dt)
        wts = to_dev(r.weights, torch.float64)
        if r.weights_off is not None:
            woff = to_dev(r.weights_off, torch.int64)
            flat, ldw = wts.reshape(-1), 0
        else:
            flat, ldw = wts.reshape(-1), wts.shape[1]
            woff = None
            if r.big:   # windows whose weights live outside the padded array: append them, address everything by offset
                woff_h = np.arange(dq_h.shape[0], dtype=np.int64) * ldw
                parts, pos = [flat], flat.numel()
                for b, v in r.big.items():
                    v = to_dev(v, torch.float64).reshape(-1)
                    woff_h[b] = pos
                    pos += v.numel()
                    parts.append(v)
                flat, woff, ldw = torch.cat(parts), torch.from_numpy(woff_h).to(dev), 0
        out, off, st = _extract(dev, to_dev(r.dict_q, torch.int32), to_dev(r.dict_keep, torch.int32),
                                to_dev(r.n_dict, torch.int32), dq_h, nd_h, flat, ldw, woff)
        host = not isinstance(r.dict_q, torch.Tensor)
        return PeriodsBatch(to_host(out) if host else out, off, dq_h, nd_h, to_host(st) if host else st)

    # ------------------------------------------------------------------ Muresan eq. 3 (QOPeriods.py:1122-1232)
    def _muresan(self, x, max_p, normalize):
        lib = _lib.load()
        w = stage_windows(x, self._device)
        max_p = w.n // 2 if max_p is None else int(max_p)
        tb = get_tables(max(max_p, 2))
        dev = w.device
        raw = torch.zeros((w.b, max_p), dtype=torch.float64, device=dev)
        pows = torch.zeros((w.b, max_p), dtype=torch.float64, device=dev)
        best = torch.zeros((w.b,), dtype=torch.int32, device=dev)
        args = (ptr(w.tensor), w.ldx, w.b, w.n, max_p, int(bool(normalize)), ptr(tb.mu_device(dev)), tb.pmax, ptr(raw),
                ptr(pows), ptr(best))
        if w.b and self._long(dev, _lib.QO_KIND_MURESAN, w.n, max_p, 1, 2):
            ws = long_qo_workspace(lib, dev, _lib.QO_KIND_MURESAN, w.b, w.n, max_p, 1, 2)
            call(lib.pp_long_muresan_powers, "pp_long_muresan_powers", dev, *args, ptr(ws), ws.numel(), stream_ptr(dev))
        else:
            call(lib.pp_muresan_powers, "pp_muresan_powers", dev, *args, stream_ptr(dev))
        return w, raw, pows, best, max_p

    def get_best_period_orthogonal(self, x, max_p=None, normalize=False, return_powers=False):
        """Muresan's equation-3 period finder (QOPeriods.py:1175-1232), 1-D or (B, N): powers of every period below
        max_p with the powers of its proper divisors removed; the strongest period, or the powers themselves."""
        w, _, pows, best, max_p = self._muresan(x, max_p, normalize)
        if return_powers:
            out = _export(w, pows)
            return out[0] if w.was_1d else out
        out = _export(w, best)
        if w.was_1d:
            if int(out[0]) >= max_p - 1 and max_p > 2:
                raise IndexError(f"index {int(out[0])} is out of bounds for axis 0 with size {max_p - 1}")  # Q[argmax], :1228
            return int(out[0])
        return out

    def eq_3(self, x, P):
        """Equation 3 of Muresan & Parks for period P (QOPeriods.py:1123-1150); 1-D -> float, (B, N) -> (B,).  A sum
        of squares minus the one lag it leaves out: it can be negative (the finder clamps it, :1210)."""
        w, raw, _, _, _ = self._muresan(x, int(P) + 1, False)
        out = _export(w, raw[:, int(P)].contiguous())
        return float(out[0]) if w.was_1d else out

    def auto_corr(self, x, k):
        """sum_n x[n] x[n + k] (QOPeriods.py:1152-1173)."""
        w = stage_windows(x, self._device)
        xs = torch.as_strided(w.tensor, (w.b, w.n), (w.ldx, 1))
        out = _export(w, (xs[:, : w.n - int(k)] * xs[:, int(k):]).sum(dim=1))
        return float(out[0]) if w.was_1d else out

    @staticmethod
    def solve_quadratic(x, A, type="solve", window=None, k=0):
        """Normal equations (A A^T) w = A x and reconstruction A^T w (QOPeriods.py:743-805) for a caller-supplied dense
        matrix A, on torch tensors (torch.linalg on the device).  A public helper of the reference's surface only: no
        algorithm of this package calls it -- find_periods, find_periods_with_weights and get_periods solve their
        structured systems in the library's own kernels."""
        x = torch.as_tensor(x, dtype=torch.float64, device=A.device if isinstance(A, torch.Tensor) else None)
        A = torch.as_tensor(A, dtype=torch.float64, device=x.device)
        gram, rhs = A @ A.T, A @ x
        if type == "solve":
            w = torch.linalg.solve(gram, rhs)  # raises torch.linalg.LinAlgError on a singular matrix
        else:
            w = torch.linalg.lstsq(gram, rhs.unsqueeze(1)).solution.squeeze(1)
        return w, A.T @ w

    @staticmethod
    def concatenate_periods(weights, dictionary):
        """QOPeriods.py:854-887."""
        pos, parts = 0, []
        for q, r in dictionary.items():
            v = np.zeros(int(q))
            v[0:r] = np.asarray(weights)[pos:pos + r]
            pos += r
            parts.append(v)
        return np.concatenate(parts) if parts else np.zeros(0)

    @staticmethod
    def stack_pairwise_gcd_subspaces(periods):
        """QOPeriods.py:889-938: +/- combs of every pair's gcd, all shifts."""
        periods = [int(p) for p in periods]
        if len(periods) > 1:
            rows = []
            for a, b in itertools.combinations(periods, 2):
                g = int(np.gcd(a, b))
                segs = []
                for p in periods:
                    if p in (a, b):
                        comb = np.tile((np.arange(g) == 0).astype(np.float64), p // g)
                        segs.append(-comb if p == a else comb)
                    else:
                        segs.append(np.zeros(p))
                row = np.concatenate(segs)
                rows.append(row)
                for s in range(1, g):
                    rows.append(np.roll(row, s))
            return np.vstack(rows)
        if len(periods) == 1:
            return np.ones((1, periods[0]))
        return np.ones((1, 1))

    @staticmethod
    def Pp(p, N=1, keep=None, type="natural"):
        """QOPeriods.py:940-974: natural (indicator) or Ramanujan-sum rows."""
        if type == "ramanujan":
            return ramanujan_rows(p, N, keep)
        return indicator_rows(p, N, keep)

    def get_subspaces(self, Q, N):
        """QOPeriods.py:807-852: (A, {str(q): rows kept}); layout rule identical to the device kernel's."""
        phi = get_tables(max([int(q) for q in Q] + [2])).phi
        seen, dim_before, layout = set(), 0, {}
        for q in Q:
            q = int(q)
            seen |= {d for d in range(1, q + 1) if q % d == 0}
            dim = int(sum(int(phi[r]) for r in seen))
            layout[str(q)] = dim - dim_before
            dim_before = dim
        return build_subspaces([int(q) for q in layout], list(layout.values()), N, self._basis_type), layout

    # ------------------------------------------------------------------ properties (QOPeriods.py:1237-1310)
    basis_type = property(lambda s: s._basis_type, lambda s, v: setattr(s, "_basis_type", v))
    verbose = property(lambda s: s._verbose, lambda s, v: setattr(s, "_verbose", v))
    k = property(lambda s: s._k, lambda s, v: setattr(s, "_k", v))
    output_bases = property(lambda s: s._output_bases, lambda s, v: setattr(s, "_output_bases", v))


# ---------------------------------------------------------------------------------------------------------------
# QOPeriodsWithGCDsExtracted (pyPeriod/QOPeriodsWithGCDsExtracted.py:93-143)
# ---------------------------------------------------------------------------------------------------------------
def gcds_extracted_layout(periods) -> dict:
    """{str(p): rows kept} of QOPeriodsWithGCDsExtracted.get_subspaces (QOPeriodsWithGCDsExtracted.py:98-143).

    The dictionary holds the found periods plus every common factor of every pair, in the iteration order of
    `set(sorted(P))` -- a CPython set of ints, evaluated here exactly as the reference evaluates it -- and a period
    keeps p - sum(phi(f)) rows over its proper factors f that are themselves in P (0 = all rows, QOPeriods.py:972).
    """
    q = [int(v) for v in periods]
    phi = get_tables(max(q + [2])).phi
    divisors = lambda n: {d for d in range(1, n + 1) if n % d == 0}
    pset = set()
    for a, b in itertools.combinations(q, 2):
        pset = pset.union(set.intersection(divisors(a), divisors(b)))
    pset = pset.union(q)
    pset = set(sorted(pset))
    layout = {}
    for p in pset:
        f = divisors(p)
        if p != 1:  # get_factors(p, remove_n=True) keeps n when n == 1 (QOPeriods.py:73)
            f = f - {p}
        layout[str(p)] = int(p - sum(int(phi[v]) for v in f.intersection(pset)))
    return layout


@dataclass
class QOGcdBatchResult:
    """Batch outputs of QOPeriodsWithGCDsExtracted.find_periods (numpy)."""
    base: QOBatchResult   # the inherited loop's periods / norms / status
    layouts: list         # per window: {str(p): keep} in dictionary order (None where nothing was solved)
    weights: np.ndarray   # (B, rmax)
    n_weights: np.ndarray
    res: np.ndarray       # (B, N)
    status: np.ndarray    # (B,) status of the re-solve with the GCD-extracted dictionary
    n: int = 0

    def window(self, b: int):
        out, res = self.base.window(b)
        st = int(np.asarray(self.base.status if not isinstance(self.base.status, torch.Tensor)
                            else self.base.status.cpu())[b])
        if st == _lib.STATUS_ZERO_INPUT or self.layouts[b] is None:
            return out, res
        if st != _lib.STATUS_OK or int(self.status[b]) != _lib.STATUS_OK:
            raise NotImplementedError("window %d: the inherited loop stopped on a singular / oversized system; the "
                                      "GCD-extracted dictionary has no duplicate rows there and the reference "
                                      "would carry on differently" % b)
        lay = self.layouts[b]
        out = dict(out)
        out["basis_dictionary"] = dict(lay)
        out["weights"] = np.array(self.weights[b, : int(self.n_weights[b])])
        out["subspaces"] = build_subspaces([int(k) for k in lay], list(lay.values()), self.n)
        return out, np.array(self.res[b])


class QOPeriodsWithGCDsExtracted(QOPeriods):
    """Drop-in for pyPeriod.QOPeriodsWithGCDsExtracted: the inherited residualisation loop with a dictionary that
    also holds the common factors of every pair of found periods.  Both dictionaries span the same space, so the
    loop (sweeps, residuals, stop test) is the device loop of QOPeriods; the layout is evaluated on the host
    (CPython set order is part of the reference's output) and the weights are re-solved on the device."""

    def __init__(self, basis_type="natural", trunc_to_integer_multiple=False, device=None, staging="auto"):
        super().__init__(basis_type, trunc_to_integer_multiple, device=device, staging=staging)

    def get_subspaces(self, Q, N):
        lay = gcds_extracted_layout(Q)
        return build_subspaces([int(k) for k in lay], list(lay.values()), N), lay

    def find_periods(self, data, num=None, thresh=None, min_length=2, max_length=None, update_weights=True,
                     rmax=None, kmax=64, refine=1, **kwargs):
        arr = data if isinstance(data, torch.Tensor) else np.asarray(data, dtype=np.float64)
        was_1d = arr.ndim == 1
        batch = arr.reshape(1, -1) if was_1d else arr
        base = QOPeriods.find_periods(self, batch, num, thresh, min_length, max_length, update_weights,
                                      return_res=True, rmax=rmax, refine=refine, **kwargs)
        g = (lambda t: t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t))
        dq, nd, st = g(base.dict_q), g(base.n_dict), g(base.status)
        bsz, n = dq.shape[0], base.n
        lq = np.zeros((bsz, kmax), np.int32)
        lr = np.zeros((bsz, kmax), np.int32)
        ln = np.zeros((bsz,), np.int32)
        layouts = []
        for b in range(bsz):
            if st[b] == _lib.STATUS_ZERO_INPUT or nd[b] == 0:
                layouts.append(None)
                continue
            lay = gcds_extracted_layout(dq[b, : nd[b]])
            if len(lay) > kmax:
                raise ValueError(f"window {b}: {len(lay)} dictionary entries > kmax={kmax}")
            layouts.append(lay)
            ln[b] = len(lay)
            lq[b, : len(lay)] = [int(k) for k in lay]
            lr[b, : len(lay)] = list(lay.values())
        lib = _lib.load()
        w = stage_windows(batch, self._device)
        dev = w.device
        if rmax is None:
            # rows of the largest layout (0 = all rows of that period), capped at N (more is singular by rank)
            need = max([sum(v if v else int(k) for k, v in lay.items()) for lay in layouts if lay] + [32])
            rmax = min(n, need)
        pmax = int(max(int(lq.max()), 2))
        long = self._long(dev, _lib.QO_KIND_SOLVE, n, pmax, kmax, int(rmax))
        ws = long_qo_workspace(lib, dev, _lib.QO_KIND_SOLVE, bsz, n, pmax, kmax, int(rmax)) if long else \
            qo_workspace(lib, dev, n, pmax, kmax, int(rmax))
        t_lq, t_lr, t_ln = (torch.from_numpy(a).to(dev) for a in (lq, lr, ln))
        ldw = (int(rmax) + 31) // 32 * 32
        weights = torch.zeros((bsz, ldw), dtype=torch.float64, device=dev)
        res = torch.empty((bsz, n), dtype=torch.float64, device=dev)
        n_weights = torch.zeros((bsz,), dtype=torch.int32, device=dev)
        status = torch.zeros((bsz,), dtype=torch.int32, device=dev)
        fn, name = (lib.pp_long_qo_solve_rows, "pp_long_qo_solve_rows") if long else (lib.pp_qo_solve_rows,
                                                                                        "pp_qo_solve_rows")
        call(fn, name, dev, ptr(w.tensor), w.ldx, bsz, n, kmax, ptr(t_lq), ptr(t_lr),
             ptr(t_ln), pmax, int(refine), int(rmax), ptr(n_weights), ptr(weights), ldw, ptr(res), ptr(status),
             ptr(ws), ws.numel(), stream_ptr(dev))
        out = QOGcdBatchResult(base, layouts, to_host(weights), to_host(n_weights), to_host(res), to_host(status), n=n)
        if was_1d:
            pair = out.window(0)
            self._output = self._output_bases = pair[0]
            return pair
        return out
