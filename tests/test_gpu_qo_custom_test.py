"""GPU tests of QOPeriods.find_periods with a custom test_function on (B, N) batches and with the Ramanujan basis, and
of the solve entry points behind it (pp_qo_solve_ramanujan, pp_long_qo_solve_ramanujan)."""
import contextlib
import hashlib
import io

import numpy as np
import pytest

from oracle import qo as oq
from pyperiod_b200 import synth

pytestmark = pytest.mark.gpu


def QO(**kw):
    from pyperiod_b200 import QOPeriods
    return QOPeriods(**kw)


def rms(v):
    return np.sqrt(np.sum(np.power(v, 2)) / len(v))


def _oracle(x, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return oq.find_periods(x, **kw)


def _key(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


def _close(u, v, rel):
    u, v = np.asarray(u, dtype=np.float64), np.asarray(v, dtype=np.float64)
    assert u.shape == v.shape
    assert np.max(np.abs(u - v), initial=0.0) <= rel * max(np.max(np.abs(v), initial=0.0), 1e-300)


def _same(d, res, d1, res1, rel=1e-13):
    """window(b) of a batch against the 1-D call on row b."""
    assert np.asarray(d["periods"]).tolist() == np.asarray(d1["periods"]).tolist()
    assert d["basis_dictionary"] == d1["basis_dictionary"]
    _close(d["norms"], d1["norms"], rel)
    _close(d["weights"], d1["weights"], rel)
    if res1 is None:
        assert res is None
    else:
        _close(res, res1, rel)


# ---------------------------------------------------------------- Ramanujan basis, 1-D, against the oracle
@pytest.mark.parametrize("n,seed,num,max_length", [(600, 5, 3, None), (1024, 50_001, 4, None), (2000, 7, 4, 300)])
def test_ramanujan_custom_test_vs_oracle(n, seed, num, max_length):
    x = synth.synth(n, seed)
    stops = {}

    def stop_after(k):
        calls = []

        def f(_s, a, y):
            calls.append(rms(y))
            return len(calls) < k
        return f, calls

    for k in (1, 2, num):
        f, calls = stop_after(k)
        d, res = QO(basis_type="ramanujan").find_periods(x, num=num, thresh=None, max_length=max_length, test_function=f)
        g, calls0 = stop_after(k)
        e, r = _oracle(x, num=num, max_length=max_length, test_function=g, basis="ramanujan")
        assert len(calls) == len(calls0)                  # stop round
        assert np.asarray(d["periods"]).tolist() == np.asarray(e["periods"]).tolist()
        assert d["basis_dictionary"] == e["basis_dictionary"]
        np.testing.assert_allclose(d["norms"], e["norms"], rtol=1e-10)
        np.testing.assert_allclose(res, r, rtol=0, atol=1e-10)
        # weights are the minimum-norm solution (the reference's are one solution of a singular system): compare the
        # reconstruction they give
        np.testing.assert_allclose(d["subspaces"].T @ d["weights"], x - r, rtol=0, atol=1e-10)
        np.testing.assert_allclose(calls, calls0, rtol=1e-10)
        stops[k] = len(calls)
    assert stops[1] == 1
    # the default test written out gives the default path's result
    d0, r0 = QO(basis_type="ramanujan").find_periods(x, num, 0.05, max_length=max_length)
    d1, r1 = QO(basis_type="ramanujan").find_periods(x, num, 0.05, max_length=max_length,
                                                     test_function=lambda s, a, y: rms(y) > rms(a) * 0.05)
    assert np.asarray(d0["periods"]).tolist() == np.asarray(d1["periods"]).tolist()
    assert d0["basis_dictionary"] == d1["basis_dictionary"]
    np.testing.assert_allclose(r1, r0, rtol=0, atol=1e-10)


# ---------------------------------------------------------------- batches, both bases
N_BATCH = 96


def _batch():
    """40 windows of 96 samples: a zero window (0), a window whose test stops after round 1 (1), one dominated by
    period 2 (2: the Ramanujan basis' exact singularity), and noisy periodic windows that stop at different rounds
    or run on until their natural-basis dictionary has more rows than samples (singular by rank)."""
    rng = np.random.default_rng(2024)
    t = np.arange(N_BATCH)
    xb = np.zeros((40, N_BATCH))
    for b in range(1, 40):
        p1, p2 = 3 + b % 13, 5 + (7 * b) % 23
        xb[b] = rng.standard_normal(p1)[t % p1] + 0.5 * rng.standard_normal(p2)[t % p2] + 0.05 * rng.standard_normal(N_BATCH)
    xb[2] = 3.0 * (-1.0) ** t + 0.05 * rng.standard_normal(N_BATCH)
    rounds = {_key(xb[b]): (1 if b == 1 else (99 if b % 4 == 0 else 2 + b % 5)) for b in range(40)}
    return xb, rounds


class Recorder:
    """A stateful test: window k stops after rounds[k] calls; records (window key, recon) per call."""

    def __init__(self, rounds):
        self.rounds, self.calls, self.count = rounds, [], {}

    def __call__(self, _self, a, y):
        k = _key(a)
        self.calls.append((k, np.array(y)))
        self.count[k] = self.count.get(k, 0) + 1
        return self.count[k] < self.rounds[k]


@pytest.mark.parametrize("basis", ["natural", "ramanujan"])
def test_batch_equals_per_window_calls(basis, monkeypatch):
    from pyperiod_b200 import _lib, qoperiods
    monkeypatch.setattr(qoperiods, "RMAX_FIRST", 32)   # dictionaries above 32 rows go to a second, larger launch
    xb, rounds = _batch()
    kw = dict(num=8, thresh=None, max_length=32)
    rec = Recorder(rounds)
    out = QO(basis_type=basis).find_periods(xb, test_function=rec, **kw)
    st = np.asarray(out.status)
    assert st[0] == _lib.STATUS_ZERO_INPUT
    assert (st == _lib.STATUS_SINGULAR).any()
    if basis == "ramanujan":
        assert st[2] == _lib.STATUS_SINGULAR and int(out.n_dict[2]) == 0
    assert (np.asarray(out.n_weights)[st == _lib.STATUS_OK] > 32).any()   # the second launch ran
    assert (st == _lib.STATUS_OK).sum() >= 5
    per_window = {}
    for b in range(40):
        r1 = Recorder(rounds)
        d1, res1 = QO(basis_type=basis).find_periods(xb[b], test_function=r1, **kw)
        d, res = out.window(b)
        _same(d, res, d1, res1)
        one = QO(basis_type=basis).find_periods(xb[b:b + 1], test_function=Recorder(rounds), **kw)
        assert int(one.status[0]) == st[b]
        per_window[_key(xb[b])] = (b, r1.calls)
    assert len(rec.calls) == sum(len(c) for _, c in per_window.values())
    assert st[1] == _lib.STATUS_OK and len(per_window[_key(xb[1])][1]) == 1
    # round-major, ascending window index inside a round; the reconstructions are those of the 1-D calls
    expect, r = [], 0
    while True:
        now = [(b, k) for k, (b, c) in per_window.items() if len(c) > r]
        if not now:
            break
        expect += [(k, r) for b, k in sorted(now)]
        r += 1
    seen = {}
    for (k, y), (k0, r0) in zip(rec.calls, expect):
        assert k == k0
        assert seen.get(k, 0) == r0
        seen[k] = r0 + 1
        _close(y, per_window[k][1][r0][1], 1e-13)


def test_explicit_rmax_reports_too_large():
    from pyperiod_b200 import _lib
    xb, rounds = _batch()
    kw = dict(num=8, thresh=None, max_length=32)
    out = QO().find_periods(xb, test_function=Recorder(rounds), rmax=32, **kw)
    st = np.asarray(out.status)
    big = np.flatnonzero(st == _lib.STATUS_TOO_LARGE)
    assert big.size
    assert np.all(np.asarray(out.n_weights) <= 32)    # the previous round's outputs stay
    b = int(big[0])
    with pytest.raises(ValueError):
        QO().find_periods(xb[b], test_function=Recorder(rounds), rmax=32, **kw)
    ref = QO().find_periods(xb, test_function=Recorder(rounds), **kw)
    ok = st == _lib.STATUS_OK
    for b in np.flatnonzero(ok):
        _same(*out.window(b), *ref.window(b))


# ---------------------------------------------------------------- paths and inputs
@pytest.mark.parametrize("basis", ["natural", "ramanujan"])
def test_global_staging_matches_on_chip(basis):
    from pyperiod_b200 import _lib
    xb = synth.synth_batch(12, 4096, 321)
    f = lambda s, a, y: rms(y) > rms(a) * 0.05   # noqa: E731
    a = QO(basis_type=basis, staging="shared")
    a._fold_mode = _lib.FOLD_DIRECT          # the global-memory sweep folds directly
    on = a.find_periods(xb, num=4, thresh=None, test_function=f)
    lg = QO(basis_type=basis, staging="global").find_periods(xb, num=4, thresh=None, test_function=f)
    for key in ("periods", "n_periods", "dict_q", "dict_keep", "n_dict", "n_weights", "status"):
        assert np.array_equal(np.asarray(getattr(on, key)), np.asarray(getattr(lg, key))), key
    for key in ("norms", "weights", "res"):
        _close(getattr(lg, key), getattr(on, key), 1e-13)


@pytest.mark.parametrize("basis", ["natural", "ramanujan"])
def test_auto_above_on_chip_limit(basis):
    from pyperiod_b200 import _lib
    from pyperiod_b200.periods import smem_optin
    n = 16384
    xb = synth.synth_batch(2, n, 99)
    kind, bas = ((_lib.QO_KIND_SOLVE, _lib.BASIS_NATURAL) if basis == "natural"
                 else (_lib.QO_KIND_SOLVE_RAMANUJAN, _lib.BASIS_RAMANUJAN))
    import torch
    assert not _lib.qo_fits_on_chip(kind, n, n // 3, 3, 1024, bas, _lib.FOLD_DIRECT, smem_optin(torch.device("cuda")))
    out = QO(basis_type=basis).find_periods(xb, num=3, thresh=None,
                                            test_function=lambda s, a, y: rms(y) > rms(a) * 0.05)
    ref = QO(basis_type=basis).find_periods(xb, num=3, thresh=0.05)
    assert np.asarray(out.status).tolist() == [0, 0]
    for b in range(2):
        d, r = out.window(b)
        d0, r0 = ref.window(b)
        assert np.asarray(d["periods"]).tolist() == np.asarray(d0["periods"]).tolist()
        assert d["basis_dictionary"] == d0["basis_dictionary"]
        np.testing.assert_allclose(r, r0, rtol=0, atol=1e-10)


def test_hop_framed_and_device_inputs():
    import torch
    sig = synth.synth(1024 + 15 * 128, 11)
    view = np.lib.stride_tricks.sliding_window_view(sig, 1024)[::128]
    f = lambda s, a, y: rms(y) > rms(a) * 0.1   # noqa: E731
    for basis in ("natural", "ramanujan"):
        ref = QO(basis_type=basis).find_periods(np.ascontiguousarray(view), num=3, thresh=None, test_function=f)
        for data in (view, torch.from_numpy(np.ascontiguousarray(view)).cuda(),
                     torch.from_numpy(np.ascontiguousarray(view))):
            out = QO(basis_type=basis).find_periods(data, num=3, thresh=None, test_function=f)
            if isinstance(data, torch.Tensor) and data.is_cuda:
                assert out.res.is_cuda and out.weights.is_cuda
            for key in ("periods", "norms", "n_periods", "dict_q", "dict_keep", "n_dict", "n_weights", "weights",
                        "weights_off", "res", "status"):
                u, v = getattr(out, key), getattr(ref, key)
                u = u.cpu().numpy() if isinstance(u, torch.Tensor) else u
                assert np.array_equal(np.asarray(u).astype(np.float64), np.asarray(v).astype(np.float64)), key
        d, r = QO(basis_type=basis).find_periods(torch.from_numpy(view[3].copy()).cuda(), num=3, thresh=None,
                                                 test_function=f)
        _same(d, r, *ref.window(3), rel=0.0)
    empty = QO().find_periods(np.zeros((0, 512)), num=3, thresh=None, test_function=f)
    assert np.asarray(empty.status).shape == (0,)
    d, r = QO().find_periods(np.zeros(512), num=3, thresh=None, test_function=f)
    assert d["basis_dictionary"] == {"1": 512} and not r.any()
    out = QO().find_periods(view, num=3, thresh=None, test_function=f, return_res=False)
    assert out.res is None


def test_gcds_extracted_batch_with_custom_test():
    from pyperiod_b200 import QOPeriodsWithGCDsExtracted as QG
    xb = synth.synth_batch(5, 1200, 808)
    f = lambda s, a, y: rms(y) > rms(a) * 0.05   # noqa: E731
    out = QG().find_periods(xb, num=4, thresh=None, test_function=f)
    for b in range(5):
        d, r = out.window(b)
        d1, r1 = QG().find_periods(xb[b], num=4, thresh=None, test_function=f)
        _same(d, r, d1, r1, rel=0.0)
        d0, r0 = QG().find_periods(xb[b], num=4, thresh=0.05)   # the default rule written out
        assert d0["basis_dictionary"] == d["basis_dictionary"]
        np.testing.assert_allclose(r, r0, rtol=0, atol=1e-11)


# ---------------------------------------------------------------- the solve entry points
def _solve_ram(x, lists, rmax, long):
    import torch
    from pyperiod_b200 import _lib
    from pyperiod_b200._device import call, ptr, stream_ptr
    from pyperiod_b200.qoperiods import long_qo_workspace, qo_workspace
    from pyperiod_b200.tables import get_tables
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    b, n = x.shape
    kmax = max(len(v) for v in lists)
    pmax = max(max(v) for v in lists)
    per = np.zeros((b, kmax), np.int32)
    for i, v in enumerate(lists):
        per[i, : len(v)] = v
    i32 = dict(dtype=torch.int32, device=dev)
    per_d, nper = torch.from_numpy(per).to(dev), torch.tensor([len(v) for v in lists], **i32)
    tb = get_tables(pmax)
    ldw = (rmax + 31) // 32 * 32
    dq, dk = torch.zeros((b, kmax), **i32), torch.zeros((b, kmax), **i32)
    nd, nw, st = (torch.zeros((b,), **i32) for _ in range(3))
    w = torch.zeros((b, ldw), dtype=torch.float64, device=dev)
    res = torch.empty((b, n), dtype=torch.float64, device=dev)
    xd = torch.from_numpy(x).to(dev)
    if long:
        ws = long_qo_workspace(lib, dev, _lib.QO_KIND_SOLVE_RAMANUJAN, b, n, pmax, kmax, rmax, _lib.BASIS_RAMANUJAN)
        name = "pp_long_qo_solve_ramanujan"
    else:
        ws = qo_workspace(lib, dev, n, pmax, kmax, rmax, _lib.BASIS_RAMANUJAN)
        name = "pp_qo_solve_ramanujan"
    call(getattr(lib, name), name, dev, ptr(xd), n, b, n, kmax, ptr(per_d), ptr(nper), pmax, 1, ptr(tb.phi_device(dev)),
         tb.pmax, rmax, ptr(None), 0, ptr(dq), ptr(dk), ptr(nd), ptr(nw), ptr(w), ldw, ptr(None), ptr(res), ptr(st),
         ptr(ws), ws.numel(), stream_ptr(dev))
    g = lambda t: t.cpu().numpy()   # noqa: E731
    return g(dq), g(dk), g(nd), g(nw), g(w), g(res), g(st)


def test_solve_ramanujan_entry_points():
    from pyperiod_b200 import _lib
    from pyperiod_b200.qoperiods import build_subspaces
    n = 600
    lists = [[7, 12], [10, 15, 6], [9, 16], [5, 5], [13], [2], [4, 2], [37, 41], [30, 20, 12, 45]]
    x = synth.synth_batch(len(lists), n, 4711)
    on = _solve_ram(x, lists, 64, False)
    lg = _solve_ram(x, lists, 64, True)
    for u, v in zip(on, lg):
        if u.dtype == np.float64:
            _close(u, v, 1e-13)
        else:
            assert np.array_equal(u, v)
    dq, dk, nd, nw, w, res, st = on
    for b, per in enumerate(lists):
        a, layout = oq.get_subspaces(per, n, "ramanujan")
        if per in ([2], [4, 2]):                    # both rows of period 2: the reference's LU raises
            assert st[b] == _lib.STATUS_SINGULAR and nw[b] == 0 and nd[b] == 0
            assert np.array_equal(res[b], x[b])
            continue
        if a.shape[0] > 64:                         # more rows than rmax: the rows needed are reported
            assert st[b] == _lib.STATUS_TOO_LARGE and nw[b] == a.shape[0]
            assert np.array_equal(res[b], x[b])
            continue
        assert st[b] == _lib.STATUS_OK, (b, per)
        assert {str(int(q)): int(k) for q, k in zip(dq[b, : nd[b]], dk[b, : nd[b]])} == layout
        assert nw[b] == a.shape[0]
        coef = np.linalg.lstsq(a.T, x[b], rcond=None)[0]   # least-squares projection onto the row space
        np.testing.assert_allclose(x[b] - res[b], a.T @ coef, rtol=0, atol=1e-10)
        rows = build_subspaces(dq[b, : nd[b]], dk[b, : nd[b]], n, "ramanujan")
        np.testing.assert_allclose(rows.T @ w[b, : nw[b]], x[b] - res[b], rtol=0, atol=1e-10)
    assert (st == _lib.STATUS_TOO_LARGE).sum() == 2
    # with room for every row the two large dictionaries solve as well
    big = _solve_ram(x, lists, 256, False)
    assert np.all(big[6][[0, 1, 2, 3, 4, 7, 8]] == _lib.STATUS_OK)


def test_long_workspace_query_never_zero_for_valid_shapes():
    from pyperiod_b200 import _lib
    lib = _lib.load()
    for b in (1, 7, 4096):
        for n in (64, 4096, 100_000):
            for num in (1, 4, 64):
                for rmax in (2, 1024, 30_000):
                    for budget in (0, 1 << 30):
                        got = lib.pp_long_qo_workspace_bytes(_lib.QO_KIND_SOLVE_RAMANUJAN, b, n, n // 3, num, rmax,
                                                             _lib.BASIS_RAMANUJAN, budget)
                        assert got > 0, (b, n, num, rmax, budget)
