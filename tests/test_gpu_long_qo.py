"""GPU tests of the global-memory ("long") path of QOPeriods, RamanujanPeriods' solve stage and the Muresan finder.

Three groups: (1) the path forced on short windows (staging="global") against the goldens and the on-chip path;
(2) windows whose on-chip plan does not fit (staging="auto") against the oracle; (3) batch behaviour.
"""
import contextlib
import io

import numpy as np
import pytest

from conftest import load_golden
from oracle import qo as oq
from pyperiod_b200 import synth

pytestmark = pytest.mark.gpu


def QO(**kw):
    from pyperiod_b200 import QOPeriods
    return QOPeriods(**kw)


def _check(d, res, g, pre):
    assert np.array_equal(np.asarray(d["periods"]), g[pre + "periods"])
    np.testing.assert_allclose(d["norms"], g[pre + "norms"], rtol=1e-10)
    assert [int(k) for k in d["basis_dictionary"]] == g[pre + "dict_keys"].tolist()
    assert list(d["basis_dictionary"].values()) == g[pre + "dict_vals"].tolist()
    np.testing.assert_allclose(d["weights"], g[pre + "weights"], rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(res, g[pre + "res"], rtol=0, atol=1e-11)


def _oracle(x, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return oq.find_periods(x, **kw)


# ---------------------------------------------------------------- (1) forced long path on short windows
def test_global_goldens():
    g = load_golden("readme_qo_ram")
    c = synth.readme_signal(0)
    d, res = QO(staging="global").find_periods(c, num=2, thresh=0.05)
    _check(d, res, g, "qo_")
    gp = QO(staging="global").get_periods(d["weights"], d["basis_dictionary"], "lstsq")
    want = oq.get_periods(d["weights"], d["basis_dictionary"], "lstsq")
    for u, v in zip(gp, want):
        np.testing.assert_allclose(u, v, rtol=0, atol=1e-10)
    g = load_golden("qo_ram_synth")
    out = QO(staging="global").find_periods(synth.synth_batch(2, 4096, 50_000), num=4, thresh=0.05)
    assert out.status.tolist() == [0, 0]
    for b in range(2):
        _check(*out.window(b), g, f"qo_{b}_")
    from pyperiod_b200 import QOPeriodsWithGCDsExtracted as QG
    g = load_golden("qo_gcd")
    for i in range(4):
        seed, n, num, max_length = (int(v) for v in g[f"c{i}_args"])
        d, res = QG(staging="global").find_periods(synth.synth(n, seed), num=num, thresh=float(g[f"c{i}_thresh"]),
                                                   max_length=max_length or None)
        assert [int(k) for k in d["basis_dictionary"]] == g[f"c{i}_dict_keys"].tolist()
        np.testing.assert_allclose(d["weights"], g[f"c{i}_weights"], rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(res, g[f"c{i}_res"], rtol=0, atol=1e-11)
    g = load_golden("qo_rambasis")
    for i, (n, seed, num, ml) in enumerate([(600, 5, 2, None), (1024, 50_001, 3, None), (2000, 7, 4, 300)]):
        j = [0, 2, 3][i]
        d, res = QO(basis_type="ramanujan", staging="global").find_periods(synth.synth(n, seed), num=num, thresh=0.05,
                                                                          max_length=ml)
        assert np.asarray(d["periods"]).tolist() == g[f"c{j}_periods"].tolist()
        np.testing.assert_allclose(res, g[f"c{j}_res"], rtol=0, atol=1e-10)
    g = load_golden("muresan")
    for i, (n, seed, max_p) in enumerate([(600, 5, None), (1024, 50_001, 300), (2000, 7, None)]):
        x = synth.synth(n, seed)
        for norm in (False, True):
            want = g[f"c{i}_pows_{int(norm)}"]
            got = QO(staging="global").get_best_period_orthogonal(x, max_p, norm, True)
            np.testing.assert_allclose(got, want, rtol=0, atol=1e-10 * np.max(want))
            assert QO(staging="global").get_best_period_orthogonal(x, max_p, norm) == int(g[f"c{i}_best_{int(norm)}"])


def test_global_custom_test_function_and_rerun(monkeypatch):
    x = synth.synth(1024, 50_002)
    rms = lambda v: np.sqrt(np.sum(np.power(v, 2)) / len(v))   # noqa: E731
    d0, res0 = QO().find_periods(x, num=4, thresh=0.05)
    d1, res1 = QO(staging="global").find_periods(x, num=4, thresh=0.05,
                                                 test_function=lambda s, a, y: rms(y) > rms(a) * 0.05)
    assert d0["basis_dictionary"] == d1["basis_dictionary"]
    np.testing.assert_allclose(res1, res0, rtol=0, atol=1e-12)
    from pyperiod_b200 import qoperiods
    xb = synth.synth_batch(6, 1500, 8800)
    ref = QO().find_periods(xb, num=4, thresh=0.05, max_length=400)
    monkeypatch.setattr(qoperiods, "RMAX_FIRST", 96)
    monkeypatch.setattr(qoperiods, "RMAX_FACTOR", 128)
    out = QO(staging="global").find_periods(xb, num=4, thresh=0.05, max_length=400)
    assert out.big is not None and out.status.tolist() == [0] * 6
    for b in range(6):
        d, res = out.window(b)
        d1, res1 = ref.window(b)
        assert d["basis_dictionary"] == d1["basis_dictionary"]
        np.testing.assert_allclose(res, res1, rtol=0, atol=1e-13)


@pytest.mark.parametrize("basis", ["natural", "ramanujan"])
@pytest.mark.parametrize("trunc", [False, True])
def test_global_matches_on_chip_direct(basis, trunc):
    from pyperiod_b200 import _lib
    xb = synth.synth_batch(32, 4096, 123)
    kw = dict(basis_type=basis, trunc_to_integer_multiple=trunc)
    a = QO(**kw, staging="shared")
    a._fold_mode = _lib.FOLD_DIRECT
    on = a.find_periods(xb, num=4, thresh=0.05, rmax=1024)
    lg = QO(**kw, staging="global").find_periods(xb, num=4, thresh=0.05, rmax=1024)
    for key in ("periods", "n_periods", "dict_q", "dict_keep", "n_dict", "status"):
        assert np.array_equal(np.asarray(getattr(on, key)), np.asarray(getattr(lg, key))), key
    # a window that outgrew rmax: the long path reports the rows it needs, the on-chip launch its last solved rows
    ok = np.asarray(on.status) == _lib.STATUS_OK
    assert np.array_equal(np.asarray(on.n_weights)[ok], np.asarray(lg.n_weights)[ok])
    assert np.all(np.asarray(lg.n_weights)[~ok] > 1024)
    for key in ("norms", "weights", "res"):
        u, v = np.asarray(getattr(on, key)), np.asarray(getattr(lg, key))
        assert np.max(np.abs(u - v)) <= 1e-13 * max(np.max(np.abs(u)), 1e-300), key


def test_global_muresan_bit_identical():
    xb = synth.synth_batch(5, 3000, 77)
    for norm in (False, True):
        a = QO(staging="shared")._muresan(xb, None, norm)
        b = QO(staging="global")._muresan(xb, None, norm)
        assert np.array_equal(a[1].cpu().numpy(), b[1].cpu().numpy())
        assert np.array_equal(a[2].cpu().numpy(), b[2].cpu().numpy())
        assert np.array_equal(a[3].cpu().numpy(), b[3].cpu().numpy())


# ---------------------------------------------------------------- (2) above the on-chip limit, against the oracle
def _vs_oracle(d, res, x, basis="natural", trunc=False, **kw):
    e, r = _oracle(x, basis=basis, trunc=trunc, **kw)
    assert np.asarray(d["periods"]).tolist() == np.asarray(e["periods"]).tolist()
    assert d["basis_dictionary"] == e["basis_dictionary"]
    np.testing.assert_allclose(d["norms"], e["norms"], rtol=1e-10)
    if basis == "natural":
        np.testing.assert_allclose(d["weights"], e["weights"], rtol=1e-8, atol=1e-11)
        np.testing.assert_allclose(res, r, rtol=0, atol=1e-11)
    else:
        np.testing.assert_allclose(res, r, rtol=0, atol=1e-10)


@pytest.mark.parametrize("trunc", [False, True])
def test_auto_above_limit_vs_oracle(trunc):
    for n, nb in ((16384, 3), (9000, 1)):
        xb = synth.synth_batch(nb, n, 4242)
        out = QO(trunc_to_integer_multiple=trunc).find_periods(xb, num=4, thresh=0.05)
        assert np.asarray(out.status).tolist() == [0] * nb
        for b in range(nb):
            _vs_oracle(*out.window(b), xb[b], trunc=trunc, num=4, thresh=0.05)


def test_auto_above_limit_ramanujan_gcd_custom():
    x = synth.synth(16384, 99)
    d, res = QO(basis_type="ramanujan").find_periods(x, num=3, thresh=0.05)
    _vs_oracle(d, res, x, basis="ramanujan", num=3, thresh=0.05)
    from pyperiod_b200 import QOPeriodsWithGCDsExtracted as QG
    dg, rg = QG().find_periods(x, num=3, thresh=0.05)
    dn, rn = QO().find_periods(x, num=3, thresh=0.05)
    np.testing.assert_allclose(rg, rn, rtol=0, atol=1e-9)   # both dictionaries span the same space
    rms = lambda v: np.sqrt(np.sum(np.power(v, 2)) / len(v))   # noqa: E731
    dc, rc = QO().find_periods(x, num=3, thresh=0.05, test_function=lambda s, a, y: rms(y) > rms(a) * 0.05)
    assert dc["basis_dictionary"] == dn["basis_dictionary"]
    np.testing.assert_allclose(rc, rn, rtol=0, atol=1e-11)


def test_auto_65536_and_muresan_20000():
    x = synth.synth(65536, 5)
    d, res = QO().find_periods(x, num=2, thresh=0.05, max_length=1024)
    _vs_oracle(d, res, x, num=2, thresh=0.05, max_length=1024)
    x = synth.synth(20000, 8)
    q = QO()
    got = q.get_best_period_orthogonal(x, None, False, True)
    want = oq.get_best_period_orthogonal(x, None, False, True)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-10 * np.max(want))
    assert q.get_best_period_orthogonal(x) == int(np.argmax(got)) if np.max(got) > 0 else 1


def test_ramanujan_weights_long_solve():
    from pyperiod_b200 import RamanujanPeriods
    x = synth.synth(30000, 31)
    d, r = RamanujanPeriods().find_periods_with_weights(x, max_length=600)
    assert len(d["basis_dictionary"]) >= 1
    a, _ = oq.get_subspaces([int(p) for p in np.asarray(d["periods"])], len(x))
    w, recon = oq.solve_quadratic(x, a)
    np.testing.assert_allclose(d["weights"], w, rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(r, x - recon, rtol=0, atol=1e-11)


# ---------------------------------------------------------------- (3) batch behaviour on the long path
def test_long_batch_behaviour():
    import torch
    from pyperiod_b200 import _lib
    sig = synth.synth(4096 + 7 * 512, 3)
    view = np.lib.stride_tricks.sliding_window_view(sig, 4096)[::512]
    out = QO(staging="global").find_periods(view, num=3, thresh=0.05)
    for b in range(view.shape[0]):
        d1, r1 = QO(staging="global").find_periods(np.ascontiguousarray(view[b]), num=3, thresh=0.05)
        db, rb = out.window(b)
        assert db["basis_dictionary"] == d1["basis_dictionary"] and np.array_equal(rb, r1)
    xd = torch.from_numpy(synth.synth_batch(4, 4096, 9)).cuda()
    od = QO(staging="global").find_periods(xd, num=3, thresh=0.05)
    assert od.res.is_cuda and od.weights.is_cuda
    empty = QO(staging="global").find_periods(np.zeros((0, 4096)), num=3, thresh=0.05)
    assert np.asarray(empty.status).shape == (0,)
    z = QO(staging="global").find_periods(np.zeros((2, 4096)), num=3, thresh=0.05)
    assert np.asarray(z.status).tolist() == [_lib.STATUS_ZERO_INPUT] * 2
    d, r = QO(staging="global").find_periods(np.zeros(4096), num=3, thresh=0.05)
    assert d["basis_dictionary"] == {"1": 4096} and not r.any()


def test_long_pieces_are_deterministic(monkeypatch):
    from pyperiod_b200 import qoperiods
    monkeypatch.setattr(qoperiods, "WORKSPACE_FRACTION", 1e-12)   # factor budget of one window: one window a piece
    xb = synth.synth_batch(5, 4096, 17)
    a = QO(staging="global").find_periods(xb, num=4, thresh=0.05)
    b = QO(staging="global").find_periods(xb, num=4, thresh=0.05)
    for key in ("periods", "norms", "dict_q", "n_weights", "weights", "res", "status"):
        assert np.array_equal(np.asarray(getattr(a, key)), np.asarray(getattr(b, key))), key
    monkeypatch.undo()
    c = QO(staging="global").find_periods(xb, num=4, thresh=0.05)
    assert np.array_equal(np.asarray(a.res), np.asarray(c.res))


def test_long_too_large_and_shared_error():
    from pyperiod_b200 import _lib
    n = 37000
    t = np.arange(n)
    rng = np.random.default_rng(1)
    # two strong components of coprime periods near max_length: 24 017 rows, above the capacity and below N
    x = sum(a * rng.standard_normal(p)[t % p] for a, p in ((3.0, 12011), (2.0, 12007)))
    x = x + 0.01 * rng.standard_normal(n)
    kw = dict(num=2, thresh=0.0, min_length=12000, max_length=12100)
    out = QO().find_periods(x[None, :], **kw)
    cap = _lib.long_qo_max_rows(232448)
    assert int(out.status[0]) == _lib.STATUS_TOO_LARGE
    assert cap < int(out.n_weights[0]) <= n
    with pytest.raises(ValueError):
        QO().find_periods(x, **kw)
    with pytest.raises(_lib.PPError):
        QO(staging="shared").find_periods(synth.synth(16384, 99), num=4, thresh=0.05)
