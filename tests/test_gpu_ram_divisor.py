"""GPU tests of the divisor-form fp64 Ramanujan periodogram (RamanujanPeriods(method="divisor"), csrc/pp_ram_divisor.cu).

(1) small windows against the divisor-form oracle and the dense path; (2) integer-valued inputs against the exact
value; (3) config 5's shape against the dense path, with weights; (4) global-memory against shared-memory staging and
the input layouts; (5) the dispatch at the limit of the on-chip plan; (6) long windows against the oracle; (7) run to
run bit identity; (8) edge cases.
"""
from fractions import Fraction

import numpy as np
import pytest

from conftest import tie_inputs
from divisor_oracle import norms_divisor_form_f64
from oracle.numtheory import phi
from oracle.ramanujan import norms_closed_form_f64
from pyperiod_b200 import synth

pytestmark = pytest.mark.gpu

RTOL = 1e-11        # the bar of the dense fp64 path against the closed form
RTOL_DENSE = 2e-11  # divisor against dense: each within RTOL of the exact value, so within 2 RTOL of each other


def R(**kw):
    from pyperiod_b200 import RamanujanPeriods
    return RamanujanPeriods(**kw)


def D(**kw):
    return R(method="divisor", **kw)


def _norms(x, lo, hi, long=None, method="divisor"):
    import torch
    from pyperiod_b200._device import stage_windows
    r = R(method=method)
    w = stage_windows(x, r._device)
    out = r._norms_device(w, lo, hi, _long=long)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _close(got, want, lo, what, rtol=RTOL):
    assert np.all(got[..., :lo] == 0), what
    err = np.abs(got[..., lo:] - want[..., lo:])
    bad = err > rtol * np.abs(want[..., lo:])
    assert not bad.any(), (what, np.argwhere(bad)[:5], float((err / np.abs(want[..., lo:])).max()))


# ---------------------------------------------------------------- (1) small windows: oracle and dense
@pytest.mark.parametrize("n", [999, 1024, 2000])
def test_small_windows_vs_oracle_and_dense(n):
    xb = synth.synth_batch(70, n, 3 + n)
    for lo, hi in ((1, n // 3), (3, 333), (n - 5, n)):
        want = np.stack([norms_divisor_form_f64(xb[b], lo, hi) for b in range(70)])
        dense = _norms(xb, lo, hi, method="dense")
        for b in (1, 5, 8, 9, 70):
            got = D().find_periods(xb[:b], lo, hi)
            assert got.shape == (b, hi + 1) and got.dtype == np.float64
            _close(got, want[:b], lo, ("oracle", n, lo, hi, b))
            _close(got, dense[:b], lo, ("dense", n, lo, hi, b), rtol=RTOL_DENSE)
    one = D().find_periods(xb[0])
    assert one.shape == (n // 3 + 1,)
    _close(one, norms_divisor_form_f64(xb[0]), 2, ("1-D", n))


# ---------------------------------------------------------------- (2) integer-valued inputs: exact
def _exact_norms(x, hi):
    """Exact norms [hi + 1] of an integer-valued window: the divisor form in Python integers and Fractions."""
    xi = np.asarray(x).astype(np.int64)
    assert np.array_equal(xi, x)
    n = len(xi)
    idx = np.arange(n)
    mu = [0, 1] + [None] * (hi - 1)
    for q in range(2, hi + 1):   # Moebius by trial division (small q)
        t, k, m = q, 2, 1
        while k * k <= t:
            if t % k == 0:
                t //= k
                if t % k == 0:
                    m = 0
                    break
                m = -m
            k += 1
        if m != 0 and t > 1:
            m = -m
        mu[q] = m
    out = [Fraction(0)] * (hi + 1)
    for q in range(2, hi + 1):
        s = np.bincount(idx % q, weights=xi, minlength=q).astype(np.int64)
        cnt = np.bincount(idx % q, minlength=q)
        z = np.zeros(q, dtype=np.int64)
        for d in range(1, q + 1):
            if q % d == 0 and mu[q // d] != 0:
                z += mu[q // d] * d * np.tile(s.reshape(q // d, d).sum(0), q // d)
        e = sum(int(c) * int(v) * int(v) for c, v in zip(cnt, z))
        ph = phi(q)
        out[q] = Fraction(q * q, ph ** 4) * e
    return out


def test_integer_inputs_exact():
    hi = 400
    ins = tie_inputs(4096)
    names = sorted(ins)
    xb = np.stack([ins[k] for k in names])
    got = D().find_periods(xb, 2, hi)
    dense = _norms(xb, 2, hi, method="dense")
    for b, name in enumerate(names):
        exact = _exact_norms(xb[b], hi)
        for q in range(2, hi + 1):
            g, e = got[b, q], exact[q]
            if e == 0:
                assert g == 0.0, (name, q, g)
                continue
            assert abs(Fraction(g) - e) <= Fraction(1, 10 ** 13) * e, (name, q, g, float(e))
            assert abs(g - dense[b, q]) <= 1e-13 * abs(float(e)) + 1e-13 * abs(dense[b, q]), (name, q)


# ---------------------------------------------------------------- (3) config 5's shape
def test_config5_shape_vs_dense():
    n, thresh = 4096, 0.2
    xb = synth.synth_batch(256, n, 500)
    dense = R().find_periods(xb)
    got = D().find_periods(xb)
    _close(got, dense, 2, "config 5", rtol=RTOL_DENSE)
    ratio = dense / np.abs(dense.max(axis=1, keepdims=True))
    assert np.min(np.abs(ratio - thresh)) > 1e-9          # no period sits on the threshold
    a = R().find_periods_with_weights(xb, thresh=thresh)
    b = D().find_periods_with_weights(xb, thresh=thresh)
    for f in ("periods", "n_periods", "dict_q", "dict_keep", "n_dict", "weights", "n_weights", "weights_off", "res",
              "status"):
        assert np.array_equal(np.asarray(getattr(a, f)), np.asarray(getattr(b, f))), f
    np.testing.assert_allclose(np.asarray(b.norms), np.asarray(a.norms), rtol=RTOL_DENSE)
    # (7) run to run
    assert np.array_equal(D().find_periods(xb), got)


# ---------------------------------------------------------------- (4) global against shared staging, input layouts
def test_forced_global_vs_shared_and_layouts():
    import torch
    n = 999
    xb = synth.synth_batch(70, n, 11)
    for lo, hi in ((1, 333), (2, 999), (500, 520)):
        chip = _norms(xb, lo, hi, False)
        glob = _norms(xb, lo, hi, True)
        _close(glob, chip, lo, ("global vs shared", lo, hi), rtol=1e-12)
    sig = synth.synth(n + 11 * 100, 5)
    view = np.lib.stride_tricks.sliding_window_view(sig, n)[::100]     # ldx = 100 < N
    want = _norms(np.ascontiguousarray(view), 2, 300)
    for long in (None, True, False):
        assert np.array_equal(_norms(np.ascontiguousarray(view), 2, 300, long),
                              _norms(np.ascontiguousarray(view), 2, 300, long))
        hop = _norms(view, 2, 300, long)
        _close(hop, want, 2, ("hop-framed", long), rtol=1e-12)
    dev = D().find_periods(torch.from_numpy(np.ascontiguousarray(view)).cuda(), 2, 300)
    assert isinstance(dev, torch.Tensor) and dev.is_cuda
    assert np.array_equal(dev.cpu().numpy(), want)
    nc = np.asfortranarray(xb[:9])                                  # non-contiguous host input
    assert np.array_equal(D().find_periods(nc, 2, 300), _norms(xb[:9], 2, 300))
    tcols = torch.from_numpy(xb[:9].T.copy()).cuda().T                # non-contiguous device input
    assert np.array_equal(D().find_periods(tcols, 2, 300).cpu().numpy(), _norms(xb[:9], 2, 300))


# ---------------------------------------------------------------- (5) dispatch at the limit of the on-chip plan
def test_dispatch_at_the_limit(monkeypatch):
    from pyperiod_b200 import _lib
    from pyperiod_b200.periods import smem_optin
    import torch
    lib = _lib.load()
    smem = smem_optin(torch.device("cuda"))
    qmax = 500
    lo, hi = qmax, 1 << 20
    assert _lib.ramanujan_divisor_fits_on_chip(lo, 2, qmax, smem)
    assert not _lib.ramanujan_divisor_fits_on_chip(hi, 2, qmax, smem)
    while hi - lo > 1:                                    # the fit query's own boundary
        mid = (lo + hi) // 2
        if _lib.ramanujan_divisor_fits_on_chip(mid, 2, qmax, smem):
            lo = mid
        else:
            hi = mid
    seen = []
    fn = lib.pp_ramanujan_norms_divisor

    def spy(*args):
        seen.append(int(args[9]))
        return fn(*args)
    monkeypatch.setattr(lib, "pp_ramanujan_norms_divisor", spy)
    for n, staging in ((lo, _lib.STAGING_SHARED), (hi, _lib.STAGING_GLOBAL)):
        x = synth.synth(n, 21)
        seen.clear()
        got = D().find_periods(x, 2, qmax)
        assert seen == [staging], (n, seen)
        _close(got, norms_divisor_form_f64(x, 2, qmax), 2, ("dispatch", n))


# ---------------------------------------------------------------- (6) long windows, (7) run to run
def test_long_16384():
    n = 16384
    x1 = synth.synth(n, 1)
    got1 = D().find_periods(x1)
    assert got1.shape == (n // 3 + 1,)
    _close(got1, norms_divisor_form_f64(x1), 2, "1-D")
    top = norms_closed_form_f64(x1, 5454, 5461)
    _close(got1[5454:], top[5454:], 0, "closed form, top periods")
    xb = synth.synth_batch(3, n, 40)
    gotb = D().find_periods(xb)
    for b in range(3):
        _close(gotb[b], norms_divisor_form_f64(xb[b]), 2, ("batch", b))
    assert np.array_equal(D().find_periods(xb), gotb)
    assert np.array_equal(D().find_periods(x1), got1)


def test_long_131072_large_periods():
    n, lo, hi = 131072, 43680, 43690
    xb = synth.synth_batch(9, n, 70)
    want = [norms_divisor_form_f64(xb[b], lo, hi) for b in range(9)]
    _close(D().find_periods(xb[0], lo, hi), want[0], lo, "B = 1")
    got9 = D().find_periods(xb, lo, hi)
    for b in range(9):
        _close(got9[b], want[b], lo, ("B = 9", b))
    assert np.array_equal(D().find_periods(xb, lo, hi), got9)


def test_long_2_pow_20():
    n = 1 << 20
    x = synth.synth(n, 77)
    for lo, hi in ((2, 200), (349500, 349525)):
        got = D().find_periods(x, lo, hi)
        _close(got, norms_divisor_form_f64(x, lo, hi), lo, (lo, hi))
        assert np.array_equal(D().find_periods(x, lo, hi), got)


def test_omega_7_period():
    q = 510510                       # 2 3 5 7 11 13 17
    n = 3 * q
    x = synth.synth(n, 9)
    got = D().find_periods(x, q, q)
    _close(got, norms_divisor_form_f64(x, q, q, periods=[q]), q, "q = 510510")
    assert np.array_equal(D().find_periods(x, q, q), got)


# ---------------------------------------------------------------- (8) edge cases
def test_edge_cases():
    from pyperiod_b200 import _lib
    n = 4096
    empty = D().find_periods(np.zeros((0, n)))
    assert empty.shape == (0, n // 3 + 1)
    for m in (4096, 16384):
        zero = D().find_periods(np.zeros((3, m)))
        assert zero.shape == (3, m // 3 + 1) and not zero.any()
    x = synth.synth(n, 3)
    one = D().find_periods(x, 97, 97)
    assert np.count_nonzero(one[:97]) == 0 and np.count_nonzero(one) == 1
    _close(one, norms_divisor_form_f64(x, 97, 97), 97, "qmin = qmax")
    for r in (R(), D()):
        with pytest.raises(_lib.PPError):
            r.find_periods(x, 300, 200)
