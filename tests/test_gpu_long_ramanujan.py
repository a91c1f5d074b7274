"""GPU tests of the global-memory ("long") fp64 Ramanujan periodogram (csrc/pp_long_ram.cu).

(1) the long path forced on windows that fit on chip, against the fp64 closed form and the on-chip path; (2) the
dispatch at the limit of the on-chip plan; (3)-(5) windows above that limit against the divisor form of the
periodogram; (6) run-to-run and edge cases; (7) the other precisions keep their limits.
"""
import numpy as np
import pytest

from divisor_oracle import norms_divisor_form_f64
from oracle import qo as oq
from oracle import ramanujan as oram
from pyperiod_b200 import synth

pytestmark = pytest.mark.gpu

RTOL = 1e-11   # the on-chip bar of test_norms_vs_fp64_closed_form


def R(**kw):
    from pyperiod_b200 import RamanujanPeriods
    return RamanujanPeriods(**kw)


def _norms(x, lo, hi, long):
    import torch
    from pyperiod_b200._device import stage_windows
    r = R()
    w = stage_windows(x, r._device)
    out = r._norms_device(w, lo, hi, _long=long)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _close(got, want, lo, what):
    assert np.all(got[..., :lo] == 0), what
    err = np.abs(got[..., lo:] - want[..., lo:])
    bad = err > RTOL * np.abs(want[..., lo:])
    assert not bad.any(), (what, np.argwhere(bad)[:5], float((err / np.abs(want[..., lo:])).max()))


# ---------------------------------------------------------------- (1) forced long path on windows that fit
def test_forced_long_matches_closed_form_and_on_chip():
    n, lo, hi = 999, 3, 333
    xb = synth.synth_batch(70, n, 11)
    chip = _norms(xb, lo, hi, False)
    for b in (1, 5, 8, 9, 70):                      # lone windows (shift form), one full group, both, many
        got = _norms(xb[:b], lo, hi, True)
        assert got.shape == (b, hi + 1)
        _close(got, chip[:b], lo, ("on chip", b))
        for i in sorted({0, b - 1}):
            _close(got[i], oram.norms_closed_form_f64(xb[i], lo, hi), lo, ("closed form", b, i))
    x = synth.synth(1024, 50_000)                   # 1-D, default periods
    got = _norms(x, 2, 1024 // 3, True)[0]
    _close(got, oram.norms_closed_form_f64(x, 2, None), 2, "1-D")


def test_forced_long_hop_framed_and_device_inputs():
    import torch
    n = 999
    sig = synth.synth(n + 11 * 100, 5)
    view = np.lib.stride_tricks.sliding_window_view(sig, n)[::100]     # ldx = 100 < N
    assert view.shape[0] == 12
    got = _norms(view, 2, 300, True)
    want = _norms(np.ascontiguousarray(view), 2, 300, True)
    assert np.array_equal(got, want)
    dev = _norms(torch.from_numpy(np.ascontiguousarray(view)).cuda(), 2, 300, True)
    assert np.array_equal(dev, want)
    _close(got, _norms(view, 2, 300, False), 2, "hop-framed vs on chip")


# ---------------------------------------------------------------- (2) dispatch at the limit of the on-chip plan
def _spy(monkeypatch):
    from pyperiod_b200 import _lib
    lib = _lib.load()
    calls = []
    for name in ("pp_ramanujan_norms", "pp_long_ramanujan_norms"):
        fn = getattr(lib, name)

        def spy(*args, _fn=fn, _name=name):
            calls.append(_name)
            return _fn(*args)
        monkeypatch.setattr(lib, name, spy)
    return calls


def test_dispatch_at_the_limit(monkeypatch):
    n = 9600
    x = synth.synth(n, 21)
    direct = _norms(x, 2, 3200, False)[0]
    calls = _spy(monkeypatch)
    at = R().find_periods(x, 2, 3200)
    assert calls == ["pp_ramanujan_norms"]
    assert np.array_equal(at, direct)
    calls.clear()
    above = R().find_periods(x, 2, 3201)
    assert calls == ["pp_long_ramanujan_norms"]
    _close(above, norms_divisor_form_f64(x, 2, 3201), 2, "max_length 3201")


# ---------------------------------------------------------------- (3) above the limit
def test_auto_above_the_limit():
    n = 16384
    x1 = synth.synth(n, 1)
    got1 = R().find_periods(x1)
    assert got1.shape == (n // 3 + 1,)
    _close(got1, norms_divisor_form_f64(x1), 2, "1-D")
    top = oram.norms_closed_form_f64(x1, 5454, 5461)
    _close(got1[5454:], top[5454:], 0, "dense closed form, top periods")
    xb = synth.synth_batch(3, n, 40)
    gotb = R().find_periods(xb)
    for b in range(3):
        _close(gotb[b], norms_divisor_form_f64(xb[b]), 2, ("batch", b))
    # (6) run to run: bit-identical
    assert np.array_equal(R().find_periods(xb), gotb)
    assert np.array_equal(R().find_periods(x1), got1)


# ---------------------------------------------------------------- (4) large periods
def test_large_periods():
    n, lo, hi = 131072, 43680, 43690
    xb = synth.synth_batch(9, n, 70)
    want = [norms_divisor_form_f64(xb[b], lo, hi) for b in range(9)]
    got1 = R().find_periods(xb[0], lo, hi)
    _close(got1, want[0], lo, "B = 1")
    got9 = R().find_periods(xb, lo, hi)
    for b in range(9):
        _close(got9[b], want[b], lo, ("B = 9", b))


# ---------------------------------------------------------------- (5) find_periods_with_weights above the limit
def test_weights_above_the_limit():
    n, thresh = 16384, 0.2
    x = synth.synth(n, 2)
    norms = norms_divisor_form_f64(x)
    ratio = norms / np.abs(norms.max())
    assert np.min(np.abs(ratio - thresh)) > 1e-9      # no period sits on the threshold
    want = np.argwhere(ratio > thresh).flatten()
    d, r = R().find_periods_with_weights(x)
    assert np.array_equal(np.asarray(d["periods"]), want)
    _close(np.asarray(d["norms"]), norms[want], 0, "selected norms")
    a, _ = oq.get_subspaces([int(p) for p in want], n)
    w, recon = oq.solve_quadratic(x, a)
    np.testing.assert_allclose(d["weights"], w, rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(r, x - recon, rtol=0, atol=1e-11)


# ---------------------------------------------------------------- (6) edge cases
def test_edge_cases():
    n = 16384
    empty = R().find_periods(np.zeros((0, n)))
    assert empty.shape == (0, n // 3 + 1)
    zero = R().find_periods(np.zeros(n))
    assert zero.shape == (n // 3 + 1,) and not zero.any()


# ---------------------------------------------------------------- (7) the other precisions keep their limits
def test_other_precisions_still_raise():
    from pyperiod_b200 import _lib
    x = synth.synth(8000, 4)
    for prec in ("tf32", "f32_compat"):
        with pytest.raises(_lib.PPError):
            R(precision=prec).find_periods(x)
