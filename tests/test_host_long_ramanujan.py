"""CPU-only checks of the global-memory Ramanujan periodogram: the divisor-form oracle the long-window GPU tests use,
the fit query that decides the dispatch (pp_ramanujan_fits_on_chip) and argument errors of pp_long_ramanujan_norms."""
import numpy as np
import pytest

from divisor_oracle import norms_divisor_form_f64
from oracle.ramanujan import norms_closed_form_f64
from pyperiod_b200 import synth

SMEM_OPTIN_B200 = 232448   # opt-in shared memory per block of an sm_100 device


@pytest.fixture(scope="module")
def lib():
    from pyperiod_b200 import _lib, build
    build.build()
    return _lib.load()


# primes, prime powers and highly composite periods
PERIODS = [2, 3, 4, 7, 8, 9, 12, 16, 25, 27, 32, 36, 48, 60, 64, 97, 120, 125, 128, 180, 199, 240, 243, 256, 331, 360]


@pytest.mark.parametrize("n", [600, 999, 1024, 2000])
def test_divisor_form_equals_closed_form(n):
    x = synth.synth(n, n)
    qs = [q for q in PERIODS if q <= n // 3] + [n // 3]
    got = norms_divisor_form_f64(x, 2, n // 3, periods=qs)
    for q in qs:
        want = norms_closed_form_f64(x, q, q)[q]
        assert abs(got[q] - want) <= 1e-13 * abs(want), (n, q)
    # min_length > 2: the columns below it stay zero
    lo = norms_divisor_form_f64(x, 5, 40)
    assert np.all(lo[:5] == 0)
    np.testing.assert_allclose(lo[5:], norms_closed_form_f64(x, 5, 40)[5:], rtol=1e-13)


def test_fit_query_boundaries(lib):
    from pyperiod_b200 import _lib
    fits = lambda mode, n, qmax, smem=SMEM_OPTIN_B200: _lib.ramanujan_fits_on_chip(mode, n, 2, qmax, smem)  # noqa
    # fp64: the fused kernel keeps S_q[8] and c_q of the largest period; monotone in qmax, independent of N
    ok = [q for q in range(3000, 3400) if fits(_lib.RAM_FP64, 20000, q)]
    assert ok == list(range(3000, ok[-1] + 1)) and ok[-1] == 3200
    assert fits(_lib.RAM_FP64, 9600, 3200) and not fits(_lib.RAM_FP64, 9603, 3201)
    assert not fits(_lib.RAM_FP64, 16384, 16384 // 3)
    # tf32 / f32_compat stage four whole windows: N <= 7264 whatever qmax is
    for mode in (_lib.RAM_TF32, _lib.RAM_F32COMPAT):
        assert fits(mode, 7264, 100) and fits(mode, 7264, 7264 // 3)
        assert not fits(mode, 7265, 100)
    # f32_compat: N <= 32768 however much shared memory there is
    assert fits(_lib.RAM_F32COMPAT, 32768, 10, 1 << 30) and not fits(_lib.RAM_F32COMPAT, 32769, 10, 1 << 30)
    assert fits(_lib.RAM_TF32, 32769, 10, 1 << 30)


def test_fit_query_rejects_bad_arguments(lib):
    S = SMEM_OPTIN_B200
    assert lib.pp_ramanujan_fits_on_chip(3, 4096, 2, 100, S) == -1
    assert lib.pp_ramanujan_fits_on_chip(-1, 4096, 2, 100, S) == -1
    assert lib.pp_ramanujan_fits_on_chip(0, 1, 1, 1, S) == -1
    assert lib.pp_ramanujan_fits_on_chip(0, 4096, 0, 100, S) == -1
    assert lib.pp_ramanujan_fits_on_chip(0, 4096, 200, 100, S) == -1
    assert lib.pp_ramanujan_fits_on_chip(0, 4096, 2, 4097, S) == -1
    assert lib.pp_ramanujan_fits_on_chip(0, 4096, 2, 100, 0) == -1
    from pyperiod_b200 import _lib
    with pytest.raises(_lib.PPError):
        _lib.ramanujan_fits_on_chip(0, 4096, 2, 5000, S)


def test_long_argument_errors_do_not_need_a_gpu(lib):
    d = 16   # a non-null "device pointer": the checks below fail before anything is dereferenced
    ws = lib.pp_long_ramanujan_workspace_bytes(1, 4096, 2, 1365)
    assert ws > 0
    rc = lib.pp_long_ramanujan_norms(d, 4096, 1, 4096, 2, 4097, d, d, 5000, d, 5000, d, ws, None)
    assert rc == -1 and b"qmax <= N" in lib.pp_last_error()
    rc = lib.pp_long_ramanujan_norms(d, 4096, 1, 4096, 0, 100, d, d, 5000, d, 5000, d, ws, None)
    assert rc == -1 and b"qmin" in lib.pp_last_error()
    rc = lib.pp_long_ramanujan_norms(d, 4096, 1, 4096, 2, 1365, None, d, 1365, d, 1366, d, ws, None)
    assert rc == -1 and b"tables" in lib.pp_last_error()
    rc = lib.pp_long_ramanujan_norms(d, 4096, 1, 4096, 2, 1365, d, d, 1000, d, 1366, d, ws, None)
    assert rc == -1 and b"tables" in lib.pp_last_error()
    rc = lib.pp_long_ramanujan_norms(d, 4096, 1, 4096, 2, 1365, d, d, 1365, d, 1365, d, ws, None)
    assert rc == -1 and b"leading dimension" in lib.pp_last_error()
    rc = lib.pp_long_ramanujan_norms(None, 4096, 1, 4096, 2, 1365, d, d, 1365, d, 1366, d, ws, None)
    assert rc == -1
    rc = lib.pp_long_ramanujan_norms(d, 0, 1, 4096, 2, 1365, d, d, 1365, d, 1366, d, ws, None)
    assert rc == -1
    rc = lib.pp_long_ramanujan_norms(d, 4096, 1, 4096, 2, 1365, d, d, 1365, d, 1366, d, 4096, None)
    assert rc == -3 and b"workspace" in lib.pp_last_error()
    rc = lib.pp_long_ramanujan_norms(d, 4096, 1, 4096, 2, 1365, d, d, 1365, d, 1366, None, ws, None)
    assert rc == -3
    # empty batches are accepted without looking at anything else
    assert lib.pp_long_ramanujan_norms(None, 0, 0, 0, 0, 0, None, None, 0, None, 0, None, 0, None) == 0
    assert lib.pp_long_ramanujan_workspace_bytes(1, 4096, 2, 4097) == 0
    assert lib.pp_long_ramanujan_workspace_bytes(1, 4096, 0, 100) == 0
    # the workspace does not grow with qmax^2: 64 MB of folds and Ramanujan sums (plus partial norms) at any N
    assert lib.pp_long_ramanujan_workspace_bytes(1, 1 << 20, 2, (1 << 20) // 3) < (80 << 20)
    assert lib.pp_long_ramanujan_workspace_bytes(64, 131072, 2, 43690) < (80 << 20)
