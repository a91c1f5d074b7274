"""CPU-only checks of the divisor-form Ramanujan periodogram (csrc/pp_ram_divisor.cu): the smallest-prime-factor
table, a numpy emulation of the kernels' algorithm against the divisor-form oracle, the fit query, argument errors
and the workspace bound of pp_ramanujan_norms_divisor, and the constructor's checks of `method`."""
import numpy as np
import pytest

from divisor_oracle import norms_divisor_form_f64
from oracle.numtheory import phi
from pyperiod_b200 import synth
from pyperiod_b200.tables import smallest_prime_factor_table

SMEM_OPTIN_B200 = 232448   # opt-in shared memory per block of an sm_100 device

# primes, prime powers and highly composite periods (the list of the long-path host tests), plus q = 1 and
# omega(q) = 6 and 7
PERIODS = [2, 3, 4, 7, 8, 9, 12, 16, 25, 27, 32, 36, 48, 60, 64, 97, 120, 125, 128, 180, 199, 240, 243, 256, 331, 360]
EXTRA = [1, 30030, 510510]


@pytest.fixture(scope="module")
def lib():
    from pyperiod_b200 import _lib, build
    build.build()
    return _lib.load()


def _trial_spf(q):
    if q < 2:
        return q
    p = 2
    while p * p <= q:
        if q % p == 0:
            return p
        p += 1
    return q


def test_spf_against_trial_division():
    spf = smallest_prime_factor_table(100_000)
    assert spf.dtype == np.int32 and spf[0] == 0 and spf[1] == 1
    assert all(int(spf[q]) == _trial_spf(q) for q in range(100_001))
    big = smallest_prime_factor_table(1 << 20)
    rng = np.random.default_rng(5)
    for q in list(rng.integers(100_001, 1 << 20, 2000)) + [(1 << 20), 510510, 1048573, 999983 * 1]:
        assert int(big[q]) == _trial_spf(int(q)), q


def test_tables_expose_spf():
    from pyperiod_b200.tables import PeriodTables
    tb = PeriodTables(5000)
    assert np.array_equal(tb.spf, smallest_prime_factor_table(5000))


def _emulate(x, q, spf):
    """The kernels' algorithm for one period: fold, the comb factors in spf order, the count-weighted energy."""
    n = len(x)
    idx = np.arange(n)
    v = np.bincount(idx % q, weights=x, minlength=q)
    cnt = np.bincount(idx % q, minlength=q).astype(np.float64)
    t, rad = q, 1
    while t > 1:
        p = int(spf[t])
        qp = q // p
        c = v.reshape(p, qp).sum(0)
        v = p * v - np.tile(c, p)
        rad *= p
        while t % p == 0:
            t //= p
    z = (q // rad) * v
    ph = float(phi(q))
    s = q / (ph * ph)
    return s * s * np.sum(cnt * z * z)


def test_emulation_equals_divisor_oracle():
    spf = smallest_prime_factor_table(510510)
    for q in PERIODS + EXTRA:
        n = max(3 * q + 7, 1000)
        x = synth.synth(n, q)
        want = norms_divisor_form_f64(x, q, q, periods=[q])[q]
        got = _emulate(x, q, spf)
        assert abs(got - want) <= 1e-13 * abs(want), (q, got, want)


def test_fit_query(lib):
    from pyperiod_b200 import _lib
    fits = lambda n, qmax, smem=SMEM_OPTIN_B200: _lib.ramanujan_divisor_fits_on_chip(n, 2, qmax, smem)  # noqa
    assert fits(4096, 1365)                                  # config 5
    # monotone in qmax at fixed N, and in N at fixed qmax
    ok_q = [fits(8000, q) for q in range(2, 8001, 7)]
    assert ok_q == sorted(ok_q, reverse=True) and ok_q[0] and not ok_q[-1]
    ok_n = [fits(n, 500) for n in range(500, 40000, 97)]
    assert ok_n == sorted(ok_n, reverse=True) and ok_n[0] and not ok_n[-1]
    assert not fits(1 << 20, 2)
    assert fits(4096, 1365, 1 << 30)


def test_fit_query_rejects_bad_arguments(lib):
    S = SMEM_OPTIN_B200
    assert lib.pp_ramanujan_divisor_fits_on_chip(1, 1, 1, S) == -1
    assert lib.pp_ramanujan_divisor_fits_on_chip(4096, 0, 100, S) == -1
    assert lib.pp_ramanujan_divisor_fits_on_chip(4096, 200, 100, S) == -1
    assert lib.pp_ramanujan_divisor_fits_on_chip(4096, 2, 4097, S) == -1
    assert lib.pp_ramanujan_divisor_fits_on_chip(4096, 2, 100, 0) == -1
    from pyperiod_b200 import _lib
    with pytest.raises(_lib.PPError):
        _lib.ramanujan_divisor_fits_on_chip(4096, 2, 5000, S)


def test_argument_errors_do_not_need_a_gpu(lib):
    d = 16   # a non-null "device pointer": the checks below fail before anything is dereferenced
    ws = lib.pp_ramanujan_divisor_workspace_bytes(1, 4096, 2, 1365)
    assert ws > 0
    f = lib.pp_ramanujan_norms_divisor
    rc = f(d, 4096, 1, 4096, 2, 4097, d, d, 5000, 0, d, 5000, d, ws, None)
    assert rc == -1 and b"qmax <= N" in lib.pp_last_error()
    rc = f(d, 4096, 1, 4096, 0, 100, d, d, 5000, 0, d, 5000, d, ws, None)
    assert rc == -1 and b"qmin" in lib.pp_last_error()
    rc = f(d, 4096, 1, 4096, 200, 100, d, d, 5000, 0, d, 5000, d, ws, None)
    assert rc == -1 and b"qmin" in lib.pp_last_error()
    rc = f(d, 4096, 1, 4096, 2, 1365, None, d, 1365, 0, d, 1366, d, ws, None)
    assert rc == -1 and b"tables" in lib.pp_last_error()
    rc = f(d, 4096, 1, 4096, 2, 1365, d, d, 1000, 0, d, 1366, d, ws, None)
    assert rc == -1 and b"tables" in lib.pp_last_error()
    rc = f(d, 4096, 1, 4096, 2, 1365, d, d, 1365, 0, d, 1365, d, ws, None)
    assert rc == -1 and b"leading dimension" in lib.pp_last_error()
    rc = f(None, 4096, 1, 4096, 2, 1365, d, d, 1365, 0, d, 1366, d, ws, None)
    assert rc == -1
    rc = f(d, 0, 1, 4096, 2, 1365, d, d, 1365, 0, d, 1366, d, ws, None)
    assert rc == -1
    rc = f(d, 4096, 1, 4096, 2, 1365, d, d, 1365, 3, d, 1366, d, ws, None)
    assert rc == -1 and b"staging" in lib.pp_last_error()
    rc = f(d, 4096, 1, 4096, 2, 1365, d, d, 1365, 0, d, 1366, d, 16, None)
    assert rc == -3 and b"workspace" in lib.pp_last_error()
    rc = f(d, 4096, 1, 4096, 2, 1365, d, d, 1365, 0, d, 1366, None, ws, None)
    assert rc == -3
    big = lib.pp_ramanujan_divisor_workspace_bytes(1, 1 << 20, 2, 100_000)
    rc = f(d, 1 << 20, 1, 1 << 20, 2, 100_000, d, d, 100_000, 2, d, 100_001, d, 4096, None)
    assert rc == -3 and big > 4096
    # empty batches are accepted without looking at anything else
    assert f(None, 0, 0, 0, 0, 0, None, None, 0, 7, None, 0, None, 0, None) == 0
    assert lib.pp_ramanujan_divisor_workspace_bytes(1, 4096, 2, 4097) == 0
    assert lib.pp_ramanujan_divisor_workspace_bytes(1, 4096, 0, 100) == 0
    assert lib.pp_ramanujan_divisor_workspace_bytes(-1, 4096, 2, 100) == 0


def test_workspace_bound(lib):
    # include/pyperiod_b200.h: at most 256 + 296 * 8 * (qmax + ceil(qmax / 2) + 2) bytes, whatever B and N
    for b, n in ((1, 1 << 20), (64, 1 << 20), (8, 131072), (65536, 4096)):
        for qmax in (n // 3, min(n, 9000), 1365):
            got = lib.pp_ramanujan_divisor_workspace_bytes(b, n, 2, qmax)
            assert 256 <= got <= 256 + 296 * 8 * (qmax + (qmax + 1) // 2 + 2), (b, n, qmax)
    # and does not depend on B or N
    assert (lib.pp_ramanujan_divisor_workspace_bytes(1, 1 << 20, 2, 349525)
            == lib.pp_ramanujan_divisor_workspace_bytes(64, 1 << 21, 2, 349525))


def test_constructor_rejects_bad_method():
    # raised before any device is touched: these run without a GPU
    from pyperiod_b200 import RamanujanPeriods
    with pytest.raises(ValueError, match="method"):
        RamanujanPeriods(method="fft")
    for prec in ("tf32", "f32_compat"):
        with pytest.raises(ValueError, match="fp64"):
            RamanujanPeriods(method="divisor", precision=prec)
