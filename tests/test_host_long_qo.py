"""CPU-only checks of the global-memory path of QOPeriods and the Muresan finder: the fit query that decides the
dispatch (pp_qo_fits_on_chip), the capacity of the long step, argument errors of the pp_long_qo_* entry points and
the staging knob."""
import pytest

SMEM_OPTIN_B200 = 232448   # opt-in shared memory per block of an sm_100 device


@pytest.fixture(scope="module")
def lib():
    from pyperiod_b200 import _lib, build
    build.build()
    return _lib.load()


def _last_fit(kind, sizes, pmax_of, num, rmax, basis, fold):
    from pyperiod_b200 import _lib
    ok = [n for n in sizes if _lib.qo_fits_on_chip(kind, n, pmax_of(n), num, rmax, basis, fold, SMEM_OPTIN_B200)]
    assert ok == [n for n in sizes if n <= ok[-1]]   # monotone in N
    return ok[-1]


def test_qo_fit_query_boundaries(lib):
    from pyperiod_b200 import _lib
    K, NAT, RAM = _lib, _lib.BASIS_NATURAL, _lib.BASIS_RAMANUJAN
    sizes = range(8000, 30001, 50)
    # find, hierarchical fold, first launch (rmax 3072) and direct fold (rmax 1024), default max_length = N / 3
    hier = _last_fit(K.QO_KIND_FIND, sizes, lambda n: n // 3, 4, 3072, NAT, K.FOLD_HIERARCHICAL)
    direct = _last_fit(K.QO_KIND_FIND, sizes, lambda n: n // 3, 4, 1024, NAT, K.FOLD_DIRECT)
    assert 9900 <= hier <= 10300 and 12000 <= direct <= 13000
    # the re-run of a window whose dictionary outgrew the first launch (rmax grows towards N) stops fitting first
    assert not _lib.qo_fits_on_chip(K.QO_KIND_FIND, 9000, 3000, 4, 9000, NAT, K.FOLD_HIERARCHICAL, SMEM_OPTIN_B200)
    assert _lib.qo_fits_on_chip(K.QO_KIND_FIND, 9000, 3000, 4, 3072, NAT, K.FOLD_HIERARCHICAL, SMEM_OPTIN_B200)
    # Ramanujan basis: its second window-sized vector lowers the limit
    ram = _last_fit(K.QO_KIND_FIND, sizes, lambda n: n // 3, 4, 1024, RAM, K.FOLD_DIRECT)
    assert ram < direct
    # solve stage: the window is read in place only when that makes room for two CTAs per SM
    solve = _last_fit(K.QO_KIND_SOLVE, sizes, lambda n: n // 3, 32, 1024, NAT, K.FOLD_DIRECT)
    assert 12000 <= solve <= 14500
    # Muresan, default max_p = N / 2
    mur = _last_fit(K.QO_KIND_MURESAN, sizes, lambda n: n // 2, 1, 2, NAT, K.FOLD_DIRECT)
    assert 14000 <= mur <= 14600
    # the exact byte count: one byte less than the plan does not fit
    for n in (hier, hier + 50):
        fits = _lib.qo_fits_on_chip(K.QO_KIND_FIND, n, n // 3, 4, 3072, NAT, K.FOLD_HIERARCHICAL, SMEM_OPTIN_B200)
        assert fits == (n == hier)
    # the on-chip launches reject windows above 32767 samples however small the plan
    assert not _lib.qo_fits_on_chip(K.QO_KIND_FIND, 40000, 100, 4, 64, NAT, K.FOLD_DIRECT, 1 << 30)
    assert _lib.qo_fits_on_chip(K.QO_KIND_MURESAN, 40000, 100, 1, 2, NAT, K.FOLD_DIRECT, 1 << 30)


def test_qo_fit_query_rejects_bad_arguments(lib):
    from pyperiod_b200 import _lib
    S = SMEM_OPTIN_B200
    assert lib.pp_qo_fits_on_chip(7, 4096, 1024, 4, 1024, 0, 0, S) == -1
    assert lib.pp_qo_fits_on_chip(_lib.QO_KIND_FIND, 4096, 1024, 4, 1024, 5, 0, S) == -1
    assert lib.pp_qo_fits_on_chip(_lib.QO_KIND_FIND, 4096, 1024, 4, 1024, 0, 9, S) == -1
    assert lib.pp_qo_fits_on_chip(_lib.QO_KIND_FIND, 1, 1024, 4, 1024, 0, 0, S) == -1
    assert lib.pp_qo_fits_on_chip(_lib.QO_KIND_SOLVE, 4096, 1024, 4, 1024, _lib.BASIS_RAMANUJAN, 0, S) == -1
    with pytest.raises(_lib.PPError):
        _lib.qo_fits_on_chip(_lib.QO_KIND_FIND, 4096, 0, 4, 1024, 0, 0, S)


def test_long_capacity(lib):
    from pyperiod_b200 import _lib
    cap = _lib.long_qo_max_rows(SMEM_OPTIN_B200)
    assert cap % 32 == 0 and 20000 <= cap <= 29000
    assert _lib.long_qo_max_rows(1024) == 0


def test_long_qo_argument_errors_do_not_need_a_gpu(lib):
    d = 16   # a non-null "device pointer": the checks below fail before anything is dereferenced
    rc = lib.pp_long_qo_find_periods(None, 8, 1, 8, 2, 0.1, 2, 4, 0, 1, 0, d, 8, 32, d, d, d, d, d, d, d, d, 32, None,
                                     d, d, 1 << 20, None)
    assert rc == -1 and b"null" in lib.pp_last_error()
    rc = lib.pp_long_qo_find_periods(d, 8, 1, 8, 65, 0.1, 2, 4, 0, 1, 0, d, 8, 32, d, d, d, d, d, d, d, d, 32, None,
                                     d, d, 1 << 20, None)
    assert rc == -1 and b"num" in lib.pp_last_error()
    rc = lib.pp_long_qo_find_periods(d, 8, 1, 8, 2, 0.1, 2, 9, 0, 1, 0, d, 9, 32, d, d, d, d, d, d, d, d, 32, None,
                                     d, d, 1 << 20, None)
    assert rc == -1 and b"pmax" in lib.pp_last_error()
    rc = lib.pp_long_qo_find_periods(d, 8, 1, 8, 2, 0.1, 2, 4, 0, 7, 0, d, 8, 32, d, d, d, d, d, d, d, d, 32, None,
                                     d, d, 1 << 20, None)
    assert rc == -1 and b"refine" in lib.pp_last_error()
    rc = lib.pp_long_qo_find_periods(d, 8, 1, 8, 2, 0.1, 2, 4, 0, 1, 3, d, 8, 32, d, d, d, d, d, d, d, d, 32, None,
                                     d, d, 1 << 20, None)
    assert rc == -1 and b"basis" in lib.pp_last_error()
    rc = lib.pp_long_qo_find_periods(d, 8, 1, 8, 2, 0.1, 2, 4, 0, 1, 0, d, 8, 32, None, d, d, d, d, d, d, d, 32, None,
                                     d, d, 1 << 20, None)
    assert rc == -1 and b"null" in lib.pp_last_error()
    rc = lib.pp_long_qo_solve(d, 8, 1, 8, 2, None, d, 4, 1, d, 8, 32, None, 0, d, d, d, d, d, 32, None, None, d, d,
                              1 << 20, None)
    assert rc == -1 and b"null" in lib.pp_last_error()
    rc = lib.pp_long_qo_solve(d, 8, 1, 8, 2, d, d, 4, 1, d, 2, 32, None, 0, d, d, d, d, d, 32, None, None, d, d,
                              1 << 20, None)
    assert rc == -1 and b"phi" in lib.pp_last_error()
    rc = lib.pp_long_qo_solve_rows(d, 8, 1, 8, 2, d, d, d, 4, 1, 1, d, d, 32, None, d, d, 1 << 20, None)
    assert rc == -1 and b"rmax" in lib.pp_last_error()
    rc = lib.pp_long_muresan_powers(d, 8, 1, 8, 9, 0, d, 8, None, None, d, d, 1 << 20, None)
    assert rc == -1 and b"max_p" in lib.pp_last_error()
    rc = lib.pp_long_muresan_powers(None, 8, 1, 8, 4, 0, d, 8, None, None, d, d, 1 << 20, None)
    assert rc == -1
    # empty batches are accepted without looking at anything else
    assert lib.pp_long_qo_find_periods(None, 0, 0, 0, 0, 0.0, 0, 0, 0, 0, 0, None, 0, 0, None, None, None, None, None,
                                       None, None, None, 0, None, None, None, 0, None) == 0
    assert lib.pp_long_muresan_powers(None, 0, 0, 0, 0, 0, None, 0, None, None, None, None, 0, None) == 0
    assert lib.pp_long_qo_workspace_bytes(9, 1, 4096, 1024, 4, 1024, 0, 0) == 0
    assert lib.pp_long_qo_workspace_bytes(0, 1, 4096, 5000, 4, 1024, 0, 0) == 0


def test_staging_knob_is_checked():
    from pyperiod_b200 import QOPeriods, QOPeriodsWithGCDsExtracted, RamanujanPeriods
    for cls in (QOPeriods, QOPeriodsWithGCDsExtracted, RamanujanPeriods):
        for bad in ("l2", "", None, "GLOBAL"):
            with pytest.raises(ValueError):
                cls(staging=bad)
        for ok in ("auto", "shared", "global"):
            assert cls(staging=ok)._staging == ok
