"""CPU-only checks of the global-memory ("long") path: the fit query that decides the dispatch, argument errors of
the pp_long_* entry points, the staging knob, and the sieve that builds the divisor tables for large pmax."""
import numpy as np
import pytest

SMEM_OPTIN_B200 = 232448   # opt-in shared memory per block of an sm_100 device


@pytest.fixture(scope="module")
def lib():
    from pyperiod_b200 import _lib, build
    build.build()
    return _lib.load()


def test_fit_query_matches_the_on_chip_plans(lib):
    from pyperiod_b200 import _lib
    fits = lambda *a: _lib.fits_on_chip(*a, SMEM_OPTIN_B200)   # noqa: E731
    # config 3 (the headline shape) stays on chip in every fold mode
    for fold in range(4):
        assert fits(_lib.ALGO_MBEST, 4096, 1024, 10, _lib.METRIC_NORM, 0, 0, fold)
    # default max_length = N / 3 just above the on-chip limit
    assert not fits(_lib.ALGO_MBEST, 20000, 6666, 5, _lib.METRIC_NORM, 0, 0, _lib.FOLD_HIERARCHICAL)
    assert fits(_lib.ALGO_MBEST, 12000, 4000, 5, _lib.METRIC_NORM, 0, 0, _lib.FOLD_HIERARCHICAL)
    assert not fits(_lib.ALGO_S2L, 20000, 10000, 0, _lib.METRIC_IMPOSED, 0, 0, _lib.FOLD_DIRECT)
    assert not fits(_lib.ALGO_BCORR, 20000, 6666, 5, _lib.METRIC_MAXABS, 0, 0, _lib.FOLD_HIERARCHICAL)
    assert not fits(_lib.ALGO_PROJECT, 20000, 10000, 0, 0, 0, 0, _lib.FOLD_DIRECT)
    assert fits(_lib.ALGO_PROJECT, 12000, 6000, 0, 0, 0, 0, _lib.FOLD_DIRECT)
    assert not fits(_lib.ALGO_BFREQ, 20000, 0, 0, 0, 0, 0, _lib.FOLD_DIRECT)
    assert fits(_lib.ALGO_BFREQ, 8192, 0, 0, 0, 0, 0, _lib.FOLD_DIRECT)
    # the window alone: no pmax, however small, fits at N = 30 000
    assert not fits(_lib.ALGO_SWEEP, 30000, 2, 0, _lib.METRIC_NORM, 0, 0, _lib.FOLD_DIRECT)
    # monotone in N: the largest fitting M-best window at default max_length
    ok = [n for n in range(13000, 16000, 100) if fits(_lib.ALGO_MBEST, n, n // 3, 5, 0, 0, 0, 0)]
    assert ok == list(range(13000, ok[-1] + 1, 100)) and 13500 < ok[-1] < 15000
    assert lib.pp_fits_on_chip(99, 4096, 1024, 10, 0, 0, 0, 0, SMEM_OPTIN_B200) == -1
    assert lib.pp_fits_on_chip(_lib.ALGO_MBEST, 4096, 1024, 10, 0, 0, 0, 7, SMEM_OPTIN_B200) == -1


def test_long_entry_point_argument_errors_do_not_need_a_gpu(lib):
    rc = lib.pp_long_project(None, 8, 1, 8, 2, 0, None, 0, None, 8, 8, None, 0, None)
    assert rc == -1 and b"null" in lib.pp_last_error()
    rc = lib.pp_long_sweep(None, 8, 1, 8, 2, 4, 0, 0, 0, None, None, 0, None, None, None, None, 0, None)
    assert rc == -1
    dummy = 16   # a non-null "device pointer": the checks below fail before anything is dereferenced
    rc = lib.pp_long_sweep(dummy, 8, 1, 8, 2, 4, 2, 1, 0, None, None, 0, None, dummy, dummy, None, 0, None)
    assert rc == -1 and b"MAXABS" in lib.pp_last_error()
    rc = lib.pp_long_mbest(dummy, 8, 1, 8, 0, 2, 4, 0, 0, 0, None, None, dummy, dummy, 8, dummy, dummy, None, None,
                           None, dummy, None, 0, None)
    assert rc == -1 and b"num" in lib.pp_last_error()
    rc = lib.pp_long_mbest(dummy, 8, 1, 8, 2, 2, 4, 0, 0, 0, None, None, None, None, 8, dummy, dummy, None, None,
                           None, dummy, None, 0, None)
    assert rc == -1 and b"factor tables" in lib.pp_last_error()
    rc = lib.pp_long_small_to_large(dummy, 8, 1, 8, -1.0, 4, 0, 0, None, None, 0, 4, dummy, dummy, None, dummy,
                                    dummy, None, 0, None)
    assert rc == -1 and b"thresh" in lib.pp_last_error()
    rc = lib.pp_long_best_correlation(dummy, 8, 1, 8, 2, 2, 0.01, 0, 0, None, None, 0, dummy, dummy, None, dummy,
                                      None, 0, None)
    assert rc == -1 and b"max_length" in lib.pp_last_error()
    rc = lib.pp_long_best_frequency_round(None, 1, 8, None, 5, 8, 0, 0, None, None, 0, None, None, None, 0, 1,
                                          None, None, 0, None)
    assert rc == -1
    # empty batches are a no-op, as on chip
    assert lib.pp_long_project(None, 8, 0, 8, 2, 0, None, 0, None, 8, 8, None, 0, None) == 0


def test_staging_knob_is_validated():
    from pyperiod_b200 import Periods
    assert Periods(staging="global")._staging == "global"
    assert Periods()._staging == "auto"
    with pytest.raises(ValueError, match="staging"):
        Periods(staging="smem")
    with pytest.raises(ValueError, match="staging"):
        Periods.project(np.arange(10.0), 3, staging="l2")


def test_divisor_sieve_equals_the_per_period_expression():
    from pyperiod_b200 import tables
    lists = tables._nontrivial_factor_lists(1 << 16)
    for p in range(1 << 16):
        assert lists[p] == tables.nontrivial_factors(p), p
    tb = tables.PeriodTables(4096)
    for p in (2, 97, 840, 2730, 4096):
        assert tb.factors_of(p).tolist() == tables.nontrivial_factors(p)
        assert tb.chain_of(p).tolist() == tables.orth_chain(p)
