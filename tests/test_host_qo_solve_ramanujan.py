"""CPU-only checks of the Ramanujan-basis solve stage's fit query (PP_QO_KIND_SOLVE_RAMANUJAN): the on-chip limit it
reports, the arguments it rejects, and the entry points' argument errors, none of which touch a device."""
import pytest

SMEM_OPTIN_B200 = 232448   # opt-in shared memory per block of an sm_100 device


@pytest.fixture(scope="module")
def lib():
    from pyperiod_b200 import _lib, build
    build.build()
    return _lib.load()


def _last_fit(kind, basis, num, rmax):
    from pyperiod_b200 import _lib
    sizes = range(2000, 30001, 50)
    ok = [n for n in sizes if _lib.qo_fits_on_chip(kind, n, n // 3, num, rmax, basis, _lib.FOLD_DIRECT,
                                                   SMEM_OPTIN_B200)]
    assert ok == [n for n in sizes if n <= ok[-1]]   # monotone in N
    return ok[-1]


def test_solve_ramanujan_fit_query_values(lib):
    from pyperiod_b200 import _lib
    K, NAT, RAM = _lib, _lib.BASIS_NATURAL, _lib.BASIS_RAMANUJAN
    assert K.QO_KIND_SOLVE_RAMANUJAN == 3
    ram = _last_fit(K.QO_KIND_SOLVE_RAMANUJAN, RAM, 4, 1024)
    nat = _last_fit(K.QO_KIND_SOLVE, NAT, 4, 1024)
    # the Ramanujan solve holds a second window-sized vector (A^T p of the conjugate gradients) in shared memory
    assert 8000 <= ram <= 9000 and ram < nat
    # config 5's shape fits; the 16 384-sample windows of the global-memory tests do not
    assert _lib.qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 4096, 1365, 4, 1024, RAM, K.FOLD_DIRECT, SMEM_OPTIN_B200)
    assert not _lib.qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 16384, 5461, 4, 1024, RAM, K.FOLD_DIRECT,
                                    SMEM_OPTIN_B200)
    # rmax sizes the weights vector in shared memory: a large one stops fitting first
    assert not _lib.qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 8000, 2666, 4, 8000, RAM, K.FOLD_DIRECT,
                                    SMEM_OPTIN_B200)
    # the fold mode does not enter the solve plan
    for fold in (K.FOLD_HIERARCHICAL, K.FOLD_NOMINATE_F32):
        assert _lib.qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, ram, ram // 3, 4, 1024, RAM, fold, SMEM_OPTIN_B200)
    # windows above 32767 samples never fit on chip
    assert not _lib.qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 40000, 100, 4, 64, RAM, K.FOLD_DIRECT, 1 << 30)


def test_solve_ramanujan_fit_query_rejects_bad_arguments(lib):
    from pyperiod_b200 import _lib
    S, K = SMEM_OPTIN_B200, _lib
    # the natural-basis kind still rejects the Ramanujan basis, and the new kind rejects the natural one
    assert lib.pp_qo_fits_on_chip(K.QO_KIND_SOLVE, 4096, 1024, 4, 1024, K.BASIS_RAMANUJAN, 0, S) == -1
    assert lib.pp_qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 4096, 1024, 4, 1024, K.BASIS_NATURAL, 0, S) == -1
    assert b"PP_BASIS_RAMANUJAN" in lib.pp_last_error()
    assert lib.pp_qo_fits_on_chip(4, 4096, 1024, 4, 1024, K.BASIS_RAMANUJAN, 0, S) == -1
    assert lib.pp_qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 4096, 0, 4, 1024, K.BASIS_RAMANUJAN, 0, S) == -1
    assert lib.pp_qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 4096, 1024, 0, 1024, K.BASIS_RAMANUJAN, 0, S) == -1
    assert lib.pp_qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 4096, 1024, 4, 1, K.BASIS_RAMANUJAN, 0, S) == -1
    assert lib.pp_qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 4096, 1024, 4, 1024, K.BASIS_RAMANUJAN, 9, S) == -1
    with pytest.raises(_lib.PPError):
        _lib.qo_fits_on_chip(K.QO_KIND_SOLVE_RAMANUJAN, 4096, 1024, 4, 1024, K.BASIS_NATURAL, 0, S)
    # the global-memory workspace query answers 0 for the same contradiction and for bad shapes
    assert lib.pp_long_qo_workspace_bytes(K.QO_KIND_SOLVE_RAMANUJAN, 1, 4096, 1365, 4, 1024, K.BASIS_NATURAL, 0) == 0
    assert lib.pp_long_qo_workspace_bytes(K.QO_KIND_SOLVE_RAMANUJAN, 0, 4096, 1365, 4, 1024, K.BASIS_RAMANUJAN, 0) == 0
    assert lib.pp_long_qo_workspace_bytes(K.QO_KIND_SOLVE_RAMANUJAN, 1, 4096, 5000, 4, 1024, K.BASIS_RAMANUJAN, 0) == 0
    assert lib.pp_long_qo_workspace_bytes(4, 1, 4096, 1365, 4, 1024, K.BASIS_RAMANUJAN, 0) == 0


def test_solve_ramanujan_argument_errors_do_not_need_a_gpu(lib):
    d = 16   # a non-null "device pointer": the checks below fail before anything is dereferenced
    for fn in (lib.pp_qo_solve_ramanujan, lib.pp_long_qo_solve_ramanujan):
        rc = fn(d, 8, 1, 8, 2, None, d, 4, 1, d, 8, 32, None, 0, d, d, d, d, d, 32, None, None, d, d, 1 << 20, None)
        assert rc == -1 and b"null" in lib.pp_last_error()
        rc = fn(d, 8, 1, 8, 2, d, d, 4, 1, d, 2, 32, None, 0, d, d, d, d, d, 32, None, None, d, d, 1 << 20, None)
        assert rc == -1 and b"phi" in lib.pp_last_error()
        rc = fn(d, 8, 1, 8, 2, d, d, 9, 1, d, 9, 32, None, 0, d, d, d, d, d, 32, None, None, d, d, 1 << 20, None)
        assert rc == -1 and b"pmax" in lib.pp_last_error()
        rc = fn(d, 8, 1, 8, 2, d, d, 4, 1, d, 8, 1, None, 0, d, d, d, d, d, 32, None, None, d, d, 1 << 20, None)
        assert rc == -1 and b"rmax" in lib.pp_last_error()
        rc = fn(None, 8, 1, 8, 2, d, d, 4, 1, d, 8, 32, None, 0, d, d, d, d, d, 32, None, None, d, d, 1 << 20, None)
        assert rc == -1
        # an empty batch is accepted without looking at anything else
        assert fn(None, 0, 0, 0, 0, None, None, 0, 0, None, 0, 0, None, 0, None, None, None, None, None, 0, None, None,
                  None, None, 0, None) == 0
