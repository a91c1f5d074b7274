"""The default plain M-best (Periods() without fold_mode, neither trunc nor orth) ranks with the fp32 nomination
sweep.  It must select what the fp64 hierarchy selects: period lists, status, sweep counts and near-tie counts equal,
powers to the last bits (the winner's value comes from the sequential fp64 fold instead of the hierarchical sums),
bases bit for bit."""
import numpy as np
import pytest

from conftest import load_golden, sha, tie_inputs
from pyperiod_b200 import synth

pytestmark = pytest.mark.gpu

POWER_RTOL = 1e-14


@pytest.fixture(scope="module")
def P():
    from pyperiod_b200 import Periods
    return Periods


@pytest.fixture(autouse=True)
def no_module_fold_mode():
    """The default call is the one without any fold mode named (other suites leave one set module-wide)."""
    from pyperiod_b200 import _lib
    saved = _lib._module_fold_mode
    _lib.set_fold_mode(None)
    yield
    _lib._module_fold_mode = saved


def _np(t):
    return t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)


def _assert_same_selection(a, b, what):
    for field in ("periods", "status", "sweeps", "near_ties"):
        assert np.array_equal(_np(getattr(a, field)), _np(getattr(b, field))), (what, field)
    np.testing.assert_allclose(_np(a.powers), _np(b.powers), rtol=POWER_RTOL, atol=0, err_msg=str(what))


def _bench_windows(b):
    import torch
    stream = synth.synth_stream(b)   # hop-framed: 4 096-sample windows every 512 samples, as bench.py runs them
    return torch.as_strided(torch.from_numpy(stream).cuda(), (b, 4096), (512, 1))


@pytest.mark.parametrize("max_length", [64, 500, 1024])
def test_default_mbest_matches_the_fp64_hierarchy(P, max_length):
    hop = _bench_windows(2048)
    flat = synth.synth_batch(1024, 4096, 9_100 + max_length)
    hier = P(fold_mode="hierarchical")
    for name in ("m_best", "m_best_gamma"):
        for tag, x in (("hop", hop), ("flat", flat)):
            a = getattr(P(), name)(x, num=10, max_length=max_length)
            b = getattr(hier, name)(x, num=10, max_length=max_length)
            _assert_same_selection(a, b, (name, tag, max_length))


def test_default_mbest_bases_are_the_fp64_bases(P):
    x = synth.synth_batch(64, 4096, 9_200)
    for name in ("m_best", "m_best_gamma"):
        a = getattr(P(), name)(x, num=10, max_length=1024, return_bases=True)
        b = getattr(P(fold_mode="hierarchical"), name)(x, num=10, max_length=1024, return_bases=True)
        _assert_same_selection(a, b, name)
        assert np.array_equal(_np(a.bases), _np(b.bases)), name


def test_default_mbest_matches_direct_folds(P):
    """The inputs the fp32 option is pinned on against the all-fp64 direct sweep, through the default call."""
    win = _bench_windows(192)
    small = synth.synth_batch(16, 1000, 4711)
    odd = synth.synth_batch(12, 3001, 4712)
    calls = (("m", "m_best", win, dict(num=10, max_length=1024)),
             ("g", "m_best_gamma", win, dict(num=10, max_length=1024)),
             ("s", "m_best", small, dict(num=5)),
             ("o", "m_best_gamma", odd, dict(num=6, min_length=3, max_length=999)))
    for k, name, x, kw in calls:
        a = getattr(P(fold_mode="direct"), name)(x, **kw)
        b = getattr(P(), name)(x, **kw)
        assert np.array_equal(_np(a.periods), _np(b.periods)), k
        assert np.array_equal(_np(a.sweeps), _np(b.sweeps)), k
        np.testing.assert_allclose(_np(b.powers), _np(a.powers), rtol=1e-12)


def test_default_mbest_large_dynamic_range(P):
    """Windows whose float fold could overflow (N sum x^2 above 2^120) rank with the fp64 hierarchy; samples spread
    over many decades, down to float subnormals and below, still nominate exactly."""
    rng = np.random.default_rng(9_300)
    x = synth.synth_batch(8, 4096, 9_301)
    x[0] *= 1e20                                                      # beyond the float range of the fold
    x[1] *= 1e15                                                      # within it
    x[2] *= 10.0 ** rng.uniform(-50, 12, 4096)                        # decades apart, subnormal in float
    x[3] = np.where(np.arange(4096) % 7 == 0, 1e-42, x[3] * 1e-30)    # tiny everywhere
    tail = np.arange(4096) >= 4096 - 4096 % 241                       # the partial last row of p = 241 ...
    x[4][tail] *= 1e6                                                 # ... carries most of the energy
    for name in ("m_best", "m_best_gamma"):
        a = getattr(P(), name)(x, num=10, max_length=1024)
        b = getattr(P(fold_mode="hierarchical"), name)(x, num=10, max_length=1024)
        _assert_same_selection(a, b, name)


def test_default_mbest_exact_ties_vs_reference_fixture(P):
    """tests/golden/ties.npz (generated from the reference) through the default call."""
    g = load_golden("ties")
    inputs = tie_inputs()
    names = sorted(inputs)
    xb = np.stack([inputs[k] for k in names])
    for tag, gamma in (("norm", False), ("gamma", True)):
        res = (P().m_best_gamma if gamma else P().m_best)(xb, num=1, max_length=1024, return_bases=True)
        ref = (P(fold_mode="hierarchical").m_best_gamma if gamma else
               P(fold_mode="hierarchical").m_best)(xb, num=1, max_length=1024, return_bases=True)
        assert res.status.tolist() == [0] * len(names)
        assert np.array_equal(res.near_ties, ref.near_ties)
        for i, k in enumerate(names):
            assert int(res.periods[i, 0]) == int(g[f"{k}_{tag}_period"][0]), (tag, k, res.periods[i])
            np.testing.assert_allclose(res.powers[i, 0], g[f"{k}_{tag}_power"][0], rtol=1e-12)
            assert sha(res.bases[i]) == str(g[f"{k}_{tag}_base_sha"]), (tag, k)


def test_default_mbest_without_room_for_the_float_copies(P):
    """A window whose fp64 plan fits on chip but whose float copies do not keeps the on-chip fp64 hierarchy, also
    with staging="shared"."""
    from pyperiod_b200 import _lib
    from pyperiod_b200.periods import smem_optin
    import torch
    n = 13_000
    smem = smem_optin(torch.device("cuda", 0))
    args = (_lib.ALGO_MBEST, n, 1024, 10, _lib.METRIC_NORM, 0, 0)
    assert _lib.fits_on_chip(*args, _lib.FOLD_HIERARCHICAL, smem)
    assert not _lib.fits_on_chip(*args, _lib.FOLD_NOMINATE_F32, smem)
    x = synth.synth_batch(4, n, 9_400)
    for staging in ("auto", "shared"):
        a = P(staging=staging).m_best(x, num=10, max_length=1024)
        b = P(fold_mode="hierarchical", staging=staging).m_best(x, num=10, max_length=1024)
        for field in ("periods", "status", "sweeps", "near_ties", "powers"):
            assert np.array_equal(_np(getattr(a, field)), _np(getattr(b, field))), (staging, field)
