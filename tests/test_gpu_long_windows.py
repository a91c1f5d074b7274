"""GPU tests of the global-memory ("long") path of the `Periods` family.

Three groups: (1) the path forced on short windows (staging="global") against the same fixtures and bars as the
on-chip tests; (2) windows whose on-chip plan does not fit (staging="auto" dispatches them to the long path) against
the oracle; (3) batch behaviour: pieces, hop-framed views, device tensors, determinism and edge cases.
Bars: project() and bases bit-exact where the on-chip tests assert it, period lists exact, powers <= 1e-10.
"""
import warnings

import numpy as np
import pytest

from conftest import load_golden, sha, tie_inputs
from oracle import periods as op
from pyperiod_b200 import synth

pytestmark = pytest.mark.gpu

RTOL = 1e-10


@pytest.fixture(scope="module")
def P():
    from pyperiod_b200 import Periods
    return Periods


def G(*args, **kw):
    from pyperiod_b200 import Periods
    return Periods(*args, staging="global", **kw)


def _quiet():
    w = warnings.catch_warnings()
    w.__enter__()
    warnings.simplefilter("ignore")
    return w


# ---------------------------------------------------------------- (1) forced long path on short windows
def test_global_project_golden_bit_exact(P):
    g = load_golden("project")
    cache = {}
    for key in g["cases"]:
        n, seed, p, mode = str(key).split("_")
        n, seed, p = int(n), int(seed), int(p)
        x = cache.setdefault((n, seed), synth.synth(n, seed))
        y = P.project(x, p, mode[0] == "1", mode[1] == "1", staging="global")
        assert sha(y) == str(g["sha_" + str(key)]), key


def test_global_project_all_periods_vs_oracle(P):
    x = synth.synth(1000, 77)
    xb = np.stack([x, x[::-1].copy()])
    for p in range(2, 501):
        for trunc, orth in ((False, False), (True, False), (False, True), (True, True)):
            got = P.project(xb, p, trunc, orth, staging="global")
            assert np.array_equal(got[0], op.project(x, p, trunc, orth)), (p, trunc, orth)
            assert np.array_equal(got[1], op.project(xb[1], p, trunc, orth)), (p, trunc, orth)
    one = P.project(x, 12, True, True, True, staging="global")
    assert np.array_equal(one, op.project(x, 12, True, True, True))


@pytest.mark.parametrize("trunc,orth", [(False, False), (True, False), (False, True), (True, True)])
def test_global_sweep_matches_on_chip_direct_fold(P, trunc, orth):
    xb = synth.synth_batch(3, 2000, 21)
    for metric in ("norm", "gamma", "imposed", "maxabs"):
        on = P(trunc, orth, fold_mode="direct", staging="shared").sweep(xb, metric=metric, max_length=666)
        lg = G(trunc, orth).sweep(xb, metric=metric, max_length=666)
        np.testing.assert_allclose(lg[0][:, 2:], on[0][:, 2:], rtol=1e-13, atol=0)
        assert np.array_equal(lg[1], on[1]), metric
        np.testing.assert_allclose(lg[2], on[2], rtol=1e-13)
        if metric == "maxabs":
            assert np.array_equal(lg[0], on[0])   # exact sequential sums


@pytest.mark.parametrize("tag", ["00", "11"])
def test_global_readme_algorithms_vs_golden(P, tag):
    g = load_golden("readme")
    c = synth.readme_signal(0)
    trunc, orth = tag[0] == "1", tag[1] == "1"
    inst = G(c, trunc, orth)
    per, pw, bs = inst.small_to_large(thresh=0.1)
    assert per == g[f"s2l_{tag}_periods"].tolist()
    np.testing.assert_allclose(pw, g[f"s2l_{tag}_powers"], rtol=RTOL)
    np.testing.assert_allclose(np.array(bs), g[f"s2l_{tag}_bases"], rtol=RTOL, atol=1e-14)
    w = _quiet()
    try:
        for name, fn in (("mbest", inst.m_best), ("gamma", inst.m_best_gamma)):
            per, pw, bs = fn(num=10)
            assert per.dtype == np.uint32 and np.array_equal(per, g[f"{name}_{tag}_periods"]), name
            np.testing.assert_allclose(pw, g[f"{name}_{tag}_powers"], rtol=RTOL)
            np.testing.assert_allclose(bs, g[f"{name}_{tag}_bases"], rtol=RTOL, atol=1e-14)
    finally:
        w.__exit__(None, None, None)
    per, pw, bs = inst.best_correlation(num=3)
    assert np.array_equal(per, g[f"bcorr_{tag}_periods"])
    np.testing.assert_allclose(pw, g[f"bcorr_{tag}_powers"], rtol=RTOL, atol=1e-15)
    np.testing.assert_allclose(bs, g[f"bcorr_{tag}_bases"], rtol=RTOL, atol=1e-14)
    if tag == "00":
        assert np.array_equal(G().m_best(c, num=10)[2], g["mbest_00_bases"])
        assert np.array_equal(G().best_correlation(c, num=3)[2], g["bcorr_00_bases"])
        assert np.array_equal(np.array(G().small_to_large(c, 0.1)[2]), g["s2l_00_bases"])


def test_global_mbest_stream_windows_vs_golden(P):
    g = load_golden("mbest_stream")
    win = synth.windows_from_stream(synth.synth_stream(n_windows=128 * 3 + 1))
    inst = G()
    for name, fn in (("mbest", inst.m_best), ("gamma", inst.m_best_gamma)):
        res = fn(win, num=10, max_length=1024, return_bases=True)
        assert res.status.max() == 0
        for b in (0, 128, 300):
            assert np.array_equal(res.periods[b], g[f"{name}_{b}_periods"]), (name, b)
            np.testing.assert_allclose(res.powers[b], g[f"{name}_{b}_powers"], rtol=RTOL)
            assert sha(res.bases[b]) == str(g[f"{name}_{b}_bases_sha"]), (name, b)
        on = (P().m_best_gamma if name == "gamma" else P().m_best)(win, num=10, max_length=1024)
        assert np.array_equal(res.periods, on.periods) and np.array_equal(res.sweeps, on.sweeps)


def test_global_mbest_exact_ties_vs_reference_fixture(P):
    g = load_golden("ties")
    inputs = tie_inputs()
    names = sorted(inputs)
    xb = np.stack([inputs[k] for k in names])
    for tag, gamma in (("norm", False), ("gamma", True)):
        for dtype in ("fp64", "fp32"):
            algo = G(dtype=dtype)
            res = (algo.m_best_gamma if gamma else algo.m_best)(xb, num=1, max_length=1024, return_bases=True)
            assert res.status.tolist() == [0] * len(names)
            for i, k in enumerate(names):
                assert int(res.periods[i, 0]) == int(g[f"{k}_{tag}_period"][0]), (tag, k, res.periods[i])
                np.testing.assert_allclose(res.powers[i, 0], g[f"{k}_{tag}_power"][0], rtol=1e-12)
                assert sha(res.bases[i]) == str(g[f"{k}_{tag}_base_sha"]), (tag, k)
            if not gamma:
                assert (np.asarray(res.near_ties) >= 1).all()


def test_global_s2l_and_bcorr_vs_golden(P):
    g = load_golden("s2l_2048")
    xb = synth.synth_batch(4, 2048, 20_000)
    for tag in ("00", "10", "11"):
        res = G(tag[0] == "1", tag[1] == "1").small_to_large(xb, thresh=0.1, return_bases=True)
        for b in range(4):
            per, pw, bs = res.window(b)
            assert per == g[f"s2l_{b}_{tag}_periods"].tolist(), (tag, b)
            np.testing.assert_allclose(pw, g[f"s2l_{b}_{tag}_powers"], rtol=RTOL)
            if tag == "00":
                assert sha(np.array(bs)) == str(g[f"s2l_{b}_{tag}_bases_sha"])
    g = load_golden("bcorr")
    xb = synth.synth_batch(3, 2048, 40_000)
    for tag in ("00", "11"):
        res = G(tag[0] == "1", tag[1] == "1").best_correlation(xb, num=5, return_bases=True)
        for b in range(3):
            assert np.array_equal(res.periods[b], g[f"n2048_{b}_{tag}_periods"]), (tag, b)
            np.testing.assert_allclose(res.powers[b], g[f"n2048_{b}_{tag}_powers"], rtol=RTOL, atol=1e-15)
            assert sha(res.bases[b]) == str(g[f"n2048_{b}_{tag}_bases_sha"]), (tag, b)


def test_global_best_frequency_matches_on_chip(P):
    xb = synth.synth_batch(3, 2000, 901)
    for trunc, orth in ((False, False), (True, True)):
        a = P(trunc, orth, staging="shared").best_frequency(xb, num=4)
        b = G(trunc, orth).best_frequency(xb, num=4)
        assert np.array_equal(a.periods, b.periods) and np.array_equal(a.powers, b.powers)
        assert np.array_equal(a.bases, b.bases)


@pytest.mark.parametrize("trunc", [False, True])
def test_global_differential_many_windows(P, trunc):
    xb = synth.synth_batch(48, 1024, 777_000 + int(trunc))
    inst = G(trunc, False)
    mb = inst.m_best(xb, num=6, max_length=300)
    mg = inst.m_best_gamma(xb, num=6, max_length=300)
    sl = inst.small_to_large(xb, thresh=0.08)
    bc = inst.best_correlation(xb, num=4, max_length=300)
    for b in range(48):
        per, pw, _ = op.m_best(xb[b], 6, 300, 2, trunc)
        assert np.array_equal(mb.periods[b], per), ("m_best", b)
        np.testing.assert_allclose(mb.powers[b], pw, rtol=RTOL)
        per, pw, _ = op.m_best_gamma(xb[b], 6, 300, 2, trunc)
        assert np.array_equal(mg.periods[b], per), ("gamma", b)
        np.testing.assert_allclose(mg.powers[b], pw, rtol=RTOL)
        per, pw, _ = op.small_to_large(xb[b], 0.08, None, trunc)
        k = int(sl.count[b])
        assert sl.periods[b, :k].tolist() == per, ("s2l", b)
        np.testing.assert_allclose(sl.powers[b, :k], pw, rtol=1e-9)
        per, pw, _ = op.best_correlation(xb[b], 4, 300, 0.01, trunc)
        assert np.array_equal(bc.periods[b], per), ("bcorr", b)
        np.testing.assert_allclose(bc.powers[b], pw, rtol=RTOL, atol=1e-15)


# ---------------------------------------------------------------- (2) windows the on-chip path cannot take
@pytest.mark.parametrize("trunc,orth", [(False, False), (True, True)])
def test_n20000_all_algorithms_vs_oracle(P, trunc, orth):
    """N = 20 000 at default arguments is above every on-chip limit; N = 12 000 goes through the on-chip path in the
    same test (auto dispatch on both sides of the limit)."""
    w = _quiet()
    try:
        for n in (20000, 12000):
            x = synth.synth(n, 123)
            inst = P(x, trunc, orth)
            per, pw, bs = inst.m_best(num=4)
            per0, pw0, bs0 = op.m_best(x, 4, None, 2, trunc, orth)
            assert np.array_equal(per, per0), (n, per, per0)
            np.testing.assert_allclose(pw, pw0, rtol=RTOL)
            np.testing.assert_allclose(bs, bs0, rtol=RTOL, atol=1e-14)
            if not orth:
                assert np.array_equal(bs, bs0)
            per, pw, _ = inst.m_best_gamma(num=4)
            per0, pw0, _ = op.m_best_gamma(x, 4, None, 2, trunc, orth)
            assert np.array_equal(per, per0), (n, "gamma")
            np.testing.assert_allclose(pw, pw0, rtol=RTOL)
            per, pw, bs = inst.small_to_large(thresh=0.05)
            per0, pw0, bs0 = op.small_to_large(x, 0.05, None, trunc, orth)
            assert per == per0, (n, "s2l")
            np.testing.assert_allclose(pw, pw0, rtol=1e-9)
            per, pw, bs = inst.best_correlation(num=3)
            per0, pw0, bs0 = op.best_correlation(x, 3, None, 0.01, trunc, orth)
            assert np.array_equal(per, per0), (n, "bcorr")
            np.testing.assert_allclose(pw, pw0, rtol=RTOL, atol=1e-15)
            if not orth:
                assert np.array_equal(bs, bs0)
            per, pw, bs = inst.best_frequency(num=3)
            per0, pw0, bs0 = op.best_frequency(x, None, 3, trunc, orth)
            assert np.array_equal(per, per0), (n, "bfreq")
            np.testing.assert_allclose(pw, pw0, rtol=RTOL)
            for p in (2, 999, n // 2, n // 2 + 1, n):
                assert np.array_equal(P.project(x, p, trunc, orth), op.project(x, p, trunc, orth)), (n, p)
    finally:
        w.__exit__(None, None, None)


def test_n32768_max_length_2048_and_n262144(P):
    x = synth.synth(32768, 5)
    per, pw, bs = P().m_best(x, num=4, max_length=2048)
    per0, pw0, bs0 = op.m_best(x, 4, 2048)
    assert np.array_equal(per, per0)
    np.testing.assert_allclose(pw, pw0, rtol=RTOL)
    assert np.array_equal(bs, bs0)
    x = synth.synth(262144, 6)
    per, pw, bs = P().m_best(x, num=3, max_length=1024)
    per0, pw0, bs0 = op.m_best(x, 3, 1024)
    assert np.array_equal(per, per0)
    np.testing.assert_allclose(pw, pw0, rtol=RTOL)
    assert np.array_equal(bs, bs0)


def test_project_n2pow20_bit_exact(P):
    n = 1 << 20
    x = synth.synth(n, 7)
    for p in (2, 1000, n // 2 + 1):
        for trunc, orth in ((False, False), (True, True)):
            assert np.array_equal(P.project(x, p, trunc, orth), op.project(x, p, trunc, orth)), (p, trunc, orth)


def test_exactly_periodic_long_window_keeps_the_lowest_period(P):
    rng = np.random.default_rng(77)
    x = np.tile(rng.integers(-5, 6, 10).astype(float), 2000)   # N = 20 000, period 10
    per, pw, _ = P().m_best(x, num=1)
    assert per.tolist() == [10] and abs(pw[0] - 1.0) < 1e-12
    res = P().m_best(x[None, :], num=1)
    assert int(res.near_ties[0]) >= 1
    _, bp, _ = P().sweep(x, metric="norm")
    assert int(bp[0]) == 10


# ---------------------------------------------------------------- (3) batches
def test_hop_framed_batch_equals_per_window_calls(P):
    n, hop, b = 65536, 4096, 64
    stream = synth.synth(n + hop * (b - 1), 31)
    win = np.lib.stride_tricks.as_strided(stream, (b, n), (hop * 8, 8))
    res = P().m_best(win, num=3, max_length=1024, return_bases=True)
    assert res.status.max() == 0
    for i in range(b):
        per, pw, bs = P().m_best(np.ascontiguousarray(win[i]), num=3, max_length=1024)
        assert np.array_equal(res.periods[i], per) and np.array_equal(res.powers[i], pw), i
        assert np.array_equal(res.bases[i], bs), i


def test_batch_in_several_pieces_and_determinism(P):
    # 8 MB residuals: the L2-sized pieces hold only a few windows, so this batch runs in several pieces
    n, b = 1 << 20, 24
    xb = synth.synth_batch(b, n, 41)
    inst = P(staging="global")
    r1 = inst.m_best(xb, num=2, max_length=200)
    r2 = inst.m_best(xb, num=2, max_length=200)
    assert np.array_equal(r1.periods, r2.periods) and np.array_equal(r1.powers, r2.powers)
    s1 = inst.small_to_large(xb[:2], thresh=0.05, n_periods=100)
    c1 = inst.best_correlation(xb[:2], num=2, max_length=100)
    for i in range(b):
        one = inst.m_best(xb[i], num=2, max_length=200)
        assert np.array_equal(one[0], r1.periods[i]) and np.array_equal(one[1], r1.powers[i]), i
    for i in range(2):
        per, pw, _ = op.small_to_large(xb[i], 0.05, 100)
        assert s1.window(i)[0] == per
        per, pw, _ = op.best_correlation(xb[i], 2, 100)
        assert np.array_equal(c1.periods[i], per)


def test_device_tensors_empty_batch_and_zero_windows(P):
    import torch
    x = torch.from_numpy(synth.synth_batch(3, 20000, 8)).cuda()
    res = P().m_best(x, num=3, max_length=500)
    assert res.periods.is_cuda and res.powers.is_cuda and res.bases is None
    host = P().m_best(x.cpu().numpy(), num=3, max_length=500)
    assert np.array_equal(res.periods.cpu().numpy().view(np.uint32), host.periods)
    assert np.array_equal(res.powers.cpu().numpy(), host.powers)
    pj = P.project(x, 7000)
    assert pj.is_cuda and torch.equal(pj, P.project(x, 7000))
    empty = np.zeros((0, 20000))
    assert P().m_best(empty, num=3).periods.shape == (0, 3)
    assert P().small_to_large(empty, thresh=0.1).count.shape == (0,)
    assert P().best_correlation(empty, num=2).periods.shape == (0, 2)
    assert P.project(empty, 5000).shape == (0, 20000)
    with pytest.raises(TypeError):
        P().m_best(np.zeros(20000), num=3)
    with pytest.raises(TypeError):
        P().best_correlation(np.zeros(20000), num=2)
    res = P().m_best(np.zeros((2, 20000)), num=3)
    assert res.status.tolist() == [1, 1]
    res = P().best_correlation(np.zeros((2, 20000)), num=2, return_bases=True)
    assert res.status.tolist() == [1, 1] and not res.periods.any() and not res.bases.any()
    per, pw, bs = P().small_to_large(np.zeros(20000), thresh=0.1)
    assert per == [] and pw == []


def test_shared_staging_keeps_the_on_chip_error(P):
    from pyperiod_b200 import _lib
    with pytest.raises(_lib.PPError, match="shared memory"):
        P(staging="shared").m_best(synth.synth(20000, 1), num=2)
