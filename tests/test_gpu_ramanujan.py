"""GPU parity tests for RamanujanPeriods: periodogram (dense DMMA contraction on folded sums) and
find_periods_with_weights, against the golden fixtures of the reference and the fp64 closed form."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import ramanujan as oram
from pyperiod_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    from pyperiod_b200 import RamanujanPeriods
    return RamanujanPeriods


def test_norms_vs_fp64_closed_form(R):
    for n, seed, qmax in ((1024, 50_000, None), (2000, 7, 150), (999, 3, 333)):
        x = synth.synth(n, seed)
        got = R().find_periods(x, 2, qmax)
        want = oram.norms_closed_form_f64(x, 2, qmax)
        assert got.shape == want.shape and got[0] == 0 and got[1] == 0
        np.testing.assert_allclose(got[2:], want[2:], rtol=1e-11, atol=0)


def test_norms_vs_reference_float32_limited(R):
    g = load_golden("readme_qo_ram")
    c = synth.readme_signal(0)
    got = R().find_periods(c, 2, 120)
    np.testing.assert_allclose(got, g["ram_norms"], rtol=2e-6)   # the reference stores float32 (RamanujanPeriods.py:127)
    g2 = load_golden("qo_ram_synth")
    xb = synth.synth_batch(2, 1024, 50_000)
    nb = R().find_periods(xb)
    for b in range(2):
        np.testing.assert_allclose(nb[b], g2[f"ram_{b}_norms"], rtol=2e-6)


def test_f32_compat_reproduces_the_reference_numbers(R):
    """precision='f32_compat': float32 storage (RamanujanPeriods.py:127), sequential float32 row sum and numpy's
    pairwise sum of squares (:77-78) reproduced on the device.  Against the reference-generated fixtures the norms are
    equal to the last float32 bit on almost every period (fp64 path: 2e-7 .. 2e-6 away)."""
    g = load_golden("readme_qo_ram")
    c = synth.readme_signal(0)
    got = R(precision="f32_compat").find_periods(c, 2, 120)
    ref = g["ram_norms"]
    assert got.shape == ref.shape
    np.testing.assert_allclose(got, ref, rtol=3e-8)
    assert np.sum(got == ref) >= 0.95 * len(ref), int(np.sum(got == ref))
    g2 = load_golden("qo_ram_synth")
    xb = synth.synth_batch(2, 1024, 50_000)
    nb = R(precision="f32_compat").find_periods(xb)
    for b in range(2):
        ref = g2[f"ram_{b}_norms"]
        np.testing.assert_allclose(nb[b], ref, rtol=3e-8)
        assert np.sum(nb[b] == ref) >= 0.9 * len(ref), int(np.sum(nb[b] == ref))
    # ragged tile (5 windows, odd N) against the oracle's float32 emulation
    xr = synth.synth_batch(5, 777, 31)
    nr = R(precision="f32_compat").find_periods(xr, 2, 200)
    for b in range(5):
        want = oram.find_periods_f32_exact_cq(xr[b], 2, 200)
        np.testing.assert_allclose(nr[b], want, rtol=3e-8)
        assert np.sum(nr[b] == want) >= 0.9 * len(want)


def test_batch_tiles_and_odd_sizes(R):
    xb = synth.synth_batch(7, 600, 123)          # 7 windows: partial 4-window fold group and partial GEMM tile
    nb = R().find_periods(xb, 3, 200)
    for b in range(7):
        want = oram.norms_closed_form_f64(xb[b], 3, 200)
        np.testing.assert_allclose(nb[b, 3:], want[3:], rtol=1e-11)
        assert not nb[b, :3].any()


def test_find_periods_with_weights_vs_golden(R):
    g = load_golden("readme_qo_ram")
    c = synth.readme_signal(0)
    d, res = R().find_periods_with_weights(c, max_length=120, thresh=0.2)
    assert d["periods"].tolist() == g["ram_periods"].tolist() == [58, 60, 100, 102]
    assert [int(k) for k in d["basis_dictionary"]] == g["ram_dict_keys"].tolist()
    assert list(d["basis_dictionary"].values()) == g["ram_dict_vals"].tolist()
    np.testing.assert_allclose(d["norms"], g["ram_sel_norms"], rtol=2e-6)
    np.testing.assert_allclose(d["weights"], g["ram_weights"], rtol=1e-8, atol=1e-11)
    np.testing.assert_allclose(res, g["ram_res"], rtol=0, atol=1e-11)
    g2 = load_golden("qo_ram_synth")
    xb = synth.synth_batch(2, 1024, 50_000)
    out = R().find_periods_with_weights(xb, thresh=0.2)
    for b in range(2):
        d, res = out.window(b)
        assert np.asarray(d["periods"]).tolist() == g2[f"ram_{b}_periods"].tolist()
        assert list(d["basis_dictionary"].values()) == g2[f"ram_{b}_dict_vals"].tolist()
        np.testing.assert_allclose(d["weights"], g2[f"ram_{b}_weights"], rtol=1e-7, atol=1e-10)
        np.testing.assert_allclose(res, g2[f"ram_{b}_res"], rtol=0, atol=1e-10)


def test_tf32_option_tracks_fp64():
    """precision="tf32": split-TF32 contraction on the tcgen05 tensor cores (accumulator in tensor memory, fp32
    accumulate); norms within 1e-5 of the fp64 path relative to the largest norm, the thresholded period selection
    is unchanged and so are the weights (the solve stage never sees the periodogram values, only the periods)."""
    from pyperiod_b200 import RamanujanPeriods
    xb = synth.synth_batch(70, 2048, 61_000)   # one ragged 128-window unit; q <= 400 fits one accumulator tile
    a = RamanujanPeriods().find_periods(xb, 2, 400)
    b = RamanujanPeriods(precision="tf32").find_periods(xb, 2, 400)
    scale = a.max(axis=1, keepdims=True)
    assert np.max(np.abs(a - b) / scale) < 1e-5
    assert np.all(b[:, :2] == 0)
    ra = RamanujanPeriods().find_periods_with_weights(xb[:8], max_length=200, thresh=0.2)
    rb = RamanujanPeriods(precision="tf32").find_periods_with_weights(xb[:8], max_length=200, thresh=0.2)
    assert ra.status.tolist() == rb.status.tolist() == [0] * 8     # every window is solved in both modes
    for i in range(8):
        da, _ = ra.window(i)
        db, _ = rb.window(i)
        assert np.array_equal(np.asarray(da["periods"]), np.asarray(db["periods"]))
        assert da["basis_dictionary"] == db["basis_dictionary"]
        np.testing.assert_allclose(db["weights"], da["weights"], rtol=0, atol=1e-12 * np.max(np.abs(da["weights"])))


def _planted_cosines(b, n, seed, qmin, qmax, amp):
    """synth windows, each plus amp * cos(2 pi m / q) for a q drawn from [qmin, qmax]."""
    rng = np.random.default_rng(seed)
    xb = synth.synth_batch(b, n, seed)
    m = np.arange(n)
    for i in range(b):
        xb[i] += amp * np.cos(2 * np.pi * m / int(rng.integers(qmin, qmax + 1)))
    return xb


def test_tf32_at_config5_shape_across_tiles(monkeypatch):
    """precision="tf32" at config 5's shape (N = 4096, q <= 1365) on every tile path of the kernel: with 160 windows
    per fold tile, 300 windows make two tiles, each a full 128-window unit and a ragged one; q > 512 takes a second
    512-column accumulator tile.  Strong components at periods in (512, 1365] put the largest norms there.  Norms
    within 1e-5 of the fp64 path relative to the largest norm, and per q > 512 within 1e-4 of that q's own norm (a
    dropped or stale accumulator tile cannot hide below the window maximum)."""
    from pyperiod_b200 import RamanujanPeriods, ramanujan as ram_mod
    monkeypatch.setattr(ram_mod, "TILE_WINDOWS", 160)
    xb = _planted_cosines(300, 4096, 64_000, 513, 1365, 4.0)
    a = RamanujanPeriods().find_periods(xb)
    b = RamanujanPeriods(precision="tf32").find_periods(xb)
    assert a.shape == b.shape == (300, 1366)
    assert np.all(b[:, :2] == 0)
    scale = a.max(axis=1, keepdims=True)
    rel = np.abs(a - b) / scale
    hi = np.abs(a[:, 513:] - b[:, 513:]) / a[:, 513:]
    print(f"\ntf32: windows with the largest norm above q = 512: {np.mean(a.argmax(axis=1) > 512):.2f}; "
          f"worst error / largest norm {rel.max():.2g}; worst error / own norm for q > 512 {hi.max():.2g}")
    assert rel.max() < 1e-5
    assert hi.max() < 1e-4
    ra = RamanujanPeriods().find_periods_with_weights(xb, thresh=0.2)
    rb = RamanujanPeriods(precision="tf32").find_periods_with_weights(xb, thresh=0.2)
    assert np.array_equal(ra.n_periods, rb.n_periods)
    assert np.array_equal(ra.periods, rb.periods)


def test_fp64_fused_kernel_across_l2_groups(monkeypatch):
    """The fused fp64 kernel keeps L2_GROUP_WINDOWS windows (rounded up to a multiple of 8) L2-resident while every
    period passes over them.  Each window's column of the 8-window DMMA product does not depend on the grouping: with
    groups of 24 windows (24 + 24 + 5) the norms are bit-identical to one group, and so is a hop-framed view."""
    from pyperiod_b200 import RamanujanPeriods, ramanujan as ram_mod
    n, hop, count = 2048, 1000, 53
    stream = synth.synth(n + hop * (count - 1), 65_000)
    framed = np.lib.stride_tricks.as_strided(stream, (count, n), (hop * 8, 8))   # overlapping windows, ldx < N
    xb = np.ascontiguousarray(framed)
    ref = RamanujanPeriods().find_periods(xb)
    monkeypatch.setattr(ram_mod, "L2_GROUP_WINDOWS", 20)
    got = RamanujanPeriods().find_periods(xb)
    assert np.array_equal(got, ref)
    assert np.array_equal(RamanujanPeriods().find_periods(framed), ref)
    for b in (0, 26, 52):
        want = oram.norms_closed_form_f64(xb[b])
        np.testing.assert_allclose(got[b, 2:], want[2:], rtol=1e-11, atol=0)


def test_f32_compat_above_one_accumulator_tile(monkeypatch):
    """precision="f32_compat" for q up to 700 in a ragged fold tile (3 windows, 2 per tile) against the oracle's
    float32 emulation of the reference, with the bars of test_f32_compat_reproduces_the_reference_numbers."""
    from pyperiod_b200 import RamanujanPeriods, ramanujan as ram_mod
    monkeypatch.setattr(ram_mod, "TILE_WINDOWS", 4)         # f32_compat holds TILE_WINDOWS // 2 windows per tile
    xb = _planted_cosines(3, 2100, 66_000, 513, 700, 1.0)
    got = RamanujanPeriods(precision="f32_compat").find_periods(xb, 2, 700)
    for b in (0, 2):
        want = oram.find_periods_f32_exact_cq(xb[b], 2, 700)
        np.testing.assert_allclose(got[b], want, rtol=3e-8)
        assert np.sum(got[b] == want) >= 0.9 * len(want), int(np.sum(got[b] == want))


# ------------------------------------------------------------------ config 5 at its own shape (N = 4096, q <= 1365)
CFG5_PERIODS = {   # what thresh = 0.2 selects on these config-5 windows (fp64 periodogram), and the dictionary rows
    6: ([23, 24, 75, 252, 390, 528], 1234),
    14: None,      # 14 periods, 2896 rows: taken from the periodogram in the test
    18: ([80, 132, 134, 135, 136, 138, 152, 336, 396, 406, 672], 2170),   # cond(G) = 3.8e12
}


def test_cfg5_shape_periodogram_vs_closed_form(R):
    """RamanujanPeriods.find_periods at config 5's own shape (N = 4096, q = 2..1365) against the fp64 closed form."""
    x = synth.synth(4096, 50_006)
    got = R().find_periods(x)
    want = oram.norms_closed_form_f64(x)
    assert got.shape == want.shape == (1366,)
    np.testing.assert_allclose(got[2:], want[2:], rtol=1e-10, atol=0)


def _check_against_refined(x, d, res, w_ref=None, res_ref=None):
    """The device solves the reference's normal equations at least as accurately as the reference's own LU: both are
    compared with a solution refined in extended precision.  (cond(G) reaches 1e14 on config-5 dictionaries: the LU
    weights are then good to 3e-4 only, so 'equal to the reference' can mean no more than 'within its own error'.)"""
    from conftest import refined_normal_equations
    from oracle import qo as oq
    a, layout = oq.get_subspaces(np.asarray(d["periods"]), len(x))
    assert d["basis_dictionary"] == layout
    w_star, res_star, w_lu = refined_normal_equations(a, x)
    if w_ref is None:
        w_ref, res_ref = w_lu, x - a.T @ w_lu
    scale = float(np.max(np.abs(w_star)))
    err_gpu = float(np.max(np.abs(d["weights"] - w_star))) / scale
    err_ref = float(np.max(np.abs(w_ref - w_star))) / scale
    assert err_gpu <= max(1e-10, err_ref), (err_gpu, err_ref)
    assert float(np.max(np.abs(d["weights"] - w_ref))) / scale <= max(1e-10, 2.0 * err_ref)
    rerr_gpu = float(np.max(np.abs(res - res_star)))
    rerr_ref = float(np.max(np.abs(res_ref - res_star)))
    assert rerr_gpu <= max(1e-11, rerr_ref), (rerr_gpu, rerr_ref)
    assert float(np.max(np.abs(res - res_ref))) <= max(1e-11, 2.0 * rerr_ref)
    return err_gpu, err_ref


def test_cfg5_large_dictionaries_are_solved(R):
    """Dictionaries of more than 1024 rows (a quarter of config 5's windows) are solved like any other."""
    xb = np.stack([synth.synth(4096, 50_000 + b) for b in (6, 14, 18, 2)])
    out = R().find_periods_with_weights(xb, thresh=0.2)
    assert out.status.tolist() == [0, 0, 0, 0]
    rows = [int(v) for v in out.n_weights]
    assert rows[0] == 1234 and rows[1] == 2896 and rows[2] == 2170 and rows[3] == 396
    assert np.asarray(out.periods[0][: int(out.n_periods[0])]).tolist() == CFG5_PERIODS[6][0]
    assert np.asarray(out.periods[2][: int(out.n_periods[2])]).tolist() == CFG5_PERIODS[18][0]
    for i in range(4):
        d, res = out.window(i)
        _check_against_refined(xb[i], d, res)


def test_cfg5_large_dictionaries_in_two_launches(R, monkeypatch):
    """The large dictionaries go to the solve kernel in two launches (two CTAs per SM up to RMAX_TWO_CTAS rows, one
    above): with the boundary moved to 2000 rows windows 6 (1234 rows) and 14 (2896 rows) take different launches and
    the results do not change."""
    from pyperiod_b200 import ramanujan as ram_mod
    xb = np.stack([synth.synth(4096, 50_000 + b) for b in (6, 14, 18, 2)])
    ref = R().find_periods_with_weights(xb, thresh=0.2)
    monkeypatch.setattr(ram_mod, "RMAX_TWO_CTAS", 2000)
    out = R().find_periods_with_weights(xb, thresh=0.2)
    assert out.status.tolist() == ref.status.tolist() == [0, 0, 0, 0]
    for i in range(4):
        d0, r0 = ref.window(i)
        d1, r1 = out.window(i)
        assert d0["basis_dictionary"] == d1["basis_dictionary"]
        assert np.array_equal(d0["weights"], d1["weights"]) and np.array_equal(r0, r1)


def test_cfg5_reference_fixture(R):
    """Reference-generated fixture (tests/golden/ram_cfg5.npz, make_golden.py ram_cfg5): find_periods_with_weights at
    config 5's shape on windows whose dictionaries have 1234 / 2896 / 1324 rows.  Periods, dictionary layout and norms
    as the reference returns them; weights and residual within the reference's own distance from the refined
    solution of its normal equations."""
    import os
    from conftest import GOLDEN
    if not os.path.exists(os.path.join(GOLDEN, "ram_cfg5.npz")):
        pytest.skip("ram_cfg5.npz not generated")
    g = load_golden("ram_cfg5")
    for b in g["windows"].tolist():
        x = synth.synth(4096, 50_000 + b)
        d, res = R().find_periods_with_weights(x, thresh=0.2)
        assert np.asarray(d["periods"]).tolist() == g[f"w{b}_periods"].tolist()
        assert [int(k) for k in d["basis_dictionary"]] == g[f"w{b}_dict_keys"].tolist()
        assert list(d["basis_dictionary"].values()) == g[f"w{b}_dict_vals"].tolist()
        np.testing.assert_allclose(d["norms"], g[f"w{b}_sel_norms"], rtol=2e-6)
        _check_against_refined(x, d, res, g[f"w{b}_weights"], g[f"w{b}_res"])


def test_test_function_replaces_threshold(R):
    """test_function(norms) -> periods (RamanujanPeriods.py:94-101), a host callable between the two kernels."""
    from oracle import qo as oq
    x = synth.synth(1024, 50_001)
    pick = lambda norms: np.argsort(norms)[-3:][::-1]
    d, res = R().find_periods_with_weights(x, test_function=pick)
    norms = R().find_periods(x)
    want = pick(norms)
    assert np.asarray(d["periods"]).tolist() == want.tolist()
    a, layout = oq.get_subspaces(want, 1024)
    w0, rec0 = oq.solve_quadratic(x, a)
    assert d["basis_dictionary"] == layout
    np.testing.assert_allclose(d["weights"], w0, rtol=0, atol=1e-10 * np.max(np.abs(w0)))
    np.testing.assert_allclose(res, x - rec0, rtol=0, atol=1e-12)
