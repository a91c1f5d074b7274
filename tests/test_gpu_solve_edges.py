"""The FP64 normal-equations solve (csrc/pp_chol.cuh, cta_qo_solve in csrc/pp_qo.cuh) at its structural edges.

Iterative refinement converges for any factor that is a reasonable preconditioner, so a factor that is wrong in its
sixth digit still yields weights good to 1e-15 after a step or two.  These tests therefore solve with `refine=0` and
hold the bare factor to a bound in the condition number of the Gram matrix G = A A^T:

    max|w - w*| / max|w*| <= max(2 kappa_2(G) 2^-53, 1e-13),   max|res - res*| <= max(2 kappa_2(G) 2^-53 max|x|, 1e-12)

against w*, res* refined in extended precision (conftest.refined_normal_equations).  The edges:

- dictionary size R mod 32 (packed 32 x 32 blocks, identity padding, the right-hand side as a virtual row at
  32 ceil(R / 32)), R around the 128-row passes, R = N (square, full rank) and R = N + 1 (singular by rank);
- both launches of RamanujanPeriods' solve stage and both launch plans (window staged in shared memory or read in
  place), the global-memory path and a grid of one CTA that solves every window in turn;
- the incremental factorisation of find_periods, which keeps the factor rows below 32 floor(R_prev / 32) from the
  previous round: its weights must be bit-identical to a from-scratch solve of the same period list.
"""
import numpy as np
import pytest

from conftest import load_golden, refined_normal_equations
from oracle import qo as oq
from oracle.numtheory import divisor_set, phi
from pyperiod_b200 import synth

U = 2.0 ** -53
N = 4096

# Period lists (in solve order) whose natural-basis dictionary has the given number of rows at N = 4096.  Every list
# from R = 3 on has two or more periods (off-diagonal blocks in G) except R = 64, a single period (diagonal G); R = 255
# has eight, three of which start inside the first 32-row block.  kappa_2(G) <= 3e7 everywhere.  R = 4096 is a coprime
# pair with q1 + q2 - 1 = N: full rank by Fine and Wilf.  R = 4097 has more rows than samples: singular by rank.
SIZES = {
    1: [1],
    2: [2],
    31: [13, 19],
    32: [6, 10, 21],
    33: [15, 19],
    63: [27, 45],
    64: [64],
    65: [25, 45],
    127: [61, 67],
    128: [32, 112],
    129: [27, 45, 69],
    255: [9, 13, 61, 25, 43, 33, 31, 51],
    256: [76, 184],
    257: [49, 55, 161],
    1023: [285, 739],
    1024: [232, 302, 494],
    1025: [485, 545],
    2047: [511, 1537],
    2048: [444, 773, 833],
    2049: [657, 1393],
    3071: [961, 2111],
    3072: [739, 834, 1502],
    3073: [1423, 1651],
    4095: [1315, 2785],
    4096: [2048, 2049],
    4097: [1751, 2363],
}
TARGETS = sorted(SIZES)
SEED0 = 73_000          # window i is synth.synth(N, SEED0 + i)

# find_periods(num=4, thresh=0.0) on planted-period windows: (N, planted periods, amplitudes, seed) -> the periods the
# gamma sweep finds round by round and the dictionary rows after each round (the oracle's, checked on the CPU).  The
# factor rows below 32 floor(R_prev / 32) are kept from the previous round; the edges each sequence reaches:
#   31 -> 32, 31 -> 115: R_prev = 32k - 1;   64 -> 128, 32 -> 104: R_prev = 32k;   65 -> 137, 129 -> 133: 32k + 1;
#   115 -> 120, 137 -> 139, 141 -> 148, 129 -> 133: the new rows stay inside R_prev's 32-row block;
#   128 -> 256, 148 -> 366, 133 -> 679, 120 -> 188 ...: the rows redone span more than one 128-row pass.
PLANTED = [
    (1024, [31, 146, 167], [0.69, 0.56, 0.24], 1371, [31, 2, 73, 146], [31, 32, 104, 176]),
    (1024, [31, 85, 150], [0.52, 0.42, 0.42], 2838, [31, 85, 6, 75], [31, 115, 120, 188]),
    (2048, [65, 73, 165], [0.9, 0.73, 0.38], 8552, [5, 65, 73, 3], [5, 65, 137, 139]),
    (2048, [128, 657, 260], [0.84, 0.54, 0.44], 5400, [64, 128, 5, 130], [64, 128, 132, 256]),
    (2048, [127, 401, 240], [0.49, 0.4, 0.53], 8054, [127, 15, 8, 240], [127, 141, 148, 366]),
    (4096, [129, 547, 1285], [0.89, 0.46, 0.59], 2318, [43, 129, 5, 547], [43, 129, 133, 679]),
]


def planted(n, periods, amps, seed):
    """Sum of a_k * (a random pattern of length q_k, tiled) plus 1e-3 white noise."""
    rng = np.random.default_rng(seed)
    x = 1e-3 * rng.standard_normal(n)
    for q, a in zip(periods, amps):
        x += a * np.tile(rng.standard_normal(q), n // q + 1)[:n]
    return x


def dictionary_rows(periods):
    """Rows of the natural-basis dictionary of `periods`: sum of phi(d) over the union of their divisors."""
    seen = set()
    for q in periods:
        seen |= divisor_set(int(q))
    return sum(phi(d) for d in seen)


# ------------------------------------------------------------------ CPU: the tables say what they claim
def test_period_tables_give_their_rows():
    singles = []
    for r, periods in SIZES.items():
        a, layout = oq.get_subspaces(periods, N)
        assert a.shape == (r, N), (r, periods)
        assert 0 not in layout.values(), (r, layout)    # every entry adds rows (keep == 0 would mean all q rows)
        if len(periods) == 1:
            singles.append(r)
    assert singles == [1, 2, 64]
    assert max(len(p) for p in SIZES.values()) >= 8
    assert sorted(SIZES[4096]) == [2048, 2049] and np.gcd(2048, 2049) == 1
    for n, _, _, _, periods, rows in PLANTED:
        assert [dictionary_rows(periods[: k + 1]) for k in range(len(periods))] == rows
        assert len(set(periods)) == len(periods)


def test_planted_sequences_match_the_oracle():
    """The recorded period sequences are what the reference's loop finds on these windows."""
    for n, qs, amps, seed, periods, _ in PLANTED:
        d, _ = oq.find_periods(planted(n, qs, amps, seed), num=4, thresh=0.0)
        assert [int(p) for p in d["periods"]] == periods


# ------------------------------------------------------------------ shared helpers
def _bound_w(kappa):
    return max(2.0 * kappa * U, 1e-13)


def _bound_res(kappa, x):
    return max(2.0 * kappa * U * float(np.max(np.abs(x))), 1e-12)


def _reference(x, a, layout):
    """Refined solution, LU solution and kappa_2(G) of the dictionary `a` (rows) on x."""
    w_star, res_star, w_lu = refined_normal_equations(a, x)
    ev = np.linalg.eigvalsh(a @ a.T)
    return dict(layout=layout, w_star=w_star, res_star=res_star, w_lu=w_lu, res_lu=x - a.T @ w_lu,
                kappa=float(ev[-1] / ev[0]))


def _check_refine0(x, d, res, ref, what):
    """refine=0 against the bound; returns (weights error, residual error) as fractions of their bounds."""
    assert d["basis_dictionary"] == ref["layout"], what
    ew = float(np.max(np.abs(d["weights"] - ref["w_star"]))) / float(np.max(np.abs(ref["w_star"])))
    er = float(np.max(np.abs(res - ref["res_star"])))
    bw, br = _bound_w(ref["kappa"]), _bound_res(ref["kappa"], x)
    assert ew <= bw, (what, ew, bw, ref["kappa"])
    assert er <= br, (what, er, br, ref["kappa"])
    return ew / bw, er / br


def _check_refined(x, d, res, ref, what):
    """The standard of test_gpu_ramanujan._check_against_refined: no worse than numpy's LU against the refined
    solution (floor 1e-10 on the weights, 1e-11 on the residual), and within twice the LU's error of the LU."""
    assert d["basis_dictionary"] == ref["layout"], what
    scale = float(np.max(np.abs(ref["w_star"])))
    err = float(np.max(np.abs(d["weights"] - ref["w_star"]))) / scale
    err_lu = float(np.max(np.abs(ref["w_lu"] - ref["w_star"]))) / scale
    assert err <= max(1e-10, err_lu), (what, err, err_lu)
    assert float(np.max(np.abs(d["weights"] - ref["w_lu"]))) / scale <= max(1e-10, 2.0 * err_lu), what
    rerr = float(np.max(np.abs(res - ref["res_star"])))
    rerr_lu = float(np.max(np.abs(ref["res_lu"] - ref["res_star"])))
    assert rerr <= max(1e-11, rerr_lu), (what, rerr, rerr_lu)
    assert float(np.max(np.abs(res - ref["res_lu"]))) <= max(1e-11, 2.0 * rerr_lu), what


def _same_bits(a, b, count):
    for i in range(count):
        da, ra = a.window(i)
        db, rb = b.window(i)
        assert da["basis_dictionary"] == db["basis_dictionary"], i
        assert np.array_equal(da["weights"], db["weights"]), i
        assert np.array_equal(ra, rb), i
    assert a.status.tolist() == b.status.tolist()


# ------------------------------------------------------------------ (1) dictionaries of chosen size
@pytest.fixture(scope="module")
def sized():
    """One window per target size, the reference solution of every solvable one, and the refine=0 batch solve."""
    from pyperiod_b200 import RamanujanPeriods
    xb = np.stack([synth.synth(N, SEED0 + i) for i in range(len(TARGETS))])
    refs = {r: _reference(xb[i], *oq.get_subspaces(SIZES[r], N)) for i, r in enumerate(TARGETS) if r <= N}

    def solve(refine=0, **kw):
        lists = iter([SIZES[r] for r in TARGETS])
        return RamanujanPeriods(**kw).find_periods_with_weights(xb, max_length=8, refine=refine,
                                                                test_function=lambda norms: next(lists))
    return dict(x=xb, refs=refs, solve=solve, base=solve(0))


@pytest.mark.gpu
def test_sized_dictionaries_refine0_meet_the_bound(sized):
    from pyperiod_b200 import _lib
    out, xb = sized["base"], sized["x"]
    assert [int(v) for v in out.n_weights[: len(TARGETS) - 1]] == TARGETS[:-1]
    worst = {}
    for i, r in enumerate(TARGETS):
        if r > N:
            assert int(out.status[i]) == _lib.STATUS_SINGULAR
            _, res = out.window(i)
            assert np.array_equal(res, xb[i])        # res = x exactly
            continue
        assert int(out.status[i]) == _lib.STATUS_OK, r
        d, res = out.window(i)
        ref = sized["refs"][r]
        rw, rr = _check_refine0(xb[i], d, res, ref, r)
        worst[r] = (rw, rr, ref["kappa"])
        if r == N:   # square and full rank: the residual is zero within the bound
            assert float(np.max(np.abs(res))) <= _bound_res(ref["kappa"], xb[i])
    print("\nrefine=0 error / bound (weights, residual, kappa):",
          {r: ("%.2g" % a, "%.2g" % b, "%.1e" % k) for r, (a, b, k) in worst.items()})


@pytest.mark.gpu
@pytest.mark.parametrize("refine", [1, 4])
def test_sized_dictionaries_refined(sized, refine):
    out, xb = sized["solve"](refine), sized["x"]
    for i, r in enumerate(TARGETS):
        if r > N:
            continue
        assert int(out.status[i]) == 0, r
        _check_refined(xb[i], *out.window(i), sized["refs"][r], (r, refine))


@pytest.mark.gpu
def test_sized_dictionaries_one_d_singular_by_rank():
    from pyperiod_b200 import RamanujanPeriods
    x = synth.synth(N, SEED0)
    with pytest.raises(np.linalg.LinAlgError):
        RamanujanPeriods().find_periods_with_weights(x, max_length=8, refine=0,
                                                     test_function=lambda norms: SIZES[N + 1])


@pytest.mark.gpu
def test_sized_dictionaries_launch_plans(sized, monkeypatch):
    """Large dictionaries in two launches: up to 3000 rows the window is staged in shared memory, above it is read in
    place from global memory (one launch for all of them reads in place).  The weights do not change by a bit."""
    from pyperiod_b200 import ramanujan as ram_mod
    monkeypatch.setattr(ram_mod, "RMAX_TWO_CTAS", 3000)
    _same_bits(sized["base"], sized["solve"](0), len(TARGETS))


@pytest.mark.gpu
def test_sized_dictionaries_global_memory_path(sized):
    """pp_long_qo_solve runs the same cta_qo_solve on the same operands: bit-identical to the on-chip solve."""
    _same_bits(sized["base"], sized["solve"](0, staging="global"), len(TARGETS))


@pytest.mark.gpu
def test_sized_dictionaries_one_cta_solves_them_all(sized, monkeypatch):
    """A workspace with room for one factor: the grid shrinks to one CTA, which solves the windows of each launch one
    after the other on top of the previous window's factor storage.  The results do not change by a bit."""
    from pyperiod_b200 import _lib, qoperiods, ramanujan as ram_mod
    from pyperiod_b200._device import Workspace
    lib = _lib.load()
    seen = []
    real = ram_mod.qo_workspace

    def spy(lib_, dev, n, pmax, num, rmax, *a):
        ws = real(lib_, dev, n, pmax, num, rmax, *a)
        seen.append((ws.numel(), int(lib.pp_qo_workspace_bytes(n, pmax, num, rmax, 2, _lib.BASIS_NATURAL))))
        return ws
    monkeypatch.setattr(qoperiods, "WORKSPACE_FRACTION", 0.0)
    monkeypatch.setattr(ram_mod, "qo_workspace", spy)
    Workspace.release()      # a larger cached buffer would be reused as it is
    out = sized["solve"](0)
    Workspace.release()
    assert len(seen) == 2
    for got, two_ctas in seen:
        assert got < two_ctas       # room for one factor only: a grid of one CTA
    _same_bits(sized["base"], out, len(TARGETS))


@pytest.mark.gpu
def test_explicit_rows_refine0_gcd_goldens():
    """QOPeriodsWithGCDsExtracted solves an explicit layout (pp_qo_solve_rows); refine=0 meets the same bound."""
    from pyperiod_b200 import QOPeriodsWithGCDsExtracted as QG
    from pyperiod_b200.qoperiods import build_subspaces
    g = load_golden("qo_gcd")
    for i in range(4):
        seed, n, num, max_length = (int(v) for v in g[f"c{i}_args"])
        x = synth.synth(n, seed)
        d, res = QG().find_periods(x, num=num, thresh=float(g[f"c{i}_thresh"]), max_length=max_length or None,
                                   refine=0)
        lay = d["basis_dictionary"]
        assert [int(k) for k in lay] == g[f"c{i}_dict_keys"].tolist()
        ref = _reference(x, build_subspaces([int(k) for k in lay], list(lay.values()), n), lay)
        rw, rr = _check_refine0(x, d, res, ref, i)
        print(f"\ngcd case {i}: rows {len(d['weights'])} kappa {ref['kappa']:.1e} error / bound {rw:.2g} {rr:.2g}")


# ------------------------------------------------------------------ (2) the incremental factorisation
@pytest.fixture(scope="module")
def planted_windows():
    """Planted-period windows grouped by length, with the reference solution of each window's final dictionary."""
    groups = {}
    for n, qs, amps, seed, periods, rows in PLANTED:
        x = planted(n, qs, amps, seed)
        groups.setdefault(n, []).append((x, periods, rows, _reference(x, *oq.get_subspaces(periods, n))))
    return groups


@pytest.mark.gpu
@pytest.mark.parametrize("refine,staging", [(0, "auto"), (1, "auto"), (0, "global")])
def test_incremental_factor_equals_a_fresh_one(planted_windows, refine, staging):
    """find_periods grows each window's factor round by round.  Its weights and residual are bit-identical to one
    solve of the final period list from scratch: every factor row is computed from the same Gram counts and the same
    earlier rows in the same order, so any difference means a reused row is wrong."""
    from pyperiod_b200 import QOPeriods, RamanujanPeriods
    worst = 0.0
    for n, cases in planted_windows.items():
        xb = np.stack([c[0] for c in cases])
        out = QOPeriods(staging=staging).find_periods(xb, num=4, thresh=0.0, refine=refine)
        lists = iter([c[1] for c in cases])
        fresh = RamanujanPeriods(staging=staging).find_periods_with_weights(
            xb, max_length=4, refine=refine, test_function=lambda norms: next(lists))
        assert out.status.tolist() == fresh.status.tolist() == [0] * len(cases)
        for i, (x, periods, rows, ref) in enumerate(cases):
            d, res = out.window(i)
            assert [int(p) for p in d["periods"]] == periods
            assert int(out.n_weights[i]) == rows[-1]
            df, rf = fresh.window(i)
            assert d["basis_dictionary"] == df["basis_dictionary"] == ref["layout"]
            assert np.array_equal(d["weights"], df["weights"]), (n, periods)
            assert np.array_equal(res, rf), (n, periods)
            if refine == 0:
                rw, rr = _check_refine0(x, d, res, ref, (n, periods))
                worst = max(worst, rw, rr)
            else:
                _check_refined(x, d, res, ref, (n, periods))
    if refine == 0:
        print(f"\nincremental refine=0 staging={staging}: worst error / bound {worst:.2g}")
