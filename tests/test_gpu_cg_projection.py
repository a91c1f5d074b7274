"""The conjugate-gradient projections (csrc/pp_cg.cuh) against an explicit matrix and a thin SVD.

Two places project a vector t onto the row space of an implicit dictionary A whose Gram matrix A A^T is singular by
construction, and return t minus that projection (and, for the Ramanujan basis, the minimum-norm weights):

- QOPeriods.get_periods (gp_kernel, csrc/pp_extract.cu): A = the pairwise-GCD rows, t = the zero-padded weights;
- QOPeriods(basis_type="ramanujan").find_periods (cta_qo_solve_ram, csrc/pp_qo.cuh), on chip and on the global-memory
  path: A = shifted integer Ramanujan sums c_q((n - i) mod q), t = the window.

The reference takes a thin SVD A = U S V^T in float64 and the rank r at a checked gap (sigma_{r+1} / sigma_1 < 1e-12,
sigma_r / sigma_1 > 1e-8): res* = t - V_r^T V_r t and w* = U_r S_r^-1 V_r^T t, evaluated in extended precision.  CG
stops at |A e|^2 <= 1e-29 |A t|^2 with e = res - res* in the row space, so with u = 2^-53 and
kappa+ = sigma_1 / sigma_r:

    |res - res*|_2 <= 64 u kappa+ |t|_2,      |w - w*|_2 <= 64 u kappa+^2 |t|_2 / sigma_1

and the two outputs agree with each other: |t - A^T w - res|_2 <= 64 u |t|_2.  The dictionaries reach the shapes where
the implicit operators branch (odd q and odd row counts in the two-accumulator loops of RamBasisOp, repeated and divisor
periods that take all q rows, q = 4 whose rows 0 and 2 are exact negatives), row counts from 0.03 N to 0.92 N, and the
iteration budget: 1365, 1364, 1024 at N = 4096 needs about 1040 steps in one pass.
"""
import contextlib
import io
import math

import numpy as np
import pytest

from oracle import qo as oq
from oracle.numtheory import phi
from oracle.periods import periodic_norm, project
from pyperiod_b200 import synth

U = 2.0 ** -53
SLACK = 64.0


# ------------------------------------------------------------------ the dictionaries, explicitly
def mobius(n: int) -> int:
    res, d = 1, 2
    while d * d <= n:
        if n % d == 0:
            n //= d
            if n % d == 0:
                return 0
            res = -res
        d += 1
    return -res if n > 1 else res


def ramanujan_sum_int(q: int) -> np.ndarray:
    """c_q(m), m < q, exactly: mu(q/g) phi(q) / phi(q/g), g = gcd(m, q)."""
    g = np.gcd(np.arange(q), q)
    g[0] = q
    return np.array([mobius(q // int(d)) * (phi(q) // phi(q // int(d))) for d in g], dtype=np.float64)


def ramanujan_rows_int(q: int, n: int, keep) -> np.ndarray:
    """Rows c_q((m - i) mod q), m < n, i < keep; keep == 0 keeps all q rows (QOPeriods.py:972)."""
    c = ramanujan_sum_int(q)
    rows = c[(np.arange(n)[None, :] - np.arange(q)[:, None]) % q]
    return rows[:keep] if keep else rows


def ramanujan_matrix(layout: dict, n: int) -> np.ndarray:
    return np.vstack([np.zeros((0, n))] + [ramanujan_rows_int(int(q), n, k) for q, k in layout.items()])


def reference(a: np.ndarray, t: np.ndarray) -> dict:
    """Thin SVD of `a`, rank at the gap, and the projection residual and minimum-norm weights of `t`."""
    u, s, vt = np.linalg.svd(a, full_matrices=False)
    r = int(np.count_nonzero(s > 1e-10 * s[0]))
    below = float(s[r] / s[0]) if r < len(s) else 0.0
    ur, vr = u[:, :r].astype(np.longdouble), vt[:r].astype(np.longdouble)
    tl = t.astype(np.longdouble)
    c = vr @ tl
    return dict(rank=r, shape=a.shape, kappa=float(s[0] / s[r - 1]), sigma1=float(s[0]), below=below,
                above=float(s[r - 1] / s[0]), res=tl - vr.T @ c, w=ur @ (c / s[:r].astype(np.longdouble)),
                tnorm=float(np.linalg.norm(t)))


def clear_gap(ref) -> bool:
    return ref["below"] < 1e-12 and ref["above"] > 1e-8


def check_projection(res, ref, what, w=None, a=None, t=None):
    """Residual (and weights) within the bound; returns the errors as fractions of their bounds."""
    er = float(np.linalg.norm((res - ref["res"]).astype(np.float64)))
    br = SLACK * U * ref["kappa"] * ref["tnorm"]
    assert er <= br, (what, "residual", er, br, ref["kappa"])
    out = [er / br]
    if w is not None:
        assert len(w) == ref["shape"][0], what
        ew = float(np.linalg.norm((w - ref["w"]).astype(np.float64)))
        bw = SLACK * U * ref["kappa"] ** 2 * ref["tnorm"] / ref["sigma1"]
        assert ew <= bw, (what, "weights", ew, bw, ref["kappa"])
        ec = float(np.linalg.norm(t - a.T @ w - res))
        assert ec <= SLACK * U * ref["tnorm"], (what, "t - A^T w - res", ec)
        out += [ew / bw]
    return out


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


# ------------------------------------------------------------------ QOPeriods.get_periods layouts
def rand_weights(layout: dict, seed: int) -> np.ndarray:
    return np.random.default_rng(seed).standard_normal(sum(layout.values()))


GETP_LAYOUTS = {
    "coprime pair": {"35": 35, "64": 64},
    "g = q_a": {"12": 12, "36": 36},
    "chain": {"4": 4, "8": 8, "16": 16, "32": 32},
    "composite a": {"60": 60, "84": 84, "90": 90, "126": 126, "140": 140},
    "composite b": {"360": 360, "240": 240, "180": 180, "120": 120, "72": 72},
    "coprime triple": {"7": 7, "11": 11, "13": 13},
    "coprime triple 2": {"8": 8, "9": 9, "25": 25},
    "97 multiples": {"97": 97, "194": 194, "291": 291},
    "keep < q": {"30": 20, "42": 17, "70": 0, "105": 104},
    "64 periods": {str(q): q for q in range(2, 66)},
}


def gp_plan_bytes(periods, kthreads=256):
    """Shared memory of gp_kernel (GpPlan::bytes, csrc/pp_extract.cu): 2 T + 3 R doubles, reduction, integers."""
    k = len(periods)
    t = sum(periods)
    r = sum(math.gcd(a, b) for i, a in enumerate(periods) for b in periods[i + 1:])
    ev = lambda v: (max(v, 2) + 1) & ~1
    return 8 * (2 * ev(t) + 3 * ev(r)) + 2 * (kthreads // 32) * 8 + (2 * k + k * (k - 1) + 6) * 4 + 16


def pair_near(limit: int, over: bool):
    """A pair (g, g (s - 1)), gcd g, whose gp_kernel plan is the largest <= limit (over=False) or smallest > limit."""
    best = None
    for g in range(2, 600):
        for s in range(3, limit // (16 * g) + 3):
            b = gp_plan_bytes([g, g * (s - 1)])
            ok = b > limit if over else b <= limit
            if ok and (best is None or (b < best[0] if over else b > best[0])):
                best = (b, g, g * (s - 1))
    return best


# ------------------------------------------------------------------ Ramanujan-basis find_periods windows
def c_q_pattern(q: int, rng) -> np.ndarray:
    """A random pattern of length q inside the span of the shifts of c_q, unit RMS."""
    c = ramanujan_sum_int(q)
    w = rng.standard_normal(q)
    pat = np.array([np.dot(w, c[(m - np.arange(q)) % q]) for m in range(q)])
    return pat / np.sqrt(np.mean(pat ** 2))


def planted(n, periods, amps, seed):
    """Sum of a_k * (a pattern in the c_q span of period q_k, tiled) plus 1e-3 white noise."""
    rng = np.random.default_rng(seed)
    x = 1e-3 * rng.standard_normal(n)
    for q, a in zip(periods, amps):
        x += a * np.tile(c_q_pattern(q, rng), n // q + 1)[:n]
    return x


# Groups share (N, num, min_length) and run as one batch.  Each window: its signal and the period sequence with the
# dictionary find_periods(thresh=0.0) reaches (checked on the CPU).  The rows per entry (odd / even q, odd / even rows):
#   s1     11 (odd, odd) 15 -> 14 (odd, even) 25 -> 20, 3 -> all 3 rows (a divisor of 15: keep == 0); N = 1009 prime:
#          no q divides N
#   s2     12 -> 12 (even, even) 15 -> 12, 5 -> all 5 rows (keep == 0; odd, odd), 6 -> all 6 rows (keep == 0; even,
#          even); R / N = 0.035
#   m1     256 (rows i and i + 128 exact negatives), 37 -> 36, 26 -> 24
#   m2     341, 31 -> all 31 rows (keep == 0), 340 -> 339 (even, odd); R / N = 0.69
#   t1024  341, 340 -> 339, 256 -> 252: R = 932 = 0.91 N, about 470 CG steps
#   big    1365, 1364 -> 1363, 1024 -> 1020: R = 3748 = 0.92 N, about 1040 CG steps in one pass
#   q4     4 -> all 4 rows (rows 0 and 2, 1 and 3 exact negatives), 15 -> 14, 35 -> 30
#   mix    a synth window (276 rows), s1's periods at N = 4096, and 1201, 1303, 1109: R = 3611, kappa+ = 2e4
GROUPS = {
    "small": dict(n=1009, num=4, min_length=2, windows={
        "s1": ((11, 15, 25), (1.0, 0.8, 0.6), 4, [11, 15, 25, 3]),
        "s2": ((12, 6, 15, 5), (3.0, 1.0, 2.0, 1.0), 6, [12, 15, 5, 6]),
    }),
    "mid": dict(n=1024, num=3, min_length=2, windows={
        "m1": ((341, 340, 256), (1.0, 1.0, 1.0), 3, [256, 37, 26]),
        "m2": ((341, 340, 256), (3.0, 2.0, 1.0), 32, [341, 31, 340]),
    }),
    "t1024": dict(n=1024, num=3, min_length=200, windows={
        "t1024": ((341, 340, 256), (3.0, 2.0, 1.0), 3, [341, 340, 256]),
    }),
    "big": dict(n=4096, num=3, min_length=1000, windows={
        "big": ((1365, 1364, 1024), (3.0, 2.0, 1.0), 1, [1365, 1364, 1024]),
    }),
    "q4": dict(n=2050, num=3, min_length=2, windows={
        "q4": ((4, 15, 35), (2.0, 3.0, 2.0), 45, [4, 15, 35]),
    }),
    "mix": dict(n=4096, num=3, min_length=2, windows={
        "synth": (None, None, 50_001, [26, 70, 183]),
        "s4096": ((11, 15, 25), (1.0, 0.8, 0.6), 7, [11, 15, 25]),
        "guard": ((1201, 1303, 1109), (3.0, 2.0, 1.0), 2, [1201, 1303, 1109]),
    }),
}
# windows whose last dictionary does not converge within the budget: the find reports PP_STATUS_GUARD and keeps the
# previous round (this many periods)
GUARD = {"guard": 2}
# windows on which the reference's np.linalg.solve does not deliver the projection, so its loop takes another path:
#   m1  the 256 rows of c_256 come in exactly opposite pairs; the LU goes through with weights of 1e12 and a residual
#       off by more than |x| after round 1, and the reference's next round finds 39 where the projection's gives 37;
#   q4  the LU stops on the opposite rows of c_4 with a LinAlgError.
# Their sequences are those of the same loop with the exact projection (exact_find), which is what CG computes.
EXACT_ONLY = ("m1", "q4")


def window_signal(n, spec):
    qs, amps, seed, _ = spec
    return synth.synth(n, seed) if qs is None else planted(n, qs, amps, seed)


def layout_of(periods, n):
    return quiet(oq.get_subspaces, [int(p) for p in periods], 8, "natural")[1]


def exact_find(x, num, min_length):
    """The reference loop (gamma sweep, thresh 0) with the exact orthogonal projection in place of np.linalg.solve."""
    n, found = len(x), []
    res = x.copy()
    for _ in range(num):
        best_p, best = 0, 0.0
        for p in range(min_length, n // 3 + 1):
            v = periodic_norm(project(res, p), p)
            if v > best:
                best_p, best = p, v
        found.append(best_p)
        _, s, vt = np.linalg.svd(ramanujan_matrix(layout_of(found, n), n), full_matrices=False)
        vr = vt[: int(np.count_nonzero(s > 1e-10 * s[0]))]
        res = x - vr.T @ (vr @ x)
    return found


@pytest.fixture(scope="module")
def ram_cases():
    """Per window: signal, expected periods, final layout and the SVD reference of the dictionary it ends with."""
    out = {}
    for gname, g in GROUPS.items():
        for wname, spec in g["windows"].items():
            x = window_signal(g["n"], spec)
            periods = spec[3][: GUARD.get(wname, len(spec[3]))]
            lay = layout_of(periods, g["n"])
            a = ramanujan_matrix(lay, g["n"])
            out[wname] = dict(group=gname, x=x, periods=periods, layout=lay, a=a, ref=reference(a, x))
    return out


@pytest.fixture(scope="module")
def getp_refs():
    out = {}
    for i, (name, lay) in enumerate(GETP_LAYOUTS.items()):
        w = rand_weights(lay, 500 + i)
        t = oq.concatenate_periods(w, lay)
        out[name] = dict(layout=lay, w=w, ref=reference(oq.pairwise_gcd_rows([int(q) for q in lay]), t))
    return out


# ------------------------------------------------------------------ CPU: the reference checks itself
def test_integer_ramanujan_rows_are_the_references():
    """The exact rows against the reference's sums of complex exponentials (rounding noise of about 1e-14 phi(q)) and
    against the package's host copy (bit for bit)."""
    from pyperiod_b200 import qoperiods
    for q, n, keep in [(1, 5, 0), (2, 7, 1), (3, 9, 0), (4, 10, 3), (5, 12, 0), (6, 13, 2), (12, 40, 0), (15, 47, 14),
                       (30, 91, 8), (97, 300, 96), (210, 500, 0), (360, 800, 96), (341, 1024, 0)]:
        a = ramanujan_rows_int(q, n, keep)
        np.testing.assert_allclose(a, oq.ramanujan_rows(q, n, keep), rtol=0, atol=1e-12 * max(1, phi(q) // 8))
        assert np.array_equal(a, qoperiods.ramanujan_rows(q, n, keep)), q
    c4 = ramanujan_rows_int(4, 8, 0)
    assert np.array_equal(c4[0], -c4[2]) and np.array_equal(c4[1], -c4[3])


def test_every_dictionary_has_a_clear_rank_gap(ram_cases, getp_refs):
    """A dictionary without a clear gap between its nonzero and zero singular values has no well-defined rank and is
    not a valid test case."""
    refs = {k: v["ref"] for k, v in ram_cases.items()}
    refs.update({k: v["ref"] for k, v in getp_refs.items()})
    # the final dictionaries of the windows that report GUARD: the table's fourth row
    g = GROUPS["mix"]
    full = ramanujan_matrix(layout_of(g["windows"]["guard"][3], g["n"]), g["n"])
    refs["guard, all three"] = reference(full, ram_cases["guard"]["x"])
    for name, ref in refs.items():
        assert clear_gap(ref), (name, ref["below"], ref["above"])
    assert refs["guard, all three"]["shape"] == (3611, 4096) and refs["guard, all three"]["rank"] == 3610
    assert refs["guard, all three"]["kappa"] > 1e4
    assert ram_cases["big"]["ref"]["shape"] == (3748, 4096) and ram_cases["big"]["ref"]["rank"] == 1688
    assert ram_cases["t1024"]["ref"]["shape"] == (932, 1024)
    assert getp_refs["64 periods"]["ref"]["shape"] == (4844, 2144)
    print("\nrank / rows / kappa+:", {k: (r["rank"], r["shape"][0], "%.3g" % r["kappa"]) for k, r in refs.items()})


def test_planted_sequences_match_the_oracle(ram_cases):
    """The expected period sequences are what the reference's loop finds (the windows of EXACT_ONLY: the same loop with
    the exact projection)."""
    for gname, g in GROUPS.items():
        for wname, spec in g["windows"].items():
            x = ram_cases[wname]["x"]
            if wname in EXACT_ONLY:
                got = exact_find(x, g["num"], g["min_length"])
            else:
                d, _ = quiet(oq.find_periods, x, num=g["num"], thresh=0.0, min_length=g["min_length"],
                             basis="ramanujan")
                got = [int(p) for p in d["periods"]]
                assert d["basis_dictionary"] == layout_of(spec[3], g["n"]), wname
            assert got == spec[3], (wname, got)
    # the shapes the operators branch on are all present
    lays = [c["layout"] for c in ram_cases.values()]
    kinds = {(int(q) % 2, (k or int(q)) % 2) for lay in lays for q, k in lay.items()}
    assert kinds == {(0, 0), (0, 1), (1, 0), (1, 1)}
    assert any(k == 0 and int(q) % 2 for lay in lays for q, k in lay.items())
    assert any(k == 0 and int(q) % 2 == 0 for lay in lays for q, k in lay.items())
    assert ram_cases["q4"]["layout"]["4"] == 4
    assert all(g["n"] % int(q) for g in (GROUPS["small"],) for w in g["windows"].values() for q in w[3])


def test_pair_near_the_shared_memory_limit():
    for limit in (232448, 101376):
        at, over = pair_near(limit, False), pair_near(limit, True)
        assert limit - 16 < at[0] <= limit < over[0] <= limit + 24


# ------------------------------------------------------------------ GPU: get_periods
@pytest.mark.gpu
def test_get_periods_layouts_within_bound(getp_refs):
    from pyperiod_b200 import QOPeriods
    worst = {}
    for name, c in getp_refs.items():
        gp = QOPeriods().get_periods(c["w"], c["layout"], "lstsq")
        assert [len(v) for v in gp] == [int(q) for q in c["layout"]], name
        worst[name] = check_projection(np.concatenate(gp), c["ref"], name)[0]
    print("\nget_periods error / bound:", {k: "%.2g" % v for k, v in worst.items()})


@pytest.mark.gpu
def test_get_periods_period_count_limit():
    from pyperiod_b200 import QOPeriods, _lib
    lay = {str(q): q for q in range(2, 67)}
    with pytest.raises(_lib.PPError):
        QOPeriods().get_periods(rand_weights(lay, 9), lay, "lstsq")


@pytest.mark.gpu
def test_get_periods_at_the_shared_memory_limit():
    """The largest pair whose plan fits runs within the bound; the smallest that does not fit raises."""
    import torch
    from pyperiod_b200 import QOPeriods, _lib
    from pyperiod_b200.periods import smem_optin
    limit = smem_optin(torch.device("cuda", torch.cuda.current_device()))
    (_, ga, gb), (_, oa, ob) = pair_near(limit, False)[:3], pair_near(limit, True)[:3]
    lay = {str(ga): ga, str(gb): gb}
    w = rand_weights(lay, 11)
    gp = QOPeriods().get_periods(w, lay, "lstsq")
    ref = reference(oq.pairwise_gcd_rows([ga, gb]), oq.concatenate_periods(w, lay))
    assert clear_gap(ref)
    check_projection(np.concatenate(gp), ref, lay)
    lay = {str(oa): oa, str(ob): ob}
    with pytest.raises(_lib.PPError):
        QOPeriods().get_periods(rand_weights(lay, 12), lay, "lstsq")


@pytest.mark.gpu
def test_get_periods_batch_ragged_dictionaries():
    """The batch form on a find_periods result whose windows hold 1 (the mean branch) to 4 periods: every window within
    the bound and bit-identical to the reference-form call."""
    from pyperiod_b200 import QOPeriods
    rng = np.random.default_rng(77)
    xb = np.stack([rng.standard_normal(1024), synth.synth(1024, 50_011), synth.synth(1024, 50_012),
                   rng.standard_normal(1024), synth.synth(1024, 50_013)])
    r = QOPeriods().find_periods(xb, num=4, thresh=0.3, max_length=200)
    nd = np.asarray(r.n_dict).tolist()
    assert 1 in nd and 4 in nd, nd
    pb = QOPeriods().get_periods(r)
    assert np.asarray(pb.status).tolist() == [0] * len(xb)
    worst = 0.0
    for b in range(len(xb)):
        d, _ = r.window(b)
        lay = d["basis_dictionary"]
        got = pb.window(b)
        one = QOPeriods().get_periods(d["weights"], lay, "lstsq")
        assert len(got) == len(one) == len(lay)
        for u, v in zip(got, one):
            assert np.array_equal(u, v), b
        ref = reference(oq.pairwise_gcd_rows([int(q) for q in lay]), oq.concatenate_periods(d["weights"], lay))
        assert clear_gap(ref), b
        worst = max(worst, check_projection(np.concatenate(got), ref, b)[0])
    print(f"\nget_periods batch: worst error / bound {worst:.2g}")


# ------------------------------------------------------------------ GPU: Ramanujan-basis find_periods
def run_group(gname, cases, staging, names=None):
    from pyperiod_b200 import QOPeriods
    g = GROUPS[gname]
    names = list(g["windows"]) if names is None else names
    xb = np.stack([cases[w]["x"] for w in names])
    out = QOPeriods(basis_type="ramanujan", staging=staging).find_periods(
        xb, num=g["num"], thresh=0.0, min_length=g["min_length"])
    return names, out


def check_window(out, b, case, what):
    from pyperiod_b200 import _lib
    want = _lib.STATUS_GUARD if what[0] in GUARD else _lib.STATUS_OK
    assert int(out.status[b]) == want, (what, int(out.status[b]))
    d, res = out.window(b)
    assert [int(p) for p in d["periods"]] == case["periods"], what
    assert d["basis_dictionary"] == case["layout"], what
    return check_projection(res, case["ref"], what, w=d["weights"], a=case["a"], t=case["x"])


@pytest.mark.gpu
@pytest.mark.parametrize("staging", ["shared", "global"])
def test_ramanujan_find_within_bound(ram_cases, staging):
    worst = [0.0, 0.0]
    for gname in GROUPS:
        names, out = run_group(gname, ram_cases, staging)
        for b, w in enumerate(names):
            ratios = check_window(out, b, ram_cases[w], (w, staging))
            worst = [max(a, r) for a, r in zip(worst, ratios)]
    print(f"\nRamanujan find staging={staging}: worst error / bound residual {worst[0]:.2g} weights {worst[1]:.2g}")


@pytest.mark.gpu
@pytest.mark.parametrize("staging", ["shared", "global"])
def test_ramanujan_find_large_neighbours_change_nothing(ram_cases, staging):
    """Small dictionaries batched with a large one (which the first launch cannot hold and which reports GUARD) give the
    bits they give alone."""
    names, out = run_group("mix", ram_cases, staging)
    for b, w in enumerate(names):
        _, one = run_group("mix", ram_cases, staging, [w])
        assert int(out.status[b]) == int(one.status[0]), w
        d, res = out.window(b)
        d1, res1 = one.window(0)
        assert d["basis_dictionary"] == d1["basis_dictionary"], w
        assert np.array_equal(d["weights"], d1["weights"]), w
        assert np.array_equal(res, res1), w
