"""The error bound of the fp32 nomination sweep (pp_sweep.cuh: f32_energy_tol) against a numpy emulation of the
float fold at the sweep's tile shapes, with the residual's own energy as the scale of the bound."""
import math

import numpy as np

from pyperiod_b200 import synth

U = 2.0 ** -24
TILE_TERMS = 24   # kF32TileTerms
# (sets, columns) of every level a float tile evaluates: tops q = g 2^L (2^L sets of 8 >> L columns, levels 2^i <= 2^L,
# masked remainders at half the width), hosts of a rider (2^i sets of 2 columns) and riders (3 * 2^i sets of 2 columns)
SHAPES = sorted({(1 << i, max(8 >> L, 1) // w or 1) for L in range(4) for i in range(L + 1) for w in (1, 2)} |
                {(1 << i, 2) for i in range(3)} | {(3 << i, 2) for i in range(2)})


def f32_energy_tol(n, p, e):
    m, c = n // p, -(-n // p)
    terms = 2.0 * c + TILE_TERMS * (m + 2) / m
    return 2.0 * (terms * U * e + 2.0 ** -149 * (n + p + e))


def float_key(x32, p, sets, cols):
    """Energy of candidate p as the float sweep forms it: residue sums in float, then per lane and tile of `cols`
    pairs of base residues the squares of every set summed in float, the tile partials summed in double."""
    n = x32.size
    m, rr = n // p, n % p
    s = np.zeros(p, np.float32)
    for k in range(m):
        s += x32[k * p:(k + 1) * p]
    s[:rr] += x32[m * p:]
    g = p // sets
    width = 64 * cols
    gp = -(-g // width) * width
    v = np.zeros((sets, gp), np.float32)
    v[:, :g] = s.reshape(sets, g)                     # residue r + g t of p is base residue r of set t
    tail = np.zeros((sets, gp), bool)
    tail[:, :g] = (np.arange(p) < rr).reshape(sets, g)
    sq = (v * v).reshape(sets, gp // width, cols, 32, 2)
    tl = tail.reshape(sets, gp // width, cols, 32, 2)
    t = np.zeros((gp // width, 32), np.float32)
    a = np.zeros((gp // width, 32), np.float32)
    for si in range(sets):
        for j in range(cols):
            for c in range(2):
                t += sq[si, :, j, :, c]
                a += np.where(tl[si, :, j, :, c], sq[si, :, j, :, c], np.float32(0))
    tt, aa = float(t.astype(np.float64).sum()), float(a.astype(np.float64).sum())
    return tt / m + (1.0 / (m + 1) - 1.0 / m) * aa


def exact_key(x, p):
    idx = np.arange(x.size) % p
    cnt = np.bincount(idx, minlength=p).astype(np.float64)
    s = np.bincount(idx, weights=x, minlength=p)
    return float((s * s / cnt).sum())


def residual(x, p):
    idx = np.arange(x.size) % p
    mean = np.bincount(idx, weights=x, minlength=p) / np.bincount(idx, minlength=p)
    return x - mean[idx]


def worst_ratio(x, periods):
    e = float((x * x).sum())
    assert x.size * e <= 2.0 ** 120
    x32 = x.astype(np.float32)
    worst = 0.0
    for p in periods:
        want = exact_key(x, p)
        for sets, cols in SHAPES:
            if p % sets or (p // sets) < 1:
                continue
            got = float_key(x32, p, sets, cols)
            worst = max(worst, abs(got - want) / f32_energy_tol(x.size, p, e))
    return worst


PERIODS = [2, 3, 6, 24, 96, 241, 255, 383, 512, 576, 700, 768, 1000, 1023, 1024]


def test_shapes_cover_the_tile_terms():
    assert max(2 * s * c for s, c in SHAPES) == TILE_TERMS


def test_bound_holds_round_by_round():
    """Each sweep's bound scales with its residual's energy: three rounds of projecting out the strongest period."""
    x = synth.synth(4096, 32_000)
    for _ in range(3):
        assert worst_ratio(x, PERIODS) < 0.5
        best = max(range(2, 1025), key=lambda p: exact_key(x, p))
        x = residual(x, best)


def test_bound_holds_over_a_large_dynamic_range():
    rng = np.random.default_rng(32_001)
    n = 4096
    x = synth.synth(n, 32_002) * 10.0 ** rng.uniform(-50, 15, n)   # float subnormals and flushes to zero included
    assert worst_ratio(x, PERIODS) < 0.5
    y = rng.standard_normal(n) * 1e-40                              # a window entirely below the float normals
    y[::97] = 1e3
    assert worst_ratio(y, PERIODS) < 0.5


def test_bound_holds_with_every_residue_under_the_tail_row():
    """N mod p = p - 1: all residues but one hold one more sample, and the tail row carries most of the energy."""
    for n, periods in ((4096, [17, 241]), (2999, [1000, 500, 250, 125]), (4095, [512, 1024, 256, 128, 64])):
        x = synth.synth(n, 32_003 + n)
        for p in periods:
            assert n % p == p - 1
            y = x.copy()
            y[(n // p) * p:] *= 1e4
            assert worst_ratio(y, [p]) < 0.5
            assert math.isfinite(worst_ratio(y * 1e-20, [p]))
