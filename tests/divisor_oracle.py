"""Divisor form of the fp64 Ramanujan periodogram (test infrastructure, a cross-check only: SURVEY.md 8d).

c_q(n) = sum_{d | gcd(n, q)} mu(q / d) d, so the circulant product of the closed form is
    (H S_q)_m = sum_l c_q(l - m) S_q[l] = sum_{d | q} mu(q / d) d S_d[m mod d],
with S_d the fold of S_q down to period d.  That costs O(N + q tau(q)) per period instead of the O(q^2) of
oracle.ramanujan.norms_closed_form_f64 (whose value it equals to rounding), so long windows can be checked on the CPU.
"""
from __future__ import annotations

import numpy as np

from oracle.numtheory import phi


def _mobius_table(n: int) -> np.ndarray:
    mu = np.ones(n + 1, dtype=np.int64)
    mu[0] = 0
    is_p = np.ones(n + 1, dtype=bool)
    for p in range(2, n + 1):
        if is_p[p]:
            is_p[2 * p::p] = False
            mu[p::p] *= -1
            mu[p * p::p * p] = 0
    return mu


def norms_divisor_form_f64(x, min_length: int = 2, max_length=None, periods=None) -> np.ndarray:
    """Norms [max_length + 1] (zero below min_length); `periods` restricts the work to those q (others stay 0)."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    if not max_length:
        max_length = n // 3
    mu = _mobius_table(max_length)
    idx = np.arange(n)
    norms = np.zeros(max_length + 1)
    qs = range(min_length, max_length + 1) if periods is None else [int(q) for q in periods]
    for q in qs:
        s = np.bincount(idx % q, weights=x, minlength=q)
        cnt = np.bincount(idx % q, minlength=q).astype(np.float64)
        z = np.zeros(q)
        small = [d for d in range(1, int(np.sqrt(q)) + 1) if q % d == 0]
        for d in sorted(set(small + [q // d for d in small])):
            if mu[q // d] == 0:
                continue
            sd = s.reshape(q // d, d).sum(0)
            z += (mu[q // d] * d) * np.tile(sd, q // d)
        ph = float(phi(q))
        scale = q / (ph * ph)
        norms[q] = np.sum(cnt * (scale * z) ** 2)
    return norms
