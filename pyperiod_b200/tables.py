"""Host-built integer side tables for the device kernels.

The reference iterates Python `set`s of divisors directly (pyPeriod/Periods.py:73-84,
209-210, 548-549), so CPython's hash-table iteration order decides (a) the order in
which prime cofactors are projected out when orthogonalising and (b) which divisor is
"last" in M-best step 2.  The tables are therefore produced by evaluating the same set
expression in this interpreter -- never re-derived on the device.
"""
from __future__ import annotations

from functools import lru_cache

import numpy as np

PRIME_LIMIT = 10000  # reference PRIMES = primes <= 10000 (Periods.py:121)


def _divisor_set(n: int) -> set:
    seq = []
    for i in range(1, int(n ** 0.5) + 1):
        if n % i == 0:
            seq += [i, n // i]
    return set(seq)


def nontrivial_factors(n: int) -> list:
    """Divisors of n except 1 and n, in the reference's set-iteration order."""
    s = _divisor_set(int(n))
    s.discard(1)
    s.discard(int(n))
    return list(s)


@lru_cache(maxsize=None)
def _primes() -> frozenset:
    flags = np.ones(PRIME_LIMIT + 1, dtype=bool)
    flags[:2] = False
    for i in range(2, int(PRIME_LIMIT ** 0.5) + 1):
        if flags[i]:
            flags[i * i:: i] = False
    return frozenset(np.flatnonzero(flags).tolist())


def orth_chain(p: int) -> list:
    """Cofactors p//f for prime divisors f of p (f <= 10000), in the reference's loop order."""
    if p < 2:
        return []
    pr = _primes()
    return [int(p / f) for f in nontrivial_factors(p) if f in pr]


def euler_phi_table(nmax: int) -> np.ndarray:
    """phi[0..nmax] by a sieve (values equal the reference's gcd-count phi, QOPeriods.py:16-43)."""
    phi = np.arange(nmax + 1, dtype=np.int64)
    for p in range(2, nmax + 1):
        if phi[p] == p:  # prime
            phi[p::p] -= phi[p::p] // p
    phi[0] = 0
    return phi.astype(np.int32)


def moebius_table(nmax: int) -> np.ndarray:
    """mu[0..nmax] (mu[0] = 0) by a linear sieve."""
    mu = np.ones(nmax + 1, dtype=np.int32)
    mu[0] = 0
    is_comp = np.zeros(nmax + 1, dtype=bool)
    for p in range(2, nmax + 1):
        if not is_comp[p]:
            is_comp[2 * p:: p] = True
            mu[p:: p] *= -1
            mu[p * p:: p * p] = 0
    return mu


def smallest_prime_factor_table(nmax: int) -> np.ndarray:
    """spf[0..nmax] (spf[0] = 0, spf[1] = 1): the distinct primes of q follow in O(log q) steps (q /= spf[q])."""
    spf = np.zeros(nmax + 1, dtype=np.int32)
    if nmax >= 1:
        spf[1] = 1
    for p in range(2, int(nmax ** 0.5) + 1):
        if spf[p] == 0:
            blk = spf[p * p:: p]
            blk[blk == 0] = p
    rest = np.flatnonzero(spf == 0)
    spf[rest[rest >= 2]] = rest[rest >= 2]
    return spf


def _nontrivial_factor_lists(pmax: int) -> list:
    """nontrivial_factors(n) for every n in 0..pmax, by a sieve.  Each n receives the same insertion sequence as
    _divisor_set builds (every divisor i <= sqrt(n) in ascending order, immediately followed by n // i), so set()
    iterates the divisors in the same order as the per-n expression (load-bearing, SURVEY.md 8a row 3)."""
    seqs = [[] for _ in range(pmax + 1)]
    i = 1
    while i * i <= pmax:
        for n in range(i * i, pmax + 1, i):
            seqs[n] += (i, n // i)
        i += 1
    out = []
    for n, seq in enumerate(seqs):
        s = set(seq)
        s.discard(1)
        s.discard(n)
        out.append(list(s))
    return out


class PeriodTables:
    """CSR tables for all periods 0..pmax, as numpy int32 (host) and cached device tensors."""

    def __init__(self, pmax: int):
        self.pmax = int(pmax)
        chain_off = np.zeros(self.pmax + 2, dtype=np.int32)
        fac_off = np.zeros(self.pmax + 2, dtype=np.int32)
        chain, fac = [], []
        factors = _nontrivial_factor_lists(self.pmax)
        pr = _primes()
        for p in range(self.pmax + 1):
            if p >= 2:
                fs = factors[p]
                fac.extend(fs)
                chain.extend(int(p / f) for f in fs if f in pr)
            chain_off[p + 1] = len(chain)
            fac_off[p + 1] = len(fac)
        self.chain_off = chain_off
        self.fac_off = fac_off
        self.chain_q = np.asarray(chain if chain else [0], dtype=np.int32)
        self.fac = np.asarray(fac if fac else [0], dtype=np.int32)
        self.phi = euler_phi_table(self.pmax)
        self.mu = moebius_table(self.pmax)
        self.spf = smallest_prime_factor_table(self.pmax)
        self._dev = {}
        self._dev_phi = {}

    def chain_of(self, p: int) -> np.ndarray:
        return self.chain_q[self.chain_off[p]: self.chain_off[p + 1]]

    def factors_of(self, p: int) -> np.ndarray:
        return self.fac[self.fac_off[p]: self.fac_off[p + 1]]

    def phi_device(self, device):
        """Euler phi table as a torch int32 tensor on `device` (cached)."""
        import torch
        key = str(device)
        if key not in self._dev_phi:
            self._dev_phi[key] = torch.from_numpy(self.phi).to(device)
        return self._dev_phi[key]

    def mu_device(self, device):
        """Moebius table as a torch int32 tensor on `device` (cached)."""
        import torch
        key = "mu:" + str(device)
        if key not in self._dev_phi:
            self._dev_phi[key] = torch.from_numpy(self.mu).to(device)
        return self._dev_phi[key]

    def spf_device(self, device):
        """Smallest-prime-factor table as a torch int32 tensor on `device` (cached)."""
        import torch
        key = "spf:" + str(device)
        if key not in self._dev_phi:
            self._dev_phi[key] = torch.from_numpy(self.spf).to(device)
        return self._dev_phi[key]

    def device(self, device):
        """Tuple of torch int32 tensors (chain_off, chain_q, fac_off, fac) on `device` (cached)."""
        import torch
        key = str(device)
        if key not in self._dev:
            self._dev[key] = tuple(torch.from_numpy(a).to(device) for a in
                                   (self.chain_off, self.chain_q, self.fac_off, self.fac))
        return self._dev[key]


_CACHE: dict = {}


def get_tables(pmax: int) -> PeriodTables:
    """Tables covering at least pmax (rounded up so repeated calls with nearby pmax share one table)."""
    want = max(1024, 1 << (int(pmax) - 1).bit_length())
    if want not in _CACHE:
        _CACHE[want] = PeriodTables(want)
    return _CACHE[want]
