"""The root placement support statistics (DESIGN.md section 10) restated with numpy and Python
integers, item by item, for the tests: numpy.random.Philox gives the draws, Python ints the exact
sums.  Input: per partition (in global order) its rows L [records][patterns] and pattern weights."""
from __future__ import annotations

import math

import numpy as np


def exponent_of(rows) -> int:
    M = max((float(np.max(np.abs(L))) for L in rows if L.size), default=0.0)
    return 52 - math.frexp(M)[1] if M > 0 else 0


def fixed_point(L: np.ndarray, e: int) -> np.ndarray:
    return np.rint(np.ldexp(L, e)).astype(np.int64)


def counts(weights: np.ndarray, g: int, b: int, seed: int) -> np.ndarray:
    """c[p] of replicate b of global partition g"""
    w = np.asarray(weights, dtype=np.uint64)
    cumw = np.concatenate([[0], np.cumsum(w)]).astype(np.uint64)
    N = int(cumw[-1])
    x = np.random.Philox(key=[seed, (g << 32) | b]).random_raw(N).astype(np.uint64)
    hi, lo = x >> np.uint64(32), x & np.uint64(0xFFFFFFFF)
    site = (hi * np.uint64(N) + ((lo * np.uint64(N)) >> np.uint64(32))) >> np.uint64(32)  # (x * N) >> 64
    p = np.searchsorted(cumw, site, side="right") - 1
    return np.bincount(p, minlength=len(w)).astype(np.int64)


def _exact_dot(c: np.ndarray, q: np.ndarray) -> list:
    """[sum_p c[b][p] * q[r][p] for r] for each b, exactly: q split at 2^26 keeps int64 sums exact"""
    qh, ql = q >> 26, q & ((1 << 26) - 1)
    a, m = c @ qh.T, c @ ql.T
    return [[int(a[i, j]) * (1 << 26) + int(m[i, j]) for j in range(q.shape[0])] for i in range(c.shape[0])]


def support(rows, weights, replicates: int, seed: int) -> dict:
    e = exponent_of(rows)
    R = rows[0].shape[0]
    Z = [[0] * R for _ in range(replicates)]
    O = [0] * R
    for g, (L, w) in enumerate(zip(rows, weights)):
        q = fixed_point(L, e)
        for r, v in enumerate(_exact_dot(np.asarray(w, dtype=np.int64)[None, :], q)[0]):
            O[r] += v
        c = np.stack([counts(w, g, b, seed) for b in range(replicates)])
        for b, zrow in enumerate(_exact_dot(c, q)):
            for r in range(R):
                Z[b][r] += zrow[r]
    B = replicates
    best = max(range(R), key=lambda r: (O[r], -r))
    colsum = [sum(Z[b][r] for b in range(B)) for r in range(R)]
    bp, kh, sh = [0] * R, [0] * R, [0] * R
    for b in range(B):
        z = Z[b]
        bp[max(range(R), key=lambda r: (z[r], -r))] += 1
        zt = [B * z[r] - colsum[r] for r in range(R)]
        mt = max(zt)
        for r in range(R):
            if B * (z[best] - z[r]) - (colsum[best] - colsum[r]) >= B * (O[best] - O[r]):
                kh[r] += 1
            if mt - zt[r] >= B * (O[best] - O[r]):
                sh[r] += 1
    return {"exponent": e, "O": O, "best": best, "bp_count": bp, "kh_count": kh, "sh_count": sh,
            "lnl_fixed": [math.ldexp(float(o), -e) for o in O]}
