"""Gene and gene-then-site resampling of root placement support (DESIGN.md section 10, items 11-14)
restated with numpy and Python integers, for the tests: numpy.random.Philox gives the draws, Python
ints (in numpy object arrays) the exact sums.  Input as tests/rell_reference.py: per partition (in
global order) its rows L [records][patterns] and pattern weights."""
from __future__ import annotations

import math

import numpy as np

from rell_reference import exponent_of, fixed_point


def gene_draws(G: int, b: int, seed: int) -> np.ndarray:
    """m[i] of replicate b: word j of Philox from the counter {0, 0, 1, 0} picks partition (x_j G) >> 64"""
    x = np.random.Philox(counter=np.array([0, 0, 1, 0], dtype=np.uint64), key=[seed, b]).random_raw(G)
    x = x.astype(np.uint64)
    hi, lo = x >> np.uint64(32), x & np.uint64(0xFFFFFFFF)
    pick = (hi * np.uint64(G) + ((lo * np.uint64(G)) >> np.uint64(32))) >> np.uint64(32)
    return np.bincount(pick.astype(np.int64), minlength=G).astype(np.int64)


def site_counts(weights: np.ndarray, g: int, b: int, seed: int, draws: int) -> np.ndarray:
    """c[p] from the first `draws` words of item 3's stream of global partition g and replicate b"""
    w = np.asarray(weights, dtype=np.uint64)
    cumw = np.concatenate([[0], np.cumsum(w)]).astype(np.uint64)
    N = int(cumw[-1])
    x = np.random.Philox(key=[seed, (g << 32) | b]).random_raw(draws).astype(np.uint64)
    hi, lo = x >> np.uint64(32), x & np.uint64(0xFFFFFFFF)
    site = (hi * np.uint64(N) + ((lo * np.uint64(N)) >> np.uint64(32))) >> np.uint64(32)  # (x * N) >> 64
    p = np.searchsorted(cumw, site, side="right") - 1
    return np.bincount(p, minlength=len(w)).astype(np.int64)


def exact_dot(c: np.ndarray, q: np.ndarray) -> np.ndarray:
    """sum_p c[b][p] q[r][p] as Python ints, [b][r]: q in three 18-bit pieces, so that every partial sum
    of a float64 product is an integer below 2^53 when each row of c sums below 2^35"""
    c = np.asarray(c, dtype=np.int64)
    assert (c >= 0).all() and int(c.sum(axis=1).max(initial=0)) < (1 << 35)
    mask = (1 << 18) - 1
    pieces = (q & mask, (q >> 18) & mask, q >> 36)
    out = np.zeros((c.shape[0], q.shape[0]), dtype=object)
    cf = c.astype(np.float64)
    for k, piece in enumerate(pieces):
        part = (cf @ piece.astype(np.float64).T).astype(np.int64).astype(object)
        out = out + part * (1 << (18 * k))
    return out


def statistics(Z: np.ndarray, O: list) -> dict:
    """items 4-5 over Z [b][r] (object array of Python ints)"""
    B, R = Z.shape
    best = max(range(R), key=lambda r: (O[r], -r))
    Oa = np.array(O, dtype=object)
    colsum = Z.sum(axis=0)
    bp = np.bincount([int(np.argmax(z)) for z in Z], minlength=R)  # argmax: the first of equal values
    delta = B * (Oa[best] - Oa)
    kh = ((B * (Z[:, best:best + 1] - Z) - (colsum[best] - colsum)[None, :]) >= delta[None, :]).sum(axis=0)
    zt = B * Z - colsum[None, :]
    mt = zt.max(axis=1)
    sh = ((mt[:, None] - zt) >= delta[None, :]).sum(axis=0)
    return {"best": best, "bp_count": [int(v) for v in bp], "kh_count": [int(v) for v in kh],
            "sh_count": [int(v) for v in sh]}


def support(rows, weights, replicates: int, seed: int, sampling: str) -> dict:
    assert sampling in ("gene", "gene_site")
    G = len(rows)
    e = exponent_of(rows)
    R = rows[0].shape[0]
    m = np.stack([gene_draws(G, b, seed) for b in range(replicates)])
    q = [fixed_point(L, e) for L in rows]
    Oi = [[int(v) for v in exact_dot(np.asarray(w, dtype=np.int64)[None, :], qi)[0]] for w, qi in zip(weights, q)]
    O = [sum(Oi[i][r] for i in range(G)) for r in range(R)]
    Z = np.zeros((replicates, R), dtype=object)
    for i in range(G):
        if sampling == "gene":
            Z = Z + m[:, i:i + 1].astype(object) * np.array(Oi[i], dtype=object)[None, :]
            continue
        N = int(np.sum(np.asarray(weights[i], dtype=np.int64)))
        c = np.stack([site_counts(weights[i], i, b, seed, int(m[b, i]) * N) for b in range(replicates)])
        Z = Z + exact_dot(c, q[i])
    out = statistics(Z, O)
    out.update({"exponent": e, "O": O, "lnl_fixed": [math.ldexp(float(o), -e) for o in O], "partition_O": Oi,
                "partition_llh": [[math.ldexp(float(o), -e) for o in row] for row in Oi],
                "partition_best": [max(range(R), key=lambda r: (row[r], -r)) for row in Oi], "m": m})
    return out
