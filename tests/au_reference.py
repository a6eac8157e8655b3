"""The AU test's multiscale counts, its fit and the expected likelihood weights (DESIGN.md section 10,
items 6-8) restated with numpy and Python ints and floats, for the tests: numpy.random.Philox gives the
draws, Python ints the exact sums, Python floats (IEEE doubles, one rounding per operation) rd_exp and
the fit.  Input as in rell_reference: per partition (in global order) its rows L [records][patterns]
and pattern weights."""
from __future__ import annotations

import math
import struct

import numpy as np

import rell_reference


def counts(weights, g: int, b: int, seed: int, scale: int) -> np.ndarray:
    """c[p] of replicate b of global partition g at `scale` (thousandths): max(1, (s N + 500) // 1000)
    draws with the Philox counter's second word s - 1000 (mod 2^64)"""
    w = np.asarray(weights, dtype=np.uint64)
    cumw = np.concatenate([[0], np.cumsum(w)]).astype(np.uint64)
    N = int(cumw[-1])
    draws = max(1, (scale * N + 500) // 1000)
    counter = np.array([0, (scale - 1000) % (1 << 64), 0, 0], dtype=np.uint64)  # a list would be cast wrongly
    x = np.random.Philox(counter=counter, key=[seed, (g << 32) | b]).random_raw(draws).astype(np.uint64)
    hi, lo = x >> np.uint64(32), x & np.uint64(0xFFFFFFFF)
    site = (hi * np.uint64(N) + ((lo * np.uint64(N)) >> np.uint64(32))) >> np.uint64(32)  # (x * N) >> 64
    p = np.searchsorted(cumw, site, side="right") - 1
    return np.bincount(p, minlength=len(w)).astype(np.int64)


def z_at(rows, weights, replicates: int, seed: int, scale: int, e: int) -> list:
    R = rows[0].shape[0]
    Z = [[0] * R for _ in range(replicates)]
    for g, (L, w) in enumerate(zip(rows, weights)):
        q = rell_reference.fixed_point(L, e)
        c = np.stack([counts(w, g, b, seed, scale) for b in range(replicates)])
        for b, zrow in enumerate(rell_reference._exact_dot(c, q)):
            for r in range(R):
                Z[b][r] += zrow[r]
    return Z


P1, P2, P3 = 1.66666666666666019037e-01, -2.77777777770155933842e-03, 6.61375632143793436117e-05
P4, P5 = -1.65339022054652515390e-06, 4.13813679705723846039e-08
LN2HI, LN2LO, INVLN2 = 6.93147180369123816490e-01, 1.90821492927058770002e-10, 1.44269504088896338700e+00


def rd_exp(x: float) -> float:
    """fdlibm e_exp.c on [-40, 0], one rounding per operation"""
    hx = (struct.unpack("<Q", struct.pack("<d", x))[0] >> 32) & 0x7FFFFFFF
    hi = lo = 0.0
    k = 0
    if hx > 0x3FD62E42:
        if hx < 0x3FF0A2B2:
            hi, lo, k = x + LN2HI, -LN2LO, -1
        else:
            k = int(INVLN2 * x - 0.5)
            t = float(k)
            hi = x - t * LN2HI
            lo = t * LN2LO
        x = hi - lo
    elif hx < 0x3E300000:
        return 1.0 + x
    t = x * x
    c = x - t * (P1 + t * (P2 + t * (P3 + t * (P4 + t * P5))))
    if k == 0:
        return 1.0 - ((x * c) / (c - 2.0) - x)
    return math.ldexp(1.0 - ((lo - (x * c) / (2.0 - c)) - hi), k)


def elw_weight(delta: int, e: int) -> int:
    """u = rint(rd_exp(Delta 2^-e) 2^52), 0 when Delta < -40 2^e"""
    if delta * 2 ** max(0, -e) < -40 * 2 ** max(0, e):
        return 0
    return round(math.ldexp(rd_exp(math.ldexp(float(delta), -e)), 52))


def ppnd16(p: float) -> float:
    """Wichura's AS241"""
    q = p - 0.5
    if abs(q) <= 0.425:
        r = 0.180625 - q * q
        return q * (((((((2.5090809287301226727e+3 * r + 3.3430575583588128105e+4) * r + 6.7265770927008700853e+4)
                        * r + 4.5921953931549871457e+4) * r + 1.3731693765509461125e+4) * r
                      + 1.9715909503065514427e+3) * r + 1.3314166789178437745e+2) * r + 3.3871328727963666080e+0) / \
            (((((((5.2264952788528545610e+3 * r + 2.8729085735721942674e+4) * r + 3.9307895800092710610e+4) * r
                 + 2.1213794301586595867e+4) * r + 5.3941960214247511077e+3) * r + 6.8718700749205790830e+2) * r
              + 4.2313330701600911252e+1) * r + 1.0)
    r = math.sqrt(-math.log(p if q < 0 else 1.0 - p))
    if r <= 5.0:
        r -= 1.6
        v = (((((((7.74545014278341407640e-4 * r + 2.27238449892691845833e-2) * r + 2.41780725177450611770e-1) * r
                 + 1.27045825245236838258e+0) * r + 3.64784832476320460504e+0) * r + 5.76949722146069140550e+0) * r
              + 4.63033784615654529590e+0) * r + 1.42343711074968357734e+0) / \
            (((((((1.05075007164441684324e-9 * r + 5.47593808499534494600e-4) * r + 1.51986665636164571966e-2) * r
                 + 1.48103976427480074590e-1) * r + 6.89767334985100004550e-1) * r + 1.67638483018380384940e+0) * r
              + 2.05319162663775882187e+0) * r + 1.0)
    else:
        r -= 5.0
        v = (((((((2.01033439929228813265e-7 * r + 2.71155556874348757815e-5) * r + 1.24266094738807843860e-3) * r
                 + 2.65321895265761230930e-2) * r + 2.96560571828504891230e-1) * r + 1.78482653991729133580e+0) * r
              + 5.46378491116411436990e+0) * r + 6.65790464350110377720e+0) / \
            (((((((2.04426310338993978564e-15 * r + 1.42151175831644588870e-7) * r + 1.84631831751005468180e-5) * r
                 + 7.86869131145613259100e-4) * r + 1.48753612908506148525e-2) * r + 1.36929880922735805310e-1) * r
              + 5.99832206555887937690e-1) * r + 1.0)
    return -v if q < 0 else v


def au_fit(count, scales, B: int) -> dict:
    """item 7: (p_au, d, c, rss, used) of one record from its counts at the scales (thousandths)"""
    z, a, b, w = [], [], [], []
    for n_k, s in zip(count, scales):
        if 0 < n_k < B:
            p = n_k / B
            zk = -ppnd16(p)
            phi = math.exp(-zk * zk / 2.0) * 0.3989422804014327
            ak = math.sqrt(s / 1000.0)
            z.append(zk)
            a.append(ak)
            b.append(1.0 / ak)
            w.append(float(B) * phi * phi / (p * (1.0 - p)))
    if len(z) < 2:
        return {"p_au": sum(count) / (len(count) * B), "d": 0.0, "c": 0.0, "rss": 0.0, "used": len(z)}
    saa = sab = sbb = saz = sbz = 0.0
    for k in range(len(z)):
        saa += w[k] * a[k] * a[k]
        sab += w[k] * a[k] * b[k]
        sbb += w[k] * b[k] * b[k]
        saz += w[k] * a[k] * z[k]
        sbz += w[k] * b[k] * z[k]
    det = saa * sbb - sab * sab
    d = (sbb * saz - sab * sbz) / det
    c = (saa * sbz - sab * saz) / det
    rss = 0.0
    for k in range(len(z)):
        res = z[k] - d * a[k] - c * b[k]
        rss += w[k] * res * res
    return {"p_au": 0.5 * math.erfc((d - c) * math.sqrt(0.5)), "d": d, "c": c, "rss": rss, "used": len(z)}


def support(rows, weights, replicates: int, seed: int, scales) -> dict:
    """items 6-8 for every record: scale_count [scale][record], elw_fixed, and the fit per record"""
    e = rell_reference.exponent_of(rows)
    R, B = rows[0].shape[0], replicates
    scale_count = []
    for s in scales:
        n = [0] * R
        for z in z_at(rows, weights, B, seed, s, e):
            n[max(range(R), key=lambda r: (z[r], -r))] += 1
        scale_count.append(n)
    acc = [0] * R
    for z in z_at(rows, weights, B, seed, 1000, e):
        m = max(z)
        u = [elw_weight(v - m, e) for v in z]
        D = sum(u)
        for r in range(R):
            acc[r] += (u[r] << 40) // D
    fits = [au_fit([scale_count[k][r] for k in range(len(scales))], scales, B) for r in range(R)]
    out = {"scale_count": scale_count, "elw_fixed": acc,
           "elw": [math.ldexp(float(v), -40) / B for v in acc]}
    for key in ("p_au", "d", "c", "rss", "used"):
        out["au_" + key if key != "p_au" else key] = [f[key] for f in fits]
    return out
