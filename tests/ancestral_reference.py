"""The marginal ancestral states of DESIGN.md section 11, restated with numpy (no FMA: agreement with
the engine is to ~1e-13 relative, not bit for bit).  Inputs are plain arrays: the post-order operations,
the P-matrices they name, the tips' 0/1 CLVs, pi and the category weights.  The post-order CLVs are
recomputed here with the 2^-256 rescaling, then the outside vectors in reverse operation order."""
import numpy as np

SCALE_THRESHOLD = 2.0 ** -256
SCALE_FACTOR = 2.0 ** 256
LOG_SCALE = -177.44567822334599


def _rescale(x):
    """x [S][K][4]: patterns whose every entry is below 2^-256 are multiplied by 2^256"""
    small = np.all(x < SCALE_THRESHOLD, axis=(1, 2))
    x = x.copy()
    x[small] *= SCALE_FACTOR
    return x, small.astype(np.int64)


def marginal(ops, P, tips, pi, w):
    """ops: tuples (parent, parent scaler, c1, m1, s1, c2, m2, s2) in post-order; P: {matrix: [K][4][4]};
    tips: {clv index: [S][K][4]}; returns map_state, map_prob, log_norm [node][S] and posterior
    [node][S][4], nodes in operation order"""
    clv, sc = dict(tips), {}
    h = {}
    for (v, vs, c1, m1, s1, c2, m2, s2) in ops:
        h1 = np.einsum("kjl,skl->skj", P[m1], clv[c1])
        h2 = np.einsum("kjl,skl->skj", P[m2], clv[c2])
        d = h1 * h2
        S = d.shape[0]
        sig = np.zeros(S, dtype=np.int64)
        if vs >= 0:
            d, small = _rescale(d)
            sig = sc.get(c1, 0) + sc.get(c2, 0) + small
        clv[v], sc[v], h[v] = d, sig, (h1, h2)
    S, K = clv[ops[-1][0]].shape[:2]
    out = {"map_state": [], "map_prob": [], "log_norm": [], "posterior": []}
    o = {ops[-1][0]: np.broadcast_to(np.asarray(pi, dtype=np.float64), (S, K, 4)).copy()}
    tau = {ops[-1][0]: np.zeros(S, dtype=np.int64)}
    res = [None] * len(ops)
    for n in range(len(ops) - 1, -1, -1):
        v, vs, c1, m1, s1, c2, m2, s2 = ops[n]
        h1, h2 = h[v]
        t = np.einsum("k,ski->si", np.asarray(w, dtype=np.float64), o[v] * clv[v])
        Z = ((t[:, 0] + t[:, 1]) + t[:, 2]) + t[:, 3]
        post = t / Z[:, None]
        best = np.argmax(post, axis=1)
        res[n] = (best.astype(np.uint8), post[np.arange(S), best], np.log(Z) + (sc[v] + tau[v]) * LOG_SCALE, post)
        for c, Pc, hs, sib in ((c1, P[m1], h2, c2), (c2, P[m2], h1, c1)):
            if c in tips:
                continue
            oc = np.einsum("skj,kji->ski", o[v] * hs, Pc)
            oc, small = _rescale(oc)
            o[c] = oc
            tau[c] = tau[v] + sc.get(sib, 0) + small
    for r in res:
        for key, val in zip(("map_state", "map_prob", "log_norm", "posterior"), r):
            out[key].append(val)
    return {k: np.array(v) for k, v in out.items()}


def brute_force(ops, P, tips, pi, w):
    """the posterior of every internal node by enumerating all 4^(internal nodes) assignments (a few
    taxa only): [node][S][4] in operation order"""
    nodes = [op[0] for op in ops]
    root = nodes[-1]
    S, K = next(iter(tips.values())).shape[:2]
    edges = []  # (parent, child, matrix)
    for (v, _vs, c1, m1, _s1, c2, m2, _s2) in ops:
        edges += [(v, c1, m1), (v, c2, m2)]
    post = np.zeros((len(nodes), S, 4))
    idx = {v: i for i, v in enumerate(nodes)}
    for code in range(4 ** len(nodes)):
        a = {v: (code >> (2 * i)) & 3 for i, v in enumerate(nodes)}
        # per category: prior * product over edges of P[parent state][child state or tip vector]
        lk = np.broadcast_to(np.asarray(pi, dtype=np.float64)[a[root]], (S, K)).copy()
        for (v, c, m) in edges:
            if c in tips:
                lk = lk * np.einsum("kl,skl->sk", P[m][:, a[v], :], tips[c])
            else:
                lk = lk * P[m][:, a[v], a[c]][None, :]
        site = lk @ np.asarray(w, dtype=np.float64)
        for v in nodes:
            post[idx[v], :, a[v]] += site
    return post / post.sum(axis=2, keepdims=True)
