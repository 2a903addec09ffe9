"""Shared by the edge-pin tests (tests/test_oracle_edge_pins.py, CPU, and tests/test_gpu_edge_pins.py, GPU): the entry
encoding of pbn_ssd_pinned_edges, the regulatory edges of an oracle network, and the exact stationary law of a small network
with edges pinned, computed on the gather side (node dst's function evaluated on the state with each pinned source replaced
by its constant)."""
import numpy as np

EMPTY = 0xFFFFFFFF


def entry(src, dst, c):
    return dst | src << 12 | c << 24


def edge_rows(variants, E=None):
    """uint32 [K][E] rows from lists of (src, dst, c) (or raw uint32 entries), padded with empty slots."""
    E = max([len(v) for v in variants] + [0]) if E is None else E
    out = np.full((len(variants), E), EMPTY, np.uint32)
    for k, v in enumerate(variants):
        for j, e in enumerate(v):
            out[k, j] = entry(*e) if isinstance(e, tuple) else e
    return out


def inputs(onet, dst):
    """The input slots of node dst of an oracle network: per predictor [in0, in1, in2, self], or the truth table's inputs."""
    a = onet.a
    if "pr_in" in a:
        return [list(a["pr_in"][4 * q:4 * q + 4]) for q in range(a["pr_off"][dst], a["pr_off"][dst + 1])]
    return [list(a["tt_in"][a["tt_in_off"][dst]:a["tt_in_off"][dst + 1]])]


def edges_of(onet):
    """Distinct (src, dst) pairs in (dst, slot) order."""
    out = []
    for dst in range(onet.n):
        for rec in inputs(onet, dst):
            for src in rec:
                if (int(src), dst) not in out:
                    out.append((int(src), dst))
    return out


def exact_edge_law(onet, edges, p, tgt):
    """Stationary law over the target buckets of the chain x -> update(flip(x)) of an oracle network (at most ~10 nodes)
    with edge pins {(src, dst): c}: every node flips w.p. p, then one asynchronous update (node uniform in [first, n)) whose
    function reads c for each pinned input.  Predictor choice and table entries use the exact probabilities (the device's
    31-bit thresholds differ from them by less than 2^-31)."""
    a, n, first = onet.a, onet.n, onet.first
    S = 1 << n
    s = np.arange(S)
    bit = lambda x, i: (x >> i) & 1  # noqa: E731
    T = np.zeros((S, S))
    for i in range(first, n):
        seen = s.copy()  # the state as node i's function reads it
        for (src, dst), c in edges.items():
            if dst == i:
                seen = (seen & ~(1 << src)) | (c << src)
        if "pr_in" in a:
            q0, q1 = a["pr_off"][i], a["pr_off"][i + 1]
            cum = np.concatenate([[0.0], a["pr_cum"][q0:q1]]) / a["pr_codsum"][i]
            cum[-1] = 1.0  # the last predictor takes whatever the others leave
            p1 = np.zeros(S)
            for q in range(q0, q1):
                x0, x1, x2, x3 = (bit(seen, a["pr_in"][4 * q + j]) for j in range(4))
                p1 += (cum[q - q0 + 1] - cum[q - q0]) * ((int(a["pr_lut"][q]) >> (x0 << 3 | x1 << 2 | x2 << 1 | x3)) & 1)
        else:
            idx = np.zeros(S, np.int64)
            for j in a["tt_in"][a["tt_in_off"][i]:a["tt_in_off"][i + 1]]:
                idx = idx * 2 + bit(seen, j)
            p1 = a["tt_prob"][a["tt_tab_off"][i] + idx]
        w = 1.0 / (n - first)
        np.add.at(T, (s, s | (1 << i)), w * p1)
        np.add.at(T, (s, s & ~(1 << i)), w * (1.0 - p1))
    d = s[:, None] ^ s[None, :]
    flips = np.vectorize(lambda x: bin(x).count("1"))(d)
    M = (p ** flips * (1 - p) ** (n - flips)) @ T
    A = np.vstack([M.T - np.eye(S), np.ones(S)])
    b = np.zeros(S + 1)
    b[-1] = 1.0
    pi = np.linalg.lstsq(A, b, rcond=None)[0]
    bucket = np.zeros(S, np.int64)
    for i in tgt:
        bucket = bucket * 2 + ((s >> i) & 1)
    return np.bincount(bucket, weights=pi, minlength=1 << len(tgt))
