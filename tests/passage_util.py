"""Shared by the first-passage tests (tests/test_oracle_passage.py, CPU, and tests/test_gpu_passage.py, GPU): the exact
first-passage law of a small network under a node pin set and edge pins, from powers of its per-iteration transition
matrix restricted to the states outside the goal."""
import numpy as np


def iteration_matrix(onet, pin, edges, p):
    """The transition matrix [2^n][2^n] of one SSD iteration x -> update(flip(x)) of an oracle network (at most ~10 nodes)
    with node pins `pin` {node: 0 or 1} and edge pins {(src, dst): c}: every free node flips w.p. p (a pinned node never
    does), then one asynchronous update (node uniform in [first, n)); a pinned node's update gives its value, and node i's
    function reads c for each pinned input (src, i).  The update part is the one edge_pin_util.exact_edge_law builds, with
    the node pins added."""
    a, n, first = onet.a, onet.n, onet.first
    S = 1 << n
    s = np.arange(S)
    bit = lambda x, i: (x >> i) & 1  # noqa: E731
    T = np.zeros((S, S))
    for i in range(first, n):
        if i in pin:
            p1 = np.full(S, float(pin[i]))
        else:
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
    pinned = sum(1 << i for i in pin)
    d = s[:, None] ^ s[None, :]
    flips = np.vectorize(lambda x: bin(x).count("1"))(d)
    F = np.where(d & pinned, 0.0, p ** flips * (1 - p) ** (n - len(pin) - flips))
    return F @ T


def exact_passage(onet, pin, edges, p, tgt, goal, T):
    """(P(tau < T), E[min(tau, T)]) for chains started from uniform states with the pins applied, tau = the first iteration
    whose target bucket (first target most significant) lies in `goal`: E[min(tau, T)] = sum_{t < T} P(tau > t), and
    P(tau > t) = the start law on the states outside the goal times Q^t times 1, Q = the iteration matrix restricted to
    them."""
    n = onet.n
    s = np.arange(1 << n)
    bucket = np.zeros(1 << n, np.int64)
    for i in tgt:
        bucket = bucket * 2 + ((s >> i) & 1)
    out = ~np.isin(bucket, list(goal))
    care = sum(1 << i for i in pin)
    val = sum(v << i for i, v in pin.items())
    start = np.bincount((s & ~care) | val, minlength=1 << n) / float(1 << n)
    Q = iteration_matrix(onet, pin, edges, p)[np.ix_(out, out)]
    v = start[out]
    mean = 0.0
    for _ in range(T):
        surv = v.sum()  # P(tau > t)
        mean += surv
        v = v @ Q
    return 1.0 - surv, mean
