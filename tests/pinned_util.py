"""Ground truth of the pinned-SSD tests (tests/test_oracle_pinned.py, CPU, and tests/test_gpu_pinned_ssd.py, GPU): the exact
stationary law of a small truth-table network with some genes pinned, from its explicit transition matrix."""
import numpy as np

import control_util as cu


def exact_pinned_law(pbn_data, pin, p, tgt):
    """Stationary law over the target buckets of the chain x -> update(flip(x)) of the pinned network: flips of the free
    nodes w.p. p each, then one asynchronous update (PBN.step) where a pinned node's function is its constant."""
    n = len(pbn_data)
    data = [(np.zeros(n, bool), np.array(float(pin[i])), None, True) if i in pin else d for i, d in enumerate(pbn_data)]
    T = cu.transition_matrix(data)
    S = 1 << n
    s = np.arange(S)
    pinned = sum(1 << i for i in pin)
    d = s[:, None] ^ s[None, :]
    flips = np.vectorize(lambda x: bin(x).count("1"))(d)
    nfree = n - len(pin)
    F = np.where(d & pinned, 0.0, p ** flips * (1 - p) ** (nfree - flips))
    M = F @ T
    A = np.vstack([M.T - np.eye(S), np.ones(S)])
    b = np.zeros(S + 1)
    b[-1] = 1.0
    pi = np.linalg.lstsq(A, b, rcond=None)[0]
    bucket = np.zeros(S, np.int64)
    for i in tgt:
        bucket = bucket * 2 + ((s >> i) & 1)
    return np.bincount(bucket, weights=pi, minlength=1 << len(tgt))
