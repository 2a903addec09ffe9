"""Host-side ground truth for the attractor-control tests (tests/test_attractor_control_host.py, CPU, and
tests/test_gpu_attractor_control.py, GPU): the explicit asynchronous state-transition matrix of small truth-table networks,
its terminal SCCs, exact landing probabilities of one target-env step, and the oracle's run of the attractor_transitions
schedule."""
import functools
import itertools
import json

import numpy as np
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

from golden_util import GOLD, random_tt_data

CAP_CASES = {"b28": 12288, "tt31": 4096}  # oracle-schedule cases (cap 64) -> num_envs; b28's B > 8192 takes the planned step
CAP = 64
CAP_SAMPLES = {"b28": 300, "tt31": 50}  # steps per (attractor, action) cell: two and three rounds of the schedule
CAP_SEED = 11


# ------------------------------------------------------------------------------------------------ small truth-table networks
def transition_matrix(pbn_data, first=1):
    """T[s, s'] of one asynchronous update (PBN.step: node i uniform in [first, n), next value 1 w.p. its table entry);
    state s: bit i = node i."""
    n = len(pbn_data)
    S = 1 << n
    s = np.arange(S)
    T = np.zeros((S, S))
    for i in range(first, n):
        mask, tab = np.asarray(pbn_data[i][0], bool), np.asarray(pbn_data[i][1], np.float64).reshape(-1)
        idx = np.zeros(S, np.int64)
        for j in np.nonzero(mask)[0]:  # ascending inputs, first = most significant
            idx = idx * 2 + ((s >> j) & 1)
        p1 = tab[idx]
        w = 1.0 / (n - first)
        np.add.at(T, (s, s | (1 << i)), w * p1)
        np.add.at(T, (s, s & ~(1 << i)), w * (1.0 - p1))
    return T


def terminal_sccs(T):
    """Attractors of the chain: terminal strongly connected components, as sorted state lists, ordered by first state."""
    g = csr_matrix(T > 0)
    k, lab = connected_components(g, directed=True, connection="strong")
    leaves = np.ones(k, bool)
    src, dst = g.nonzero()
    leaves[lab[src[lab[src] != lab[dst]]]] = False
    return sorted((np.nonzero(lab == c)[0].tolist() for c in range(k) if leaves[c]), key=lambda a: a[0])


def cube_states(cube):
    """Every state (int, bit i = node i) of a cube over {0, 1, '*'}."""
    fixed = sum(int(v) << i for i, v in enumerate(cube) if v != "*")
    wild = [i for i, v in enumerate(cube) if v == "*"]
    return [fixed + sum(b << i for b, i in zip(bits, wild)) for bits in itertools.product((0, 1), repeat=len(wild))]


def exact_landing(T, atts, n):
    """P[a][i][b] of one target-env step from the reset distribution of attractor a (uniform cube, uniform wildcards): flip
    node i-1 (i = 0: none), one update, then updates until the state lies in a cube of `atts` (no cap: column A = 0)."""
    A, S = len(atts), 1 << n
    cls = np.full(S, -1)
    for a in reversed(range(A)):  # the first attractor with a matching cube wins
        for c in atts[a]:
            cls[cube_states(c)] = a
    att, tr = cls >= 0, np.nonzero(cls < 0)[0]
    H = np.zeros((S, A + 1))
    H[att, cls[att]] = 1.0
    if len(tr):
        Q, R = T[np.ix_(tr, tr)], T[np.ix_(tr, np.nonzero(att)[0])] @ H[att]
        H[tr] = np.linalg.solve(np.eye(len(tr)) - Q, R)
    land = T @ H  # after the one forced update
    P = np.zeros((A, n + 1, A + 1))
    for a in range(A):
        for c in atts[a]:
            st = np.asarray(cube_states(c))
            for i in range(n + 1):
                P[a, i] += land[st if i == 0 else st ^ (1 << (i - 1))].mean(0) / len(atts[a])
    return P


def random_det_data(n, seed):
    """PBN_data of a random deterministic network: 1..3 inputs per node, a random Boolean function each."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        k = int(rng.integers(1, 4))
        mask = np.zeros(n, bool)
        mask[rng.choice(n, size=k, replace=False)] = True
        out.append((mask, rng.integers(0, 2, 2**k).astype(np.float64).reshape([2] * k), f"n{i}", False))
    return out


FIXED_POINT_SEED = 50  # three fixed points; the best chance of reaching the first within 1, 2, 3 steps is 0.56, 0.85, 0.95


@functools.lru_cache(maxsize=None)
def fixed_point_net():
    """(pbn_data, attractors) of a 6-node deterministic network whose attractors are all fixed points, from the exact
    terminal SCCs: there the attractor-level MDP is the env's own MDP."""
    data = random_det_data(6, FIXED_POINT_SEED)
    return data, [[tuple((s >> i) & 1 for i in range(6)) for s in a] for a in terminal_sccs(transition_matrix(data))]


@functools.lru_cache(maxsize=None)
def ground_truth_net():
    """(pbn_data, attractors as cubes) of the first 8-node random truth-table network (seeds 0, 1, ...) with at least three
    exact attractors, one of them more than one cube or a cube with wildcards."""
    from gym_PBN.b200.attractors import states_to_cubes

    for seed in itertools.count():
        data = random_tt_data(8, seed)
        atts = [states_to_cubes(a, 8) for a in terminal_sccs(transition_matrix(data))]
        if len(atts) >= 3 and any(len(a) > 1 or "*" in a[0] for a in atts):
            return data, atts


# ------------------------------------------------------------------------------------------------ oracle schedule
def b28_attractors():
    return [[tuple(c) for c in a] for a in json.loads((GOLD / "b28_exact_attractors.json").read_text())]


def classify(states, atts):
    """Host classification, vectorised: index of the first attractor with a matching cube, -1 if none.  states: uint8
    [B][N].  (test_gpu_attractor_control checks it against attractors.cube_matches.)"""
    B, n = states.shape
    out = np.full(B, -1)
    for a in reversed(range(len(atts))):
        for c in atts[a]:
            care = np.array([v != "*" for v in c])
            val = np.array([0 if v == "*" else int(v) for v in c], np.uint8)
            out[(states[:, care] == val[care]).all(1)] = a
    return out


def deal_actions(a, offset, A, n_act):
    """The schedule of attractor_transitions: envs starting in attractor a get actions offset[a], offset[a] + 1, ... (mod
    N+1) in env order.  Returns (actions, new offset)."""
    per = np.bincount(a, minlength=A)
    order = np.argsort(a, kind="stable")
    rank = np.empty(len(a), np.int64)
    rank[order] = np.arange(len(a)) - (np.cumsum(per) - per)[a[order]]
    return (offset[a] + rank) % n_act, (offset + per) % n_act


@functools.lru_cache(maxsize=None)
def cap_case(name):
    """(reference-form network kind + data, attractors) of an oracle-schedule case."""
    from golden_util import attractor_fixture

    import oracle as orc

    if name == "b28":
        return ("pred",) + orc.load_bittner("28_15_median"), b28_attractors()
    data = random_tt_data(31, seed=5)
    return ("tt", data), attractor_fixture(orc.net_from_pbn_data(data), 7, seed=38)


def oracle_net(name):
    import oracle as orc

    ref, _ = cap_case(name)
    return orc.net_from_predictor_sets(ref[1], ref[2]) if ref[0] == "pred" else orc.net_from_pbn_data(ref[1])


@functools.lru_cache(maxsize=None)
def oracle_transitions(name, samples, seed):
    """attractor_transitions run on the oracle (Philox env_reset / env_step, host classification): counts [A][N+1][A+1]."""
    import oracle as orc

    onet, (_, atts) = oracle_net(name), cap_case(name)
    B, n, A = CAP_CASES[name], oracle_net(name).n, len(atts)
    oenv = orc.Env(orc.ENV_TARGET, n, attractors=atts, horizon=100, max_inner=CAP)
    counts = np.zeros((A, n + 1, A + 1), np.int64)
    offset = np.zeros(A, np.int64)
    for r in itertools.count():
        st, ns, ta = np.zeros((B, n), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
        orc.env_reset(onet, oenv, st, ns, ta, orc.Draws(seed=seed, epoch=2 * r))
        a = classify(st, atts)
        assert (a >= 0).all()
        act, offset = deal_actions(a, offset, A, n + 1)
        orc.env_step(onet, oenv, st, ns, ta, act.astype(np.int32), orc.Draws(seed=seed, epoch=2 * r + 1))
        b = classify(st, atts)
        np.add.at(counts, (a, act, np.where(b < 0, A, b)), 1)
        if counts.sum(2).min() >= samples:
            return counts


# ------------------------------------------------------------------------------------------------ policies
def markov_optimum(P, target, H):
    """Largest mean (over a uniform start attractor) probability of reaching `target` within H steps, by exhaustive search
    over every deterministic time-dependent attractor-level policy (one decision rule per step)."""
    A, n_act = P.shape[0], P.shape[1]
    others = [a for a in range(A) if a != target]
    rules = np.array(list(itertools.product(range(n_act), repeat=len(others))))  # [R][A-1]
    Pr = np.zeros((len(rules), A, A))  # transition matrix of each decision rule
    for r, rule in enumerate(rules):
        for a, i in zip(others, rule):
            Pr[r, a] = P[a, i, :A]
        Pr[r, target, target] = 1.0
    V = np.zeros((1, A))
    V[0, target] = 1.0
    for _ in range(H):  # V over every rule sequence: [R^k][A]
        V = np.einsum("rab,vb->rva", Pr, V).reshape(-1, A)
    return V.mean(1).max()


def stationary_optimum(P, target, H):
    """The same search restricted to stationary policies (one decision rule for every step)."""
    A, n_act = P.shape[0], P.shape[1]
    others = [a for a in range(A) if a != target]
    best = 0.0
    for rule in itertools.product(range(n_act), repeat=len(others)):
        M = np.zeros((A, A))
        for a, i in zip(others, rule):
            M[a] = P[a, i, :A]
        M[target, target] = 1.0
        v = np.zeros(A)
        v[target] = 1.0
        for _ in range(H):
            v = M @ v
        best = max(best, v.mean())
    return best
