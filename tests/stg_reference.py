"""TEST INFRASTRUCTURE — host reference of the exhaustive asynchronous state-transition graph (STG) that
gym_PBN.b200.attractors searches on the device: change masks, one breadth-first level over sets of states, the seeded
random walk and the terminal strongly connected components.  NumPy (SciPy for the components) only, built from the
reference-form network — PBN_data tuples for truth tables, the predictor arrays of the oracle's network
(oracle.net_from_predictor_sets, LUTs from oracle.predictor_lut) or hand-built NetworkSpec arrays for predictor
networks — so it shares no code with the compiler or the kernels.

A state is an integer index with bit i = node i (the device's convention).  Its change mask has bit i set when node i
can take the other value in one asynchronous update: an edge s -> s ^ (1 << i) of the STG.  Sets of states are bool
arrays over all 2^N states here; `to_bitset` / `from_bitset` convert to and from the device's uint32 words
(bit b of word w = state 32 w + b; below N = 5 one partial word whose padding bits are clear)."""
import numpy as np

import oracle as orc


def _states(n, states):
    return np.arange(1 << n, dtype=np.uint32) if states is None else np.asarray(states, dtype=np.uint32)


def _in_chunks(fn, s, step=1 << 15):
    """fn over cache-sized pieces of the state array (all 2^24 states at once would stream every intermediate array
    through memory)."""
    return np.concatenate([fn(s[k:k + step]) for k in range(0, len(s), step)]) if len(s) > step else fn(s)


def tt_change_masks(pbn_data, states=None):
    """Change masks of a truth-table network given as PBN_data tuples (input mask, table of P(next = 1), ...), at `states`
    (every state when None).  The table is indexed by the masked inputs in ascending node order, the first one the most
    significant bit.  Node i can change when p > 0 from 0 and when p < 1 from 1, for every node — node 0 included, as
    PBN.async_successors and PBN.attractors_host count it although PBN.step never updates it."""
    return _in_chunks(lambda s: _tt_masks(pbn_data, s), _states(len(pbn_data), states))


def _tt_masks(pbn_data, s):
    out = np.zeros(s.shape, np.uint32)
    for i, node in enumerate(pbn_data):
        mask = np.asarray(node[0], dtype=bool)
        table = np.asarray(node[1], dtype=np.float64).reshape(-1)
        idx = np.zeros(s.shape, np.uint32)
        for j in np.nonzero(mask)[0]:
            idx = (idx << np.uint32(1)) | ((s >> np.uint32(j)) & np.uint32(1))
        p = table[idx]
        cur = (s >> np.uint32(i)) & np.uint32(1)
        can = ((cur == 0) & (p > 0.0)) | ((cur == 1) & (p < 1.0))
        out |= can.astype(np.uint32) << np.uint32(i)
    return out


def pred_change_masks(arrays, n, states=None):
    """Change masks of a predictor network given by its arrays: pr_off (predictors of node i are pr_off[i]..pr_off[i+1]),
    pr_in (four input nodes per predictor, the first the most significant bit of the LUT index), pr_lut (16-bit LUT) and
    pr_cum (cumulative COD).  Only a predictor with positive COD weight — a cumulative COD above the one before it, 0 before
    the first — can be drawn (bittner/base.py:94-97); node i can change when one of them gives the other value."""
    return _in_chunks(lambda s: _pred_masks(arrays, n, s), _states(n, states))


def _pred_masks(arrays, n, s):
    off, ins, lut, cum = (np.asarray(arrays[k]) for k in ("pr_off", "pr_in", "pr_lut", "pr_cum"))
    out = np.zeros(s.shape, np.uint32)
    for i in range(n):
        cur = (s >> np.uint32(i)) & np.uint32(1)
        can = np.zeros(s.shape, bool)
        prev = 0.0
        for k in range(int(off[i]), int(off[i + 1])):
            c = float(cum[k])
            if c > prev:
                idx = np.zeros(s.shape, np.uint32)
                for q in range(4):
                    idx = (idx << np.uint32(1)) | ((s >> np.uint32(ins[4 * k + q])) & np.uint32(1))
                can |= ((np.uint32(lut[k]) >> idx) & np.uint32(1)) != cur
            prev = max(prev, c)
        out |= can.astype(np.uint32) << np.uint32(i)
    return out


def _n_of(masks):
    n = len(masks).bit_length() - 1
    assert len(masks) == 1 << n, "masks must cover all 2^N states"
    return n


def expand(masks, frontier, visited, within, direction):
    """One breadth-first level: the states outside `visited` (and inside `within` unless it is None) that are a successor
    (direction 0: s -> s ^ (1 << i) with node i changeable in s) or a predecessor (direction 1: t -> s, t = s ^ (1 << i)
    with node i changeable in t) of a state of `frontier`.  Bool arrays over all 2^N states."""
    masks = np.asarray(masks, dtype=np.uint32)
    n = _n_of(masks)
    src = np.nonzero(frontier)[0]
    nxt = np.zeros(len(masks), bool)
    for i in range(n):
        t = src ^ (1 << i)
        ok = ((masks[src if direction == 0 else t] >> np.uint32(i)) & 1).astype(bool)
        nxt[t[ok]] = True
    nxt &= ~np.asarray(visited, bool)
    if within is not None:
        nxt &= np.asarray(within, bool)
    return nxt


def walk(masks, start, steps, seed):
    """pbn_stg_walk's law: at move t (from 0) draw o0 = Philox4x32-10(counter (t, t >> 32, 0x57a1, 0), key = seed)[0], pick
    = umulhi(o0, popcount(m)) for the mask m of the current state, flip the pick-th set bit of m counted from the least
    significant; stop early on an empty mask (a fixed point).  `masks` is anything indexable by a state.
    -> (end state, moves made)."""
    s = int(start)
    key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    for t in range(int(steps)):
        m = int(masks[s])
        if m == 0:
            return s, t
        o0 = orc.philox((t & 0xFFFFFFFF, (t >> 32) & 0xFFFFFFFF, 0x57A1, 0), key)[0]
        pick = (o0 * bin(m).count("1")) >> 32
        for _ in range(pick):
            m &= m - 1
        s ^= m & -m
    return s, int(steps)


def terminal_sccs(masks, max_nodes=20):
    """Attractors: the strongly connected components of the STG without an edge leaving them, each a sorted uint32 array of
    state indices, the list ordered by smallest member."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components

    masks = np.asarray(masks, dtype=np.uint32)
    n = _n_of(masks)
    if n > max_nodes:
        raise ValueError(f"{n} nodes: too many states for the host reference")
    idx = np.arange(len(masks), dtype=np.int64)
    src, dst = [np.zeros(0, np.int64)], [np.zeros(0, np.int64)]
    for i in range(n):
        ch = ((masks >> np.uint32(i)) & 1).astype(bool)
        src.append(idx[ch])
        dst.append(idx[ch] ^ (1 << i))
    S, D = np.concatenate(src), np.concatenate(dst)
    g = coo_matrix((np.ones(len(S), np.int8), (S, D)), shape=(len(masks), len(masks))).tocsr()
    ncomp, lab = connected_components(g, directed=True, connection="strong")
    leaves = np.ones(ncomp, bool)
    leaves[lab[S][lab[S] != lab[D]]] = False
    order = np.argsort(lab, kind="stable")
    bounds = np.searchsorted(lab[order], np.arange(ncomp + 1))
    out = [order[bounds[c]:bounds[c + 1]].astype(np.uint32) for c in np.nonzero(leaves)[0]]
    return sorted(out, key=lambda a: int(a[0]))


def to_bitset(flags):
    """bool [2^N] -> uint32 words (one partial word below N = 5, padding bits clear)."""
    f = np.asarray(flags, bool)
    words = np.zeros(max(1, (len(f) + 31) // 32), np.uint32)
    idx = np.nonzero(f)[0]
    np.bitwise_or.at(words, idx >> 5, (np.uint32(1) << (idx & 31).astype(np.uint32)))
    return words


def from_bitset(words, n_states):
    """uint32 words -> bool [n_states] (padding bits dropped)."""
    w = np.asarray(words, dtype=np.uint32)
    bits = (w[:, None] >> np.arange(32, dtype=np.uint32)[None, :]) & 1
    return bits.reshape(-1)[:n_states].astype(bool)


def state_tuple(s, n):
    return tuple((int(s) >> i) & 1 for i in range(n))
