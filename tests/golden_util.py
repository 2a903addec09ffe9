"""Helpers shared by the oracle tests (CPU) and the CUDA parity tests (GPU): load a golden trace
recorded from the reference (oracle/make_golden.py) and build oracle-side networks/envs from it."""
from pathlib import Path

import numpy as np

GOLD = Path(__file__).resolve().parent / "golden"


def load(name):
    return np.load(GOLD / name, allow_pickle=False)


class Traj:
    def __init__(self, z, e):
        p = f"e{e}/"
        for k in ("op", "act", "int_off", "ints", "dbl_off", "dbls", "state", "obs", "reward", "term", "trunc", "target_att"):
            setattr(self, k, z[p + k])
        self.T = len(self.op)

    def draws(self, t, t1=None):
        t1 = t + 1 if t1 is None else t1
        return (self.ints[self.int_off[t]:self.int_off[t1]], self.dbls[self.dbl_off[t]:self.dbl_off[t1]])


def pbn_data_from(z):
    """(input_mask, table[2]*k) tuples back from the padded arrays stored in a truth-table golden."""
    out = []
    for m, t in zip(z["masks"], z["tables"]):
        k = int(m.sum())
        out.append((m.astype(bool), t[: 2**k].reshape([2] * k) if k else np.array(t[0])))
    return out


def cubes_to_attractors(cubes, off):
    atts = []
    for a in range(len(off) - 1):
        atts.append([tuple("*" if v == 2 else int(v) for v in c) for c in cubes[off[a]:off[a + 1]]])
    return atts


from gym_PBN.b200.synthetic import synthetic_pbcn  # noqa: E402,F401  (configs[4]: lives in the package, bench.py uses it too)


# ------------------------------------------------------------------------------------------------ synthetic networks
def random_predictor_sets(n, fmax, seed):
    """Synthetic predictor sets with 1..fmax predictors per node (node 0 has fmax; the last column of some nodes empty, as
    add_to_buff leaves it) -> (sets, node ids) in the form of the shipped pickles."""
    rng = np.random.default_rng(seed)
    ids = [1000 + 3 * i for i in range(n)]
    sets = []
    for i in range(n):
        f = fmax if i == 0 else int(rng.integers(1, fmax + 1))
        buf = np.empty((3, fmax), dtype=object)
        others = [x for x in range(n) if x != i]
        for k in range(f):
            trio = rng.choice(others, 3, replace=False)
            buf[0, k], buf[1, k], buf[2, k] = float(rng.uniform(0.05, 1.0)), rng.normal(size=(4, 1)), np.array([ids[t] for t in trio])
        sets.append(buf)
    return sets, ids


def random_predictor_net(eng, n, fmax, seed):
    """(device network, oracle network) of random_predictor_sets(n, fmax, seed)."""
    import oracle as orc

    sets, ids = random_predictor_sets(n, fmax, seed)
    return eng.engine.Network(eng.compiler.compile_predictor_sets(sets, ids)), orc.net_from_predictor_sets(sets, ids)


def random_tt_data(n, seed):
    """PBN_data tuples of a random truth-table network: 0..5 inputs per node, each table a mix of two Boolean functions."""
    rng = np.random.default_rng(seed)
    pbn_data = []
    for i in range(n):
        k = int(rng.integers(0, 6))
        mask = np.zeros(n, bool)
        mask[rng.choice(n, size=k, replace=False)] = True
        f1, f2 = rng.integers(0, 2, 2**k), rng.integers(0, 2, 2**k)
        c = float(rng.uniform(0.05, 0.95))
        pbn_data.append((mask, (c * f1 + (1 - c) * f2).reshape([2] * k), f"n{i}", k == 0))
    return pbn_data


# ------------------------------------------------------------------------------------------------ attractor fixtures
def hittable_cubes(onet, count, seed, care=4, B=64, steps=2000):
    """`count` cubes that an asynchronous walk can reach: each copies `care` positions of a state that a long oracle rollout
    from random states visits (Philox draws), every other position '*'."""
    import oracle as orc

    rng = np.random.default_rng(seed)
    st = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0))
    orc.rollout(onet, st, steps, orc.Draws(seed=seed, epoch=1))
    n = onet.n
    lo = n - onet.first  # truth-table networks never update node 0 (first updatable = 1): leave it uncared
    cubes = []
    for _ in range(count):
        s = st[int(rng.integers(0, B))]
        c = ["*"] * n
        for i in (n - lo) + rng.choice(lo, size=care, replace=False):
            c[i] = int(s[i])
        cubes.append(tuple(c))
    return cubes


# hittable positions of each fixture size, and its attractor sizes.  Where a hit sits in the cube list decides which branch
# of the attractor test must see it: a lane group of g lanes tests cubes sub and sub + g itself (sub < g) and loops over the
# rest; the lockstep first pass keeps incremental mismatch counts for one or two cubes.
FIXTURE_HITS = {1: (0,), 2: (1,), 7: (5,), 14: (9, 12), 72: (66, 69)}


def _fixture_sizes(n_cubes):
    if n_cubes <= 2:
        return [1] * n_cubes
    if n_cubes == 7:
        return [1, 2, 1, 2, 1]
    if n_cubes == 14:
        return [1, 2, 3, 1, 1, 2, 2, 2]
    sizes, left, k = [], n_cubes - 7, 0  # 72: runs of 1, 2, 3 cubes, then [65, 66], [67, 68], [69, 70, 71]
    while left:
        sizes.append(min(k % 3 + 1, left))
        left -= sizes[-1]
        k += 1
    return sizes + [2, 2, 3]


def attractor_fixture(onet, n_cubes, seed, care=4):
    """Decoys + hittable cubes: n_cubes cubes, hittable (hittable_cubes) at FIXTURE_HITS[n_cubes] and decoys (random full
    states, practically never reached) everywhere else, grouped into attractors of 1..3 cubes.  The first hittable cube is
    the SECOND cube of its attractor (TARGET's reward tests every cube of the target attractor) except in the 1- and 2-cube
    fixtures; in the 14- and 72-cube fixtures the last one starts the last attractor (MULTI's reward looks at the first
    cube of the last attractor only).  Returns the attractors (lists of cubes)."""
    hits = FIXTURE_HITS[n_cubes]
    rng = np.random.default_rng(seed + 1)
    hc = iter(hittable_cubes(onet, len(hits), seed, care=care))
    cubes = [next(hc) if c in hits else tuple(int(v) for v in rng.integers(0, 2, onet.n)) for c in range(n_cubes)]
    atts, a = [], 0
    for size in _fixture_sizes(n_cubes):
        atts.append(cubes[a:a + size])
        a += size
    assert a == n_cubes
    return atts
