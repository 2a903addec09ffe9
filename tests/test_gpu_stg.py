"""GPU: the exhaustive state-transition-graph kernels (k_change_masks, k_stg_expand, k_stg_walk) and the exact attractor
search built on them (gym_PBN.b200.attractors) against the host reference of tests/stg_reference.py, at every width the
kernels accept (N = 1..32): bit-exact change masks, one breadth-first level in each direction with and without `within`,
replayed random walks, terminal SCCs end to end, and the restricted-network route inside trap spaces.

Conventions the tests pin: the exhaustive STG lets every node change, node 0 of a truth-table network included (as
PBN.async_successors and compute_attractors do, although PBN.step never updates node 0); a predictor can be drawn only
with positive COD weight.  test_cases_reach_their_regime (CPU only) shows from the host reference that the cases reach the
regimes they are there for."""
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

import oracle as orc  # noqa: E402
import stg_reference as ref  # noqa: E402
from golden_util import random_predictor_sets  # noqa: E402

# table entries at the edges of the two comparisons p > 0 and p < 1
P_EDGE = (0.0, 1.0, 5e-324, 1.0 - 2.0**-53, 0.5)
P_E2E = (0.0, 1.0, 0.0, 1.0, 0.0, 1.0, 0.5, 5e-324)
KINDS_AT = {n: ("tt", "pred") + (("sets",) if n >= 5 else ()) for n in (1, 2, 3, 4, 5, 6, 12, 20, 24)}
E2E_AT = {n: ("ttd", "pred") + (("sets",) if n >= 8 else ()) for n in (1, 2, 3, 4, 8, 13, 17, 20)}
WIDE = [("b28", 28), ("tt", 29), ("pred", 29), ("tt", 30), ("pred", 30), ("tt", 31), ("pred", 31), ("tt", 32), ("pred", 32)]
TRAP_NETS = ("28_15_median", "70_5_kmeans", "synthetic-100")
WALKS = [("ttd", 6), ("ttd", 17), ("pred", 4)]
LIST_LIMIT = 100


def _seed(kind, n):
    return 100 * sum(map(ord, kind)) + n


# ------------------------------------------------------------------------------------------------ networks
def tt_data(n, seed, kmax=4, p=P_EDGE, frozen=0.0):
    """PBN_data tuples: 0..kmax inputs per node drawn from all nodes (its own included), table entries drawn from `p`; the
    last node has no inputs; a `frozen` share of the others copies its own value."""
    rng = np.random.default_rng(seed)
    data = []
    for i in range(n):
        if i < n - 1 and rng.random() < frozen:
            mask = np.zeros(n, bool)
            mask[i] = True
            data.append((mask, np.array([0.0, 1.0]), f"g{i}", False))
            continue
        k = 0 if i == n - 1 else int(rng.integers(0, min(kmax, n) + 1))
        mask = np.zeros(n, bool)
        mask[rng.choice(n, size=k, replace=False)] = True
        table = rng.choice(p, size=2**k)
        data.append((mask, table.reshape([2] * k) if k else np.array(table[0]), f"g{i}", False))
    return data


def pred_arrays(n, seed, fmax=18, frozen=0.3):
    """A predictor network as NetworkSpec arrays, built directly the way restricted_network builds one: four inputs per
    predictor drawn with repetition from all nodes (so N = 1..3 exist), LUTs constant 0x0000 / 0xFFFF, a copy of the node's
    own value (0xAAAA) or random; a third of the predictors has zero COD weight (cumulative COD equal to the one before, a
    first predictor at 0).  Node 0 has fmax predictors, a tenth of the others too, the rest 1..6.  In a `frozen` share of the
    nodes, and in the last one when N >= 2, every positive-weight predictor copies the node's own value: only a zero-weight
    predictor could flip it (the first one, at cumulative COD 0, would set it to 1)."""
    rng = np.random.default_rng(seed)
    off, ins, luts, cums, sums = [0], [], [], [], []
    for i in range(n):
        f = fmax if i == 0 or rng.random() < 0.1 else int(rng.integers(1, 7))
        freeze = rng.random() < frozen or (i == n - 1 and n >= 2)
        cum = 0.0
        for k in range(f):
            zero = (freeze and k == 0 and f > 1) or (rng.random() < 0.35 and (k < f - 1 or cum > 0.0))
            if not zero:
                cum += float(rng.uniform(0.05, 1.0))
            src = rng.integers(0, n, 4)
            if rng.random() < 0.3:
                src[1] = src[0]
            lut = 0xAAAA if freeze and not zero else int(rng.choice([0x0000, 0xFFFF, 0xAAAA, int(rng.integers(0, 1 << 16))]))
            if freeze and k == 0 and zero:
                lut = 0xFFFF
            if lut == 0xAAAA:
                src[3] = i
            ins += [int(v) for v in src]
            luts.append(lut)
            cums.append(cum)
        sums.append(cum)
        off.append(len(luts))
    return dict(pr_off=np.array(off, np.int32), pr_in=np.array(ins, np.int32), pr_lut=np.array(luts, np.uint16),
                pr_cum=np.array(cums, np.float64), pr_codsum=np.array(sums, np.float64))


def tt_spec(data):
    from gym_PBN.b200 import compiler

    spec = compiler.compile_pbn_data(data)
    if spec.n == 1:  # pbn_net_create needs an updatable node; k_change_masks does not look at first_updatable
        spec.first_updatable = 0
    return spec


def pred_spec(arrays, n):
    from gym_PBN.b200 import abi
    from gym_PBN.b200.compiler import NetworkSpec

    return NetworkSpec(abi.NET_PRED, n, 0, [f"g{i}" for i in range(n)], arrays=arrays)


@functools.lru_cache(maxsize=None)
def case(kind, n, fmax=18, frozen=0.3):
    """-> (NetworkSpec for the device, host reference of the change masks: states (None = all) -> uint32 masks).
    kind: "tt" (tt_data), "ttd" (tt_data, mostly deterministic tables and frozen nodes), "pred" (pred_arrays), "sets" (random predictor sets: the device compiles them, the reference
    reads the oracle's arrays), "b28" (the shipped Bittner-28 predictor sets)."""
    from gym_PBN.b200 import compiler

    seed = _seed(kind, n)
    if kind in ("tt", "ttd"):
        data = tt_data(n, seed) if kind == "tt" else tt_data(n, seed, p=P_E2E, frozen=frozen)
        return tt_spec(data), functools.partial(ref.tt_change_masks, data)
    if kind == "pred":
        arrays = pred_arrays(n, seed, fmax, frozen)
        return pred_spec(arrays, n), functools.partial(ref.pred_change_masks, arrays, n)
    sets, ids = random_predictor_sets(n, 5, seed) if kind == "sets" else orc.load_bittner("28_15_median")
    onet = orc.net_from_predictor_sets(sets, ids)
    return compiler.compile_predictor_sets(sets, ids), functools.partial(ref.pred_change_masks, onet.a, onet.n)


@functools.lru_cache(maxsize=None)
def full_masks(*args):
    return case(*args)[1]()


def e2e_case(kind, n):
    return (kind, n, 6, 0.1) if kind == "pred" and n >= 13 else (kind, n)  # fewer frozen nodes: fewer attractors to list


def one_scc_data(n=12):
    """Every node is a coin flip without inputs: all 2^n states form one strongly connected component."""
    return [(np.zeros(n, bool), np.array(0.5), f"g{i}", False) for i in range(n)]


def fixed_point_data():
    """Nine nodes: 0..6 keep their value (table = own value); nodes 7 and 8 copy each other while node 6 is 0 and are coin
    flips while it is 1.  -> 2 x 64 fixed points (node 6 = 0, x7 = x8) and 64 four-state cycles (node 6 = 1)."""
    n, data = 9, []
    for i in range(7):
        mask = np.zeros(n, bool)
        mask[i] = True
        data.append((mask, np.array([0.0, 1.0]), f"g{i}", False))
    for i, other in ((7, 8), (8, 7)):
        mask = np.zeros(n, bool)
        mask[[6, other]] = True
        data.append((mask, np.array([[0.0, 1.0], [0.5, 0.5]]), f"g{i}", False))
    return data


@functools.lru_cache(maxsize=None)
def trap_net(name):
    """-> (NetworkSpec, oracle network) of a shipped predictor set, or of "synthetic-100": pred_arrays with 60 % frozen nodes.
    (The sampled trap spaces of Bittner-100 have 19 or more wildcards; the synthetic network stands in for it.)"""
    from gym_PBN.b200 import compiler

    if name == "synthetic-100":
        arrays = pred_arrays(100, 77, fmax=6, frozen=0.6)
        return pred_spec(arrays, 100), orc.Net(orc.ORC_PRED, 100, 0, **arrays)
    sets, ids = orc.load_bittner(name)
    return compiler.load_bittner(name), orc.net_from_predictor_sets(sets, ids)


@functools.lru_cache(maxsize=None)
def trap_cubes(name, max_free=18, keep=16):
    """Trap spaces of sampled end states as verified_attractors forms them (asynchronous rollouts from random states; a state
    inside a trap space already found is skipped), the oracle standing in for the device rollout (the same law); the `keep`
    with the most wildcards among those with at most max_free."""
    from gym_PBN.b200.attractors import SuccessorModel, trap_space

    spec, onet = trap_net(name)
    model = SuccessorModel(spec)
    st = orc.rand_state(onet, 128, orc.Draws(seed=11, epoch=0))
    orc.rollout(onet, st, 512 * onet.n, orc.Draws(seed=11, epoch=1))
    spaces = []
    for s in np.unique(st, axis=0):
        if not any(all(c == "*" or c == int(v) for c, v in zip(t, s)) for t in spaces):
            spaces.append(trap_space(model, s))
    free = lambda t: sum(v == "*" for v in t)  # noqa: E731
    return sorted((t for t in spaces if free(t) <= max_free), key=free, reverse=True)[:keep]


# ------------------------------------------------------------------------------------------------ device helpers
def _cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _need_gib(gib):
    """Skip when the device has less than `gib` GiB free (checked once per test; never retried)."""
    free, _ = torch.cuda.mem_get_info()
    if free < gib * (1 << 30):
        pytest.skip(f"needs {gib} GiB of free device memory, {free / (1 << 30):.1f} GiB free")


def stg_of(spec):
    from gym_PBN.b200 import attractors, engine

    return attractors.StateTransitionGraph(engine.Network(spec))


def host_words(t):
    return t.cpu().numpy().view(np.uint32)


def dev_words(words):
    return torch.from_numpy(np.ascontiguousarray(words, np.uint32).view(np.int32)).cuda()


def with_masks(stg, masks):
    """Point the graph at host-reference masks, so expand / walk are tested on their own."""
    stg.masks = torch.from_numpy(np.ascontiguousarray(masks, np.uint32).view(np.int32)).cuda()
    return stg


def cube_states(cube):
    """State indices (bit i = node i) of a cube in node order."""
    s = np.zeros(1, np.int64)
    for i, v in enumerate(cube):
        if v == "*":
            s = np.concatenate([s, s | (1 << i)])
        elif int(v):
            s |= 1 << i
    return s


def check_cover(cubes, states):
    """Cubes are disjoint and their union is exactly `states`."""
    got = np.concatenate([cube_states(c) for c in cubes])
    assert len(np.unique(got)) == len(got), "cubes overlap"
    assert np.array_equal(np.sort(got), np.sort(np.asarray(states, np.int64)))


# ------------------------------------------------------------------------------------------------ host reference (CPU)
def _host_pbn(data):
    from gym_PBN.envs.common.node import Node
    from gym_PBN.envs.common.pbn import PBN

    pbn = PBN.__new__(PBN)
    pbn.N = len(data)
    pbn.nodes = np.empty(pbn.N, dtype=object)
    for i, (m, t, *_r) in enumerate(data):
        pbn.nodes[i] = Node(m, t, i)
    return pbn


def _host_graph(spec):
    """Graph over a compiled spec without a device network: genSTG only reads the spec's arrays."""
    from gym_PBN.envs.bittner import base

    g = base.Graph(2)
    g.spec = spec
    g.nodes = [base.Node(i, i, spec.names[i], i) for i in range(spec.n)]
    for node in g.nodes:
        node._graph = g
    return g


@pytest.mark.parametrize("n", [1, 2, 3, 5, 8])
def test_reference_matches_async_successors(n):
    """Truth tables: reference masks == the nodes PBN.async_successors flips; terminal SCCs == PBN.attractors_host."""
    data = tt_data(n, _seed("tt", n))
    masks = ref.tt_change_masks(data)
    pbn = _host_pbn(data)
    for s in range(1 << n):
        st = np.array(ref.state_tuple(s, n), bool)
        want = 0
        for nxt, _p in pbn.async_successors(st):
            want |= 1 << int(np.nonzero(nxt != st)[0][0])
        assert int(masks[s]) == want, s
    got = sorted(sorted(ref.state_tuple(s, n) for s in a) for a in ref.terminal_sccs(masks))
    assert got == sorted(sorted(a) for a in pbn.attractors_host())


@pytest.mark.parametrize("kind,n", [("pred", 2), ("pred", 3), ("pred", 6), ("pred", 10), ("sets", 6), ("sets", 10)])
def test_reference_matches_genstg(kind, n):
    """Predictor networks: reference masks == the non-loop edges of Graph.genSTG; terminal SCCs == findAttractors."""
    from gym_PBN.envs.bittner import base

    spec, fn = case(kind, n)
    masks = fn()
    stg = _host_graph(spec).genSTG()
    want = np.zeros(1 << n, np.uint32)
    for u, v in stg.edges():
        d = [i for i in range(n) if u[i] != v[i]]
        if d:
            want[sum(b << i for i, b in enumerate(u))] |= 1 << d[0]
    assert np.array_equal(masks, want)
    got = sorted(sorted(ref.state_tuple(s, n) for s in a) for a in ref.terminal_sccs(masks))
    assert got == sorted(sorted(a) for a in base.findAttractors(stg))


def test_reference_bitsets_and_walk_law():
    """to_bitset / from_bitset round trip with clear padding; the walk stops on a fixed point and flips one changeable
    node per move."""
    rng = np.random.default_rng(0)
    for n in (1, 2, 4, 5, 7):
        f = rng.random(1 << n) < 0.5
        w = ref.to_bitset(f)
        assert len(w) == max(1, (1 << n) >> 5) and np.array_equal(ref.from_bitset(w, 1 << n), f)
        if n < 5:
            assert int(w[0]) >> (1 << n) == 0
    masks = full_masks("ttd", 6)
    fixed = int(np.nonzero(masks == 0)[0][0])
    assert ref.walk(masks, fixed, 50, 3) == (fixed, 0)
    s = 5
    for t in range(1, 30):
        e, moves = ref.walk(masks, 5, t, 9)
        if moves < t:
            break
        assert bin(e ^ s).count("1") == 1 and (int(masks[s]) >> ((e ^ s).bit_length() - 1)) & 1
        s = e


@pytest.mark.parametrize("fn", ["expand", "walk"])
def test_expand_and_walk_argument_errors(fn):
    """pbn_stg_expand: N < 1, N > 32 or a null bitset -> 1; pbn_stg_walk: steps < 0 -> 1 (both checked before any launch)."""
    import ctypes as C

    from gym_PBN.b200 import abi

    buf = (C.c_uint32 * 64)()
    p = C.cast(buf, C.c_void_p)
    lib = abi.lib()
    if fn == "expand":
        assert lib.pbn_stg_expand(p, 0, p, p, None, p, 0, None) == 1
        assert lib.pbn_stg_expand(p, 33, p, p, None, p, 0, None) == 1
        for k in range(4):
            args = [p, p, p, p]
            args[k] = None
            assert lib.pbn_stg_expand(args[0], 4, args[1], args[2], None, args[3], 0, None) == 1
    else:
        assert lib.pbn_stg_walk(p, 4, 0, -1, 0, p, None) == 1
        assert lib.pbn_stg_walk(p, 0, 0, 1, 0, p, None) == 1
        assert lib.pbn_stg_walk(p, 33, 0, 1, 0, p, None) == 1


def test_cases_reach_their_regime():
    """From the host reference (all states up to N = 12, 2^16 random ones above): every predictor case of N >= 2 has a state
    where a zero-weight predictor would flip a node that no positive-weight predictor flips; every truth-table case has a
    state where node 0 can change, a zero entry reached from 0 (p >= 0 would count it) and, from N = 3, tables whose index
    order matters; each walk case has a fixed point and a state whose only move enters it; the list_limit case has more
    fixed points than the limit; the one-SCC case has one component."""
    rng = np.random.default_rng(0)
    for n in KINDS_AT:
        states = None if n <= 12 else rng.integers(0, 1 << n, 1 << 16)
        if n >= 2:
            a = dict(case("pred", n)[0].arrays)
            a["pr_cum"] = np.arange(1, len(a["pr_cum"]) + 1, dtype=np.float64)  # every predictor drawable
            assert np.any(ref.pred_change_masks(a, n, states) != case("pred", n)[1](states)), n
        data = tt_data(n, _seed("tt", n))
        masks = ref.tt_change_masks(data, states)
        assert np.any(masks & 1), n
        ge = [(m, np.where(np.asarray(t) == 0.0, 5e-324, t), *r) for m, t, *r in data]
        assert np.any(ref.tt_change_masks(ge, states) != masks), n
        lsb = [(m, np.asarray(t).transpose(), *r) for m, t, *r in data]
        if n >= 3:  # (at N = 2 no node has two inputs)
            assert np.any(ref.tt_change_masks(lsb, states) != masks), n
    for kind, n in WALKS:
        masks = full_masks(kind, n)
        assert np.any(masks == 0) and _into_fixed(masks) is not None, (kind, n)
    fixed = ref.tt_change_masks(fixed_point_data()) == 0
    assert fixed.sum() == 128 > LIST_LIMIT
    assert len(ref.terminal_sccs(ref.tt_change_masks(one_scc_data()))) == 1


def test_restricted_route_premise():
    """Each network gives trap spaces of at most 18 wildcards, and some of them fix nodes at 1 (the fold in
    restricted_network reads a constant 1)."""
    for name in TRAP_NETS:
        cubes = trap_cubes(name)
        assert cubes, name
        assert any(any(v == 1 for v in c) for c in cubes), name
        assert any(sum(v == "*" for v in c) >= 2 for c in cubes), name


# ------------------------------------------------------------------------------------------------ change masks (GPU)
@gpu
@pytest.mark.parametrize("kind,n", [(k, n) for n, kinds in KINDS_AT.items() for k in kinds])
def test_change_masks_every_state(kind, n):
    """Every state of truth-table, hand-built predictor and predictor-set networks of N = 1..24 nodes."""
    _cuda()
    stg = stg_of(case(kind, n)[0])
    assert np.array_equal(host_words(stg.masks), full_masks(kind, n))


@gpu
@pytest.mark.parametrize("kind,n", WIDE)
def test_wide_networks(kind, n):
    """N = 28..32: change masks on 2^20 random states and the top indices 2^N - 1, 2^N - 2^k; one expand level in each
    direction from a state >= 2^(N-1) (node N - 1 set: state bit 31 at N = 32); a 64 N-step walk from such a state."""
    _cuda()
    _need_gib(4 * 2 ** (n - 30) + 3 * 2 ** (n - 33) + 1)
    spec, fn = case(kind, n)
    stg = stg_of(spec)
    top = (1 << n) - 1
    rng = np.random.default_rng(n)
    states = np.concatenate([rng.integers(0, 1 << n, 1 << 20, dtype=np.uint64),
                             np.array([top - (1 << k) + 1 for k in range(n + 1)], np.uint64)])  # 2^N - 2^k, k = 0..N
    states = states[states < (1 << n)]
    got = stg.masks[torch.from_numpy(states.astype(np.int64)).cuda()].cpu().numpy().view(np.uint32)
    assert np.array_equal(got, fn(states))
    # one level from a single top state: exactly its successors / predecessors
    s = int(rng.integers(1 << (n - 1), 1 << n))
    nb = np.array([s ^ (1 << i) for i in range(n)], np.uint64)
    ms, mt = int(fn([s])[0]), fn(nb)
    for direction in (0, 1):
        want = {int(t) for i, t in enumerate(nb) if ((ms if direction == 0 else int(mt[i])) >> i) & 1}
        nxt = stg.empty()
        stg.expand(stg.single(s), stg.empty(), nxt, direction)
        nz = torch.nonzero(nxt).reshape(-1)
        words = nxt[nz].cpu().numpy().view(np.uint32)
        got = {(int(w) << 5) | b for w, v in zip(nz.cpu().numpy(), words) for b in range(32) if (int(v) >> b) & 1}
        assert got == want, direction
        del nxt
    lazy = type("Lazy", (), {"__getitem__": lambda self, t: int(fn([t])[0])})()
    seed = (7 << 32) | 123
    assert stg.walk(s, 64 * n, seed) == ref.walk(lazy, s, 64 * n, seed)[0]
    del stg
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ expand (GPU)
def _padding_ok(words, n):
    return n >= 5 or int(words[0]) >> (1 << n) == 0


@gpu
@pytest.mark.parametrize("n", [1, 3, 4, 5, 6, 10, 16])
def test_expand_one_level(n):
    """Random frontier / visited / within sets, both directions, with and without `within`, on the reference masks."""
    _cuda()
    kind = "pred" if n % 2 == 0 else "tt"
    masks = full_masks(kind, n)
    stg = with_masks(stg_of(case(kind, n)[0]), masks)
    S = 1 << n
    rng = np.random.default_rng(n)
    trials = [(np.ones(S, bool), np.zeros(S, bool), np.ones(S, bool))]  # the whole state set, padding clear
    for density in (0.05, 0.3, 0.7):
        trials.append((rng.random(S) < density, rng.random(S) < 0.3, rng.random(S) < 0.6))
    for frontier, visited, within in trials:
        win = ref.to_bitset(within)
        if n < 5:
            win[0] |= np.uint32(0xFFFFFFFF) << np.uint32(S)  # padding set in `within`: the output's must stay clear
        for direction in (0, 1):
            for w in (None, within):
                nxt = stg.empty()
                stg.expand(dev_words(ref.to_bitset(frontier)), dev_words(ref.to_bitset(visited)), nxt, direction,
                           None if w is None else dev_words(win))
                want = ref.to_bitset(ref.expand(masks, frontier, visited, w, direction))
                got = host_words(nxt)
                assert _padding_ok(got, n)
                assert np.array_equal(got, want), (direction, w is None)
    assert any(ref.expand(masks, f, v, None, 1).any() for f, v, _w in trials)


@gpu
@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6])
def test_bitset_helpers(n):
    """StateTransitionGraph.full / pack / single / count / first / members against the reference bitsets."""
    _cuda()
    stg = stg_of(case("tt", n)[0])
    S = 1 << n
    assert np.array_equal(host_words(stg.full()), ref.to_bitset(np.ones(S, bool)))
    rng = np.random.default_rng(n)
    f = rng.random(S) < 0.5
    f[S - 1] = True
    bits = stg.pack(torch.from_numpy(f).cuda())
    assert np.array_equal(host_words(bits), ref.to_bitset(f))
    assert stg.count(bits) == int(f.sum()) and stg.first(bits) == int(np.nonzero(f)[0][0])
    assert np.array_equal(stg.members(bits), np.nonzero(f)[0].astype(np.uint32))
    for s in (0, S - 1, min(31, S - 1)):
        one = np.zeros(S, bool)
        one[s] = True
        assert np.array_equal(host_words(stg.single(s)), ref.to_bitset(one))


# ------------------------------------------------------------------------------------------------ walk (GPU)
def _into_fixed(masks):
    """A state whose only move enters a fixed point (a walk from it stops after one move), or None."""
    n = len(masks).bit_length() - 1
    for f in np.nonzero(masks == 0)[0]:
        for i in range(n):
            if masks[f ^ (1 << i)] == 1 << i:
                return int(f ^ (1 << i))
    return None


@gpu
@pytest.mark.parametrize("kind,n", WALKS)
def test_walk_replays(kind, n):
    """Walks of 0, 1, 7 and 64 N steps (what exact_attractors asks for), seeds with high key words, from random states, a
    fixed point, the top state and a state next to a fixed point, replayed exactly."""
    _cuda()
    masks = full_masks(kind, n)
    stg = with_masks(stg_of(case(kind, n)[0]), masks)
    rng = np.random.default_rng(n)
    fixed = int(np.nonzero(masks == 0)[0][0])
    starts = [int(v) for v in rng.integers(0, 1 << n, 6)] + [fixed, (1 << n) - 1, _into_fixed(masks)]
    early = 0
    for k, s in enumerate(starts):
        for steps, seed in ((0, 1), (1, 2), (7, 3 + k), (64 * n, 11 + k), (64 * n, (k + 1) << 32 | 5), (3, 0xFFFFFFFFFFFFFFFF)):
            want, moves = ref.walk(masks, s, steps, seed)
            assert stg.walk(s, steps, seed) == want, (s, steps, seed)
            early += moves < steps
        assert stg.walk(s, 0, 4) == s
    assert stg.walk(fixed, 64 * n, 9) == fixed
    assert early > 0  # some walk ended on a fixed point before its step count


# ------------------------------------------------------------------------------------------------ end to end (GPU)
def _check_found(found, want, n):
    """exact_attractors' entries == the reference's terminal SCCs: every attractor, its listed states, its bitset."""
    assert len(found) == len(want)
    for a, w in zip(sorted(found, key=lambda a: int(a["states"][0])), want):
        assert a["size"] == len(w) and np.array_equal(np.sort(a["states"]), w)
        if a["bits"] is not None:
            assert np.array_equal(host_words(a["bits"]), ref.to_bitset(np.isin(np.arange(1 << n), w)))


@gpu
@pytest.mark.parametrize("kind,n", [(k, n) for n, kinds in E2E_AT.items() for k in kinds])
def test_exact_attractors_equal_terminal_sccs(kind, n):
    """exact_attractors == terminal_sccs; attractor_state_sets lists them as state tuples, or raises when one is larger
    than its list_limit; states_to_cubes covers each exactly."""
    from gym_PBN.b200 import attractors, engine

    _cuda()
    net = engine.Network(case(*e2e_case(kind, n))[0])
    want = ref.terminal_sccs(full_masks(*e2e_case(kind, n)))
    _check_found(attractors.exact_attractors(net, list_limit=1 << 20), want, n)
    if max(map(len, want)) <= 1 << 16:
        sets = attractors.attractor_state_sets(net)
        assert sorted(map(sorted, sets)) == sorted(sorted(ref.state_tuple(s, n) for s in w) for w in want)
    else:
        with pytest.raises(ValueError):
            attractors.attractor_state_sets(net)
    for w in want[:64]:
        check_cover(attractors.states_to_cubes(w, n), w)


@gpu
def test_one_scc():
    from gym_PBN.b200 import attractors, engine

    _cuda()
    data = one_scc_data()
    net = engine.Network(tt_spec(data))
    found = attractors.exact_attractors(net)
    assert len(found) == 1 and found[0]["size"] == 1 << 12
    _check_found(found, ref.terminal_sccs(ref.tt_change_masks(data)), 12)
    assert attractors.exact_attractor_cubes(net) == [[("*",) * 12]]


@gpu
def test_more_fixed_points_than_list_limit():
    from gym_PBN.b200 import attractors, engine

    _cuda()
    data = fixed_point_data()
    masks = ref.tt_change_masks(data)
    net = engine.Network(tt_spec(data))
    found = attractors.exact_attractors(net, list_limit=LIST_LIMIT)
    fp = [a for a in found if a.get("fixed_points")]
    assert len(fp) == 1 and fp[0]["size"] == 128 and fp[0]["states"] is None
    assert np.array_equal(host_words(fp[0]["bits"]), ref.to_bitset(masks == 0))
    cycles = [a for a in found if not a.get("fixed_points")]
    want = [w for w in ref.terminal_sccs(masks) if len(w) > 1]
    _check_found(cycles, want, 9)
    assert len(cycles) == 64
    with pytest.raises(ValueError):
        attractors.attractor_state_sets(net, list_limit=LIST_LIMIT)
    with pytest.raises(ValueError):
        attractors.exact_attractor_cubes(net, list_limit=LIST_LIMIT)
    assert len(attractors.attractor_state_sets(net, list_limit=128)) == 128 + 64


def test_states_to_cubes_cover():
    """states_to_cubes: disjoint cubes whose union is the state set (random sets, a full space, one state, a cube)."""
    from gym_PBN.b200.attractors import states_to_cubes

    rng = np.random.default_rng(4)
    for n in (1, 3, 6, 9):
        for density in (0.1, 0.5, 0.9):
            s = np.nonzero(rng.random(1 << n) < density)[0]
            if len(s):
                check_cover(states_to_cubes(s, n), s)
        check_cover(states_to_cubes(np.arange(1 << n), n), np.arange(1 << n))
        assert states_to_cubes(np.arange(1 << n), n) == [("*",) * n]
        check_cover(states_to_cubes([(1 << n) - 1], n), [(1 << n) - 1])
    cube = (1, "*", 0, "*", "*", 1)
    assert states_to_cubes(cube_states(cube), 6) == [cube]


# ------------------------------------------------------------------------------------------------ restricted route (GPU)
@gpu
@pytest.mark.parametrize("name", TRAP_NETS)
def test_restricted_route_equals_host_enumeration(name):
    """terminal_sccs_on_device (restricted_network folded, exhaustive device search) == terminal_sccs_in_cube on the host,
    for every sampled trap space of at most 18 wildcards."""
    from gym_PBN.b200 import attractors as at, engine

    _cuda()
    spec = trap_net(name)[0]
    net, model = engine.Network(spec), at.SuccessorModel(spec)
    for cube in trap_cubes(name):
        dev = at.terminal_sccs_on_device(net, cube)
        host = at.terminal_sccs_in_cube(model, cube, 18)
        norm = lambda atts: sorted(sorted("".join(map(str, c)) for c in cubes) for cubes in atts)  # noqa: E731
        assert norm(dev) == norm(host), cube


# ------------------------------------------------------------------------------------------------ argument errors (GPU)
@gpu
def test_change_masks_rejects_33_nodes():
    import ctypes as C

    from gym_PBN.b200 import abi, attractors, engine

    _cuda()
    net = engine.Network(case("pred", 33, 4)[0])
    buf = torch.zeros(8, dtype=torch.int32, device="cuda")
    assert abi.lib().pbn_stg_change_masks(net.handle, C.c_void_p(buf.data_ptr()), None) == 3
    assert abi.lib().pbn_stg_change_masks(net.handle, None, None) == 1
    with pytest.raises(ValueError):
        attractors.StateTransitionGraph(net)
    assert int(buf.abs().sum()) == 0
