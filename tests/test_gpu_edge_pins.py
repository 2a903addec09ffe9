"""GPU: pbn_ssd_pinned_edges (SSD estimates with regulatory edges pinned) against the oracle's gather-side
orc_ssd_pinned_edges bit for bit on every path of the SSD loop, against pbn_ssd_pinned without edge pins, against the
node pin it must equal and the exact stationary law of small networks, and through gym_PBN.utils.control (pinned_ssd,
rank_edge_pins)."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402
import edge_pin_oracle as eo  # noqa: E402
from edge_pin_util import EMPTY, edge_rows, edges_of, entry, exact_edge_law, inputs  # noqa: E402
from golden_util import random_predictor_sets, random_tt_data  # noqa: E402


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gym_PBN.b200 import abi, compiler, engine

    class E:
        pass

    e = E()
    e.abi, e.compiler, e.engine = abi, compiler, engine
    e.nets = {}
    return e


def _nets(eng, which):
    if which not in eng.nets:
        if which.startswith("pred"):
            n = int(which[4:])
            sets, ids = random_predictor_sets(n, 3 if n < 64 else 5, seed=n)
            eng.nets[which] = (eng.engine.Network(eng.compiler.compile_predictor_sets(sets, ids)), orc.net_from_predictor_sets(sets, ids))
        elif which.startswith("tt"):
            data = random_tt_data(int(which[2:]), seed=7)
            eng.nets[which] = (eng.engine.Network(eng.compiler.compile_pbn_data(data)), orc.net_from_pbn_data(data))
        else:
            sets, ids = orc.load_bittner(which)
            eng.nets[which] = (eng.engine.Network(eng.compiler.load_bittner(which)), orc.net_from_predictor_sets(sets, ids))
    return eng.nets[which]


def _masks(pins, n):
    w32 = (n + 31) // 32
    care, value = np.zeros((len(pins), w32), np.uint32), np.zeros((len(pins), w32), np.uint32)
    for k, pin in enumerate(pins):
        for i, v in pin.items():
            care[k, i >> 5] |= np.uint32(1 << (i & 31))
            value[k, i >> 5] |= np.uint32(v << (i & 31))
    return care, value


def _unpack(eng, planes, B, n):
    out = torch.empty((B, n), dtype=torch.uint8, device=planes.device)
    eng.abi.check(eng.abi.lib().pbn_unpack_state(C.c_void_p(planes.data_ptr()), B, n, C.c_void_p(out.data_ptr()),
                                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out.cpu().numpy()


def _run(eng, net, pins, edges, chains, iters, p, tgt, seed, env0):
    """Device run from rand_state (epoch 0), the pinned SSD in epoch 1: (hist [K][2^g], final states [K][chains][N])."""
    K = len(pins)
    sim = eng.engine.Simulator(net, chains, seed=seed, env0=env0)
    sim.rand_state()
    state = sim.state.repeat(1, K)
    hist = torch.zeros((K, 1 << len(tgt)), dtype=torch.int64, device=sim.device)
    care, value = _masks(pins, net.n)
    if isinstance(edges, str):  # "pbn_ssd_pinned": the entry without edge arguments
        d, t, dev = sim._draws(), np.ascontiguousarray(tgt, np.int32), lambda a: torch.from_numpy(a.view(np.int32)).cuda()  # noqa: E731
        care, value = dev(care), dev(value)
        eng.abi.check(eng.abi.lib().pbn_ssd_pinned(net.handle, C.c_void_p(state.data_ptr()), chains, env0, iters, p,
                                                   C.c_void_p(care.data_ptr()), C.c_void_p(value.data_ptr()), K,
                                                   t.ctypes.data_as(C.c_void_p), len(t), C.c_void_p(hist.data_ptr()),
                                                   C.byref(d), None))
    else:
        eng.engine.ssd_pinned(sim, state, iters, p, tgt, care, value, hist, edges=edges)
    return hist.cpu().numpy().astype(np.uint64), _unpack(eng, state, K * chains, net.n).reshape(K, chains, net.n)


def _oracle(onet, pins, edges, chains, iters, p, tgt, seed, env0):
    ost = orc.rand_state(onet, chains, orc.Draws(seed=seed, epoch=0), env0=env0)
    return eo.ssd_pinned(onet, ost, iters, p, pins, tgt, orc.Draws(seed=seed, epoch=1), env0=env0, edges=edges)


def _variants(onet, K, tgt, rng):
    """{} without edges first, then K - 1 variants of 0..3 node pins and 1..10 edge pins, among them: two inputs of one
    predictor record, a self-input, an edge into a node-pinned node, an edge out of a target gene, a non-edge entry, an
    entry with dst >= N, and empty slots."""
    n, all_edges = onet.n, edges_of(onet)
    pins, rows = [{}], [[]]
    for k in range(1, K):
        pin = {int(i): int(rng.integers(0, 2)) for i in rng.choice(n, size=int(rng.integers(0, 4)), replace=False)}
        c = lambda: int(rng.integers(0, 2))  # noqa: E731
        row = [all_edges[int(j)] + (c(),) for j in rng.choice(len(all_edges), size=int(rng.integers(1, 5)), replace=False)]
        dst = int(rng.integers(onet.first, n))
        rec = inputs(onet, dst)[0]
        if k % 4 == 1 and len(set(rec[:2])) == 2:
            row += [(int(rec[0]), dst, c()), (int(rec[1]), dst, c())]  # two edges into one record
        if k % 4 == 2 and (dst, dst) in all_edges:
            row.append((dst, dst, c()))  # self-input
        if k % 4 == 3 and pin:
            into = next((e for e in all_edges if e[1] in pin), None)
            if into:
                row.append(into + (c(),))  # into a node-pinned node
        t = int(tgt[k % len(tgt)])
        out_of_target = next((e for e in all_edges if e[0] == t and e[1] != t), None)
        if out_of_target:
            row.append(out_of_target + (c(),))
        if k % 3 == 0:
            non = next((s, d) for d in range(onet.first, n) for s in range(n) if (s, d) not in all_edges)
            row += [non + (1,), entry(1, n + 3, 1), EMPTY]
        rng.shuffle(row)
        pins.append(pin)
        rows.append(row)
    return pins, edge_rows(rows)


def _edge_screen(onet):
    """rank_edge_pins' variant set: {} and every edge at 0 and at 1."""
    es = edges_of(onet)
    return [{}] * (1 + 2 * len(es)), edge_rows([[]] + [[(s, d, c)] for s, d in es for c in (0, 1)])


CASES = [  # which, chains, iters, p, targets, K (0: the full single-edge screen)
    ("pred20", 96, 41, 0.3, list(range(0, 7)), 6),              # static loop, several rounds per iteration
    ("pred256", 64 + 5, 40, 0.01, list(range(200, 207)), 5),    # 8-word states, a partial warp next to the static loop
    ("28_15_median", 160, 9, 0.01, [20, 21, 22, 23], 6),        # two-level threshold rows (TQ 4), odd iteration count
    ("100_5_kmeans", 96, 7, 1e-6, list(range(0, 7)), 0),        # rank_edge_pins' 1 921 variants; rounds far apart
    ("100_5_kmeans", 3000, 400, 0.01, list(range(0, 7)), 5),    # the headline shape, smaller
    ("100_5_kmeans", 64, 10, 0.0, [3, 41, 69, 7], 5),           # no perturbation, scattered targets (generic loop)
    ("100_5_kmeans", 128, 10, 0.3, list(range(40, 53)), 5),     # g = 13: global-memory histogram
    ("100_5_kmeans", 32, 1, 0.01, list(range(0, 7)), 1),        # K = 1, one iteration (the generic tail only)
    ("tt70", 96, 9, 0.3, [1, 2, 3], 6),                          # truth table, threshold table in shared memory
]


@pytest.mark.parametrize("which,chains,iters,p,tgt,K", CASES)
def test_edge_pins_match_oracle(eng, which, chains, iters, p, tgt, K):
    net, onet = _nets(eng, which)
    tgt = np.array(tgt, np.int32)
    if K == 0:
        pins, edges = _edge_screen(onet)
        assert len(pins) == 1921
    elif K == 1:
        pins, edges = [{5: 1}], edge_rows([[(int(inputs(onet, 2)[0][0]), 2, 1), (0, 0, 0)]])
    else:
        pins, edges = _variants(onet, K, tgt, np.random.default_rng(len(tgt) + K))
    seed, env0 = 17, 64
    hist, out = _run(eng, net, pins, edges, chains, iters, p, tgt, seed, env0)
    ohist, oout = _oracle(onet, pins, edges, chains, iters, p, tgt, seed, env0)
    assert (hist.sum(1) == chains * iters).all()
    assert np.array_equal(hist, ohist)
    assert np.array_equal(out, oout)


def test_no_edges_is_pbn_ssd_pinned(eng):
    """E = 0 and rows of empty slots give pbn_ssd_pinned's histograms and final states bit for bit."""
    for which in ("100_5_kmeans", "tt70"):
        net, onet = _nets(eng, which)
        tgt = np.arange(1, 6, dtype=np.int32)
        pins = [{}, {2: 1}, {4: 0, 30: 1}]
        ref = _run(eng, net, pins, "pbn_ssd_pinned", 256, 300, 0.05, tgt, 9, 0)
        for edges in (None, np.zeros((3, 0), np.uint32), edge_rows([[]] * 3, E=7)):
            got = _run(eng, net, pins, edges, 256, 300, 0.05, tgt, 9, 0)
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])


@pytest.mark.parametrize("which", ["28_15_median", "tt70"])
def test_out_edges_equal_the_node_pin(eng, which):
    """Pinning every out-edge (u, v), v != u, of a node u outside the targets at c gives the node pin {u: c}'s histogram bit
    for bit, and the same final states but for u's bit, at p = 0.3, 0.01 and 0."""
    net, onet = _nets(eng, which)
    tgt = np.array([3, 4, 5, 6], np.int32)
    outs = {u: [(u, v) for s, v in edges_of(onet) if s == u and v != u] for u in range(onet.n) if u not in tgt}
    u = max((x for x in outs if len(outs[x]) <= 64), key=lambda x: len(outs[x]))
    for p in (0.3, 0.01, 0.0):
        for c in (0, 1):
            hn, sn = _run(eng, net, [{u: c}], None, 300, 200, p, tgt, 2, 0)
            he, se = _run(eng, net, [{}], edge_rows([[(s, v, c) for s, v in outs[u]]]), 300, 200, p, tgt, 2, 0)
            others = np.arange(net.n) != u
            assert np.array_equal(hn, he) and np.array_equal(sn[..., others], se[..., others])


@pytest.mark.parametrize("kind", ["pred", "tt"])
def test_exact_law(eng, kind):
    """8-node networks with two edge pins: 16 independent batches of 8192 chains x 20 000 iterations (after a burn-in) are
    within 0.005 in total variation of the exact gather-side law, and within 5 batch-means standard errors per bucket."""
    if kind == "tt":
        data = random_tt_data(8, seed=12)
        net, onet = eng.engine.Network(eng.compiler.compile_pbn_data(data)), orc.net_from_pbn_data(data)
        edges = {(5, 1): 1, (4, 7): 0}
    else:
        sets, ids = random_predictor_sets(8, 3, seed=5)
        net, onet = eng.engine.Network(eng.compiler.compile_predictor_sets(sets, ids)), orc.net_from_predictor_sets(sets, ids)
        edges = {(1, 7): 1, (6, 6): 1}
    p, tgt = 0.05, np.array([1, 4, 6, 7], np.int32)
    assert all(e in edges_of(onet) for e in edges)
    exact = exact_edge_law(onet, edges, p, tgt)
    rows = edge_rows([[(s, d, c) for (s, d), c in edges.items()]])
    care, value = _masks([{}], net.n)
    batches = []
    for b in range(16):
        sim = eng.engine.Simulator(net, 8192, seed=21, env0=8192 * b)
        sim.rand_state()
        state = sim.state.clone()
        burn = torch.zeros((1, 16), dtype=torch.int64, device=sim.device)
        eng.engine.ssd_pinned(sim, state, 500, p, tgt, care, value, burn, edges=rows)
        hist = torch.zeros((1, 16), dtype=torch.int64, device=sim.device)
        eng.engine.ssd_pinned(sim, state, 20000, p, tgt, care, value, hist, edges=rows)
        h = hist.cpu().numpy()[0].astype(np.float64)
        batches.append(h / h.sum())
    batches = np.array(batches)
    est, se = batches.mean(0), batches.std(0, ddof=1) / np.sqrt(len(batches))
    assert 0.5 * np.abs(est - exact).sum() < 0.005
    assert (np.abs(est - exact) <= 5 * se + 1e-12).all()


def test_sharded_launches_sum_to_one(eng):
    """Chains 0..95 and 96..255 in two launches (env0 = 0 and 96) give the histogram and final states of one launch."""
    net, onet = _nets(eng, "100_5_kmeans")
    tgt = np.arange(7, dtype=np.int32)
    pins, edges = _variants(onet, 5, tgt, np.random.default_rng(2))
    full_h, full_s = _run(eng, net, pins, edges, 256, 300, 0.01, tgt, 4, 0)
    h0, s0 = _run(eng, net, pins, edges, 96, 300, 0.01, tgt, 4, 0)
    h1, s1 = _run(eng, net, pins, edges, 160, 300, 0.01, tgt, 4, 96)
    assert np.array_equal(full_h, h0 + h1)
    assert np.array_equal(full_s, np.concatenate([s0, s1], axis=1))


def test_argument_errors(eng):
    lib, abi = eng.abi.lib(), eng.abi
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    def call(which, E=2, null_edges=False):
        net, _ = _nets(eng, which)
        state = torch.zeros((net.w32, 64 * 2), dtype=torch.int32, device="cuda")
        masks = torch.zeros((2, net.w32), dtype=torch.int32, device="cuda")
        edges = torch.full((2, 65), -1, dtype=torch.int32, device="cuda")
        hist = torch.zeros((2, 1 << 5), dtype=torch.int64, device="cuda")
        tgt = np.arange(5, dtype=np.int32)
        d = abi.PbnDraws(mode=abi.DRAW_PHILOX, seed=1, epoch=1)
        rc = lib.pbn_ssd_pinned_edges(net.handle, ptr(state), 64, 0, 10, 0.01, ptr(masks), ptr(masks), 2,
                                      None if null_edges else ptr(edges), E, tgt.ctypes.data_as(C.c_void_p), 5, ptr(hist),
                                      C.byref(d), None)
        torch.cuda.synchronize()
        return rc

    assert call("100_5_kmeans", E=-1) == 1 and call("100_5_kmeans", E=65) == 1  # PBN_ERR_ARG
    assert call("100_5_kmeans", E=3, null_edges=True) == 1
    assert call("100_5_kmeans", E=0, null_edges=True) == 0 and call("100_5_kmeans", E=64) == 0
    assert call("tt600", E=1) == 3  # PBN_ERR_UNSUPPORTED: threshold table in global memory
    assert call("tt600", E=0) == 0


def _tt_env():
    """A 6-node truth-table target env with an obvious best edge pin: targets 3 and 4 copy node 1, node 1 copies node 2 (a
    coin flip) nine times in ten.  Forcing node 1 to read 1 from node 2 puts the favourable pattern (1, 1) on about 3/4 of
    the mass (exact law at p = 0.01: 0.749, against 0.371 unpinned); a pin on one target's input reaches 0.481 at most."""
    from gym_PBN.b200 import compiler
    from gym_PBN.envs.bittner import base
    from gym_PBN.envs.pbn_target import PBNTargetEnv

    def node(inputs, table, name):
        mask = np.zeros(6, bool)
        mask[list(inputs)] = True
        return (mask, np.asarray(table, np.float64).reshape([2] * len(inputs)) if inputs else np.array(table), name, not inputs)

    data = [node([], 0.5, "n0"), node([2], [0.1, 0.9], "n1"), node([], 0.5, "n2"), node([1], [0.0, 1.0], "n3"),
            node([1], [0.0, 1.0], "n4"), node([3, 4], [0.5, 0.5, 0.5, 0.5], "n5")]
    spec = compiler.compile_pbn_data(data)
    spec.ids = list(range(spec.n))
    goal = {"target_nodes": [3, 4], "intervene_on": [1], "target_node_values": ((1, 1),), "undesired_node_values": ((0, 0),),
            "horizon": 100}
    return PBNTargetEnv(base.Graph.from_spec(spec), goal)


def test_rank_edge_pins_finds_the_obvious_edge(eng):
    from gym_PBN.utils import control

    env = _tt_env()
    edges = control.regulatory_edges(env)
    assert edges == [(2, 1), (1, 3), (1, 4), (3, 5), (4, 5)]
    res = control.rank_edge_pins(env, iters=4000, chains=2048, bit_flip_prob=0.01, seed=3)
    assert len(res["ranking"]) == 2 * len(edges)
    assert all(a["increase"] >= b["increase"] for a, b in zip(res["ranking"], res["ranking"][1:]))
    best = res["ranking"][0]
    assert (best["src"], best["dst"], best["value"]) == (2, 1, 1) and (best["src_node"], best["dst_node"]) == (2, 1)
    assert best["target_mass"] > 0.7 and best["increase"] > res["ranking"][1]["increase"] + 0.2  # exact: 0.749, next 0.481
    worst = res["ranking"][-1]
    assert worst["value"] == 0 and worst["target_mass"] < 0.1
    assert 0.3 < res["unpinned"]["target_mass"] < 0.7
    # the rows are pinned_ssd's on the same seed
    h = control.pinned_ssd(env, [{}, {(2, 1): 1}, {(1, 3): 0}], 4000, 2048, seed=3).astype(np.float64)
    assert abs(h[1][3] / h[1].sum() - best["target_mass"]) < 1e-12
    row = next(r for r in res["ranking"] if (r["src"], r["dst"], r["value"]) == (1, 3, 0))
    assert abs(h[2][3] / h[2].sum() - row["target_mass"]) < 1e-12 and abs(h[0][3] / h[0].sum() - res["unpinned"]["target_mass"]) < 1e-12
    with pytest.raises(ValueError, match="not a regulatory edge"):
        control.pinned_ssd(env, [{(3, 1): 1}], 10, 64)
    with pytest.raises(ValueError, match="0 or 1"):
        control.pinned_ssd(env, [{(2, 1): 2}], 10, 64)


def test_gene_id_edges_on_a_bittner_env(eng):
    """Edge keys by gene id give the node-index form's histograms, and a pair of genes that is not an edge is refused."""
    import gym_PBN
    from gym_PBN.utils import control

    env = gym_PBN.make("gym-PBN/Bittner-28-v0").unwrapped
    ids = env.graph.getIDs()
    edges = control.regulatory_edges(env)
    assert len(edges) == 420 and all(s in ids and d in ids for s, d in edges)
    (s, d), (s2, d2) = edges[40], edges[77]
    by_id = control.pinned_ssd(env, [{}, {(s, d): 1}, {(s2, d2): 0, ids[3]: 1}], 200, 256, seed=1)
    by_idx = control.pinned_ssd(env, [{}, {(ids.index(s), ids.index(d)): 1}, {(ids.index(s2), ids.index(d2)): 0, 3: 1}],
                                200, 256, seed=1)
    assert np.array_equal(by_id, by_idx) and not np.array_equal(by_id[0], by_id[2])
    non = next((a, b) for b in ids for a in ids if (a, b) not in edges)
    with pytest.raises(ValueError, match="not a regulatory edge"):
        control.pinned_ssd(env, [{non: 1}], 10, 64)

