"""GPU: pbn_first_passage (first-passage times into goal patterns under node and edge pins) against the oracle's
orc_first_passage bit for bit on every path of the SSD loop, against pbn_ssd_pinned_edges with an empty goal, chunked and
sharded, against the exact first-passage law of small networks, and through gym_PBN.utils.control (first_passage, the
passage measure of rank_pins and rank_edge_pins)."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402
import passage_oracle as pao  # noqa: E402
from edge_pin_util import edge_rows, edges_of  # noqa: E402
from golden_util import random_predictor_sets, random_tt_data  # noqa: E402
from passage_util import exact_passage  # noqa: E402


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
    """(device network, oracle network); truth-table networks of 600 and 1024 nodes read their threshold table from global
    memory, the 70-node one stages it."""
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


def _words(goal, g):
    w = np.zeros(max(1, (1 << g) // 32), np.uint32)
    for b in goal:
        w[b >> 5] |= np.uint32(1 << (b & 31))
    return w


def _unpack(eng, planes, B, n):
    out = torch.empty((B, n), dtype=torch.uint8, device=planes.device)
    eng.abi.check(eng.abi.lib().pbn_unpack_state(C.c_void_p(planes.data_ptr()), B, n, C.c_void_p(out.data_ptr()),
                                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out.cpu().numpy()


def _run(eng, net, pins, edges, chains, chunks, p, tgt, goal, seed, env0, t_hit=None):
    """Device run from rand_state (epoch 0), then one first-passage launch per entry of `chunks` (iteration counts, epochs
    1, 2, ..., t0 carried): (t_hit [K][chains], final states [K][chains][N])."""
    K = len(pins)
    sim = eng.engine.Simulator(net, chains, seed=seed, env0=env0)
    sim.rand_state()
    state = sim.state.repeat(1, K)
    hit = torch.full((K, chains), -1, dtype=torch.int64, device=sim.device) if t_hit is None else \
        torch.from_numpy(np.ascontiguousarray(t_hit, np.int64)).to(sim.device)
    care, value = _masks(pins, net.n)
    t0 = 0
    for it in chunks:
        eng.engine.first_passage(sim, state, it, t0, p, tgt, _words(goal, len(tgt)), care, value, hit, edges=edges)
        t0 += it
    return hit.cpu().numpy(), _unpack(eng, state, K * chains, net.n).reshape(K, chains, net.n)


def _oracle(onet, pins, edges, chains, chunks, p, tgt, goal, seed, env0, t_hit=None):
    st = orc.rand_state(onet, chains, orc.Draws(seed=seed, epoch=0), env0=env0)
    t0 = 0
    for e, it in enumerate(chunks):
        t_hit, st = pao.first_passage(onet, st, it, p, pins, tgt, goal, orc.Draws(seed=seed, epoch=1 + e), env0=env0,
                                      edges=edges, t0=t0, t_hit=t_hit)
        t0 += it
    return t_hit, st


def _variants(onet, K, rng, edges=True):
    """{} first, then K - 1 variants of 0..3 node pins and (edges=True) 0..4 edge pins, empty slots among them."""
    n, all_edges = onet.n, edges_of(onet)
    pins, rows = [{}], [[]]
    for k in range(1, K):
        pins.append({int(i): int(rng.integers(0, 2)) for i in rng.choice(n, size=int(rng.integers(0, 4)), replace=False)})
        m = int(rng.integers(0, 5)) if edges else 0
        rows.append([all_edges[int(j)] + (int(rng.integers(0, 2)),) for j in rng.choice(len(all_edges), size=m, replace=False)])
    return pins, (edge_rows(rows, E=max(len(r) for r in rows) + 1) if edges else None)


def _goal(g, frac):
    """A fixed random set of buckets (each in it w.p. frac), or frac itself when it is a list of buckets."""
    if isinstance(frac, list):
        return frac
    return [int(b) for b in np.flatnonzero(np.random.default_rng(g).random(1 << g) < frac)]


CASES = [  # which, chains, iters, p, targets, K (201: every single-gene pin), goal (bucket fraction or list), edge pins
    ("pred20", 96, 41, 0.3, list(range(0, 7)), 6, 0.02, True),             # static loop, several rounds per iteration
    ("pred256", 64 + 5, 40, 0.01, list(range(200, 207)), 5, 0.1, True),    # 8-word states, a partial warp next to it
    ("28_15_median", 160, 9, 0.01, [20, 21, 22, 23], 6, 0.4, True),        # two-level threshold rows (TQ 4), odd count
    ("100_5_kmeans", 96, 7, 1e-6, list(range(0, 7)), 201, 0.25, False),    # every single-gene pin; rounds far apart
    ("100_5_kmeans", 3000, 400, 0.01, list(range(0, 7)), 5, 0.02, True),   # the headline shape, smaller
    ("100_5_kmeans", 64, 10, 0.0, [3, 41, 69, 7], 5, 0.4, True),           # no perturbation, scattered targets (generic)
    ("tt70", 96, 9, 0.3, [1, 2, 3], 6, [0], True),                         # truth table, threshold table in shared memory
    ("tt600", 70, 11, 0.01, [3, 41, 69, 7, 500], 3, 0.25, False),          # threshold table in global memory: E = 0
    ("tt1024", 64, 5, 0.3, list(range(1000, 1006)), 3, 0.1, False),        # 32-word states (table in global memory)
]
IDS = [f"{c[0]}-{c[1]}x{c[2]}-p{c[3]}" for c in CASES]


def _case(eng, which, chains, iters, p, tgt, K, frac, with_edges):
    net, onet = _nets(eng, which)
    tgt = np.array(tgt, np.int32)
    if K == 201:
        pins, edges = [{}] + [{i: v} for i in range(net.n) for v in (0, 1)], None
    else:
        pins, edges = _variants(onet, K, np.random.default_rng(len(tgt) + K), with_edges)
    return net, onet, tgt, pins, edges, _goal(len(tgt), frac)


@pytest.mark.parametrize("which,chains,iters,p,tgt,K,frac,with_edges", CASES, ids=IDS)
def test_passage_matches_oracle(eng, which, chains, iters, p, tgt, K, frac, with_edges):
    net, onet, tgt, pins, edges, goal = _case(eng, which, chains, iters, p, tgt, K, frac, with_edges)
    hit, out = _run(eng, net, pins, edges, chains, [iters], p, tgt, goal, 17, 64)
    ohit, oout = _oracle(onet, pins, edges, chains, [iters], p, tgt, goal, 17, 64)
    assert 0.1 < (ohit >= 0).mean() < 0.9  # some chains arrive, some do not
    assert np.array_equal(hit, ohit)
    assert np.array_equal(out[hit < 0], oout[ohit < 0])


@pytest.mark.parametrize("which,chains,iters,p,tgt,K,frac,with_edges", CASES, ids=IDS)
def test_empty_goal_is_ssd_pinned_edges(eng, which, chains, iters, p, tgt, K, frac, with_edges):
    """No chain stops, and every final state is pbn_ssd_pinned_edges's with the same arguments, bit for bit."""
    net, _, tgt, pins, edges, _ = _case(eng, which, chains, iters, p, tgt, K, frac, with_edges)
    hit, out = _run(eng, net, pins, edges, chains, [iters], p, tgt, [], 17, 64)
    assert (hit == -1).all()
    sim = eng.engine.Simulator(net, chains, seed=17, env0=64)
    sim.rand_state()
    state = sim.state.repeat(1, len(pins))
    care, value = _masks(pins, net.n)
    hist = torch.zeros((len(pins), 1 << len(tgt)), dtype=torch.int64, device=sim.device)
    eng.engine.ssd_pinned(sim, state, iters, p, tgt, care, value, hist, edges=edges)
    assert np.array_equal(out, _unpack(eng, state, len(pins) * chains, net.n).reshape(out.shape))


@pytest.mark.parametrize("which,chains,iters,p,tgt,K,frac,with_edges", CASES, ids=IDS)
def test_full_goal_stops_at_t0(eng, which, chains, iters, p, tgt, K, frac, with_edges):
    """With every bucket in the goal, every chain arrives at t0."""
    net, _, tgt, pins, edges, _ = _case(eng, which, chains, iters, p, tgt, K, frac, with_edges)
    sim = eng.engine.Simulator(net, chains, seed=17, env0=64)
    sim.rand_state()
    state = sim.state.repeat(1, len(pins))
    t_hit = torch.full((len(pins), chains), -1, dtype=torch.int64, device=sim.device)
    care, value = _masks(pins, net.n)
    eng.engine.first_passage(sim, state, iters, 5, p, tgt, _words(range(1 << len(tgt)), len(tgt)), care, value, t_hit,
                             edges=edges)
    assert (t_hit.cpu().numpy() == 5).all()


def test_chunked_launches(eng):
    """Three launches carrying t0 and t_hit give the oracle's run with the same chunks and epochs; chains that entered with
    t_hit >= 0 keep their entry and their state column."""
    net, onet = _nets(eng, "100_5_kmeans")
    tgt = np.arange(7, dtype=np.int32)
    pins, edges = _variants(onet, 5, np.random.default_rng(3))
    goal = _goal(7, 0.02)
    entered = np.full((5, 256), -1, np.int64)
    entered[:, ::7] = 3  # arrived before the first launch
    hit, out = _run(eng, net, pins, edges, 256, [60, 61, 80], 0.01, tgt, goal, 5, 0, t_hit=entered)
    ohit, oout = _oracle(onet, pins, edges, 256, [60, 61, 80], 0.01, tgt, goal, 5, 0, t_hit=entered)
    assert np.array_equal(hit, ohit) and np.array_equal(out[hit < 0], oout[ohit < 0])
    assert (hit[:, ::7] == 3).all() and 0.1 < (hit >= 0).mean() < 0.9 and (hit >= 60).any()
    start = orc.rand_state(onet, 256, orc.Draws(seed=5, epoch=0))
    assert np.array_equal(out[:, ::7], np.repeat(start[None, ::7], 5, axis=0))


def test_sharded_launches(eng):
    """Chains 0..95 and 96..255 in two launches (env0 = 0 and 96) give the times and final states of one launch."""
    net, onet = _nets(eng, "100_5_kmeans")
    tgt = np.arange(7, dtype=np.int32)
    pins, edges = _variants(onet, 5, np.random.default_rng(2))
    goal = _goal(7, 0.02)
    full_h, full_s = _run(eng, net, pins, edges, 256, [300], 0.01, tgt, goal, 4, 0)
    h0, s0 = _run(eng, net, pins, edges, 96, [300], 0.01, tgt, goal, 4, 0)
    h1, s1 = _run(eng, net, pins, edges, 160, [300], 0.01, tgt, goal, 4, 96)
    assert np.array_equal(full_h, np.concatenate([h0, h1], axis=1))
    s = np.concatenate([s0, s1], axis=1)
    assert np.array_equal(full_s[full_h < 0], s[full_h < 0])


@pytest.mark.parametrize("kind", ["pred", "tt"])
def test_exact_law(eng, kind):
    """8-node networks with a node pin and an edge pin, 2^18 chains from uniform states: P(tau < T) and E[min(tau, T)]
    within 5 standard errors of the exact values."""
    if kind == "tt":
        data = random_tt_data(8, seed=12)
        net, onet = eng.engine.Network(eng.compiler.compile_pbn_data(data)), orc.net_from_pbn_data(data)
        pin, edges = {2: 1}, {(5, 1): 1}
    else:
        sets, ids = random_predictor_sets(8, 3, seed=5)
        net, onet = eng.engine.Network(eng.compiler.compile_predictor_sets(sets, ids)), orc.net_from_predictor_sets(sets, ids)
        pin, edges = {3: 0}, {(1, 7): 1}
    p, T, chains = 0.05, 20, 1 << 18
    tgt, goal = np.array([1, 4, 6], np.int32), [0b111]
    reached, mean = exact_passage(onet, pin, edges, p, tgt, goal, T)
    hit, _ = _run(eng, net, [pin], edge_rows([[(s, d, c) for (s, d), c in edges.items()]]), chains, [T], p, tgt, goal, 21, 0)
    r = (hit[0] >= 0).astype(np.float64)
    m = np.where(hit[0] >= 0, hit[0], T).astype(np.float64)
    assert abs(r.mean() - reached) <= 5 * r.std(ddof=1) / np.sqrt(chains)
    assert abs(m.mean() - mean) <= 5 * m.std(ddof=1) / np.sqrt(chains)


def test_argument_errors(eng):
    lib, abi = eng.abi.lib(), eng.abi
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    def call(which="100_5_kmeans", g=5, K=2, E=2, t0=0, iters=10, env0=0, null_goal=False, null_hit=False, replay=False):
        net, _ = _nets(eng, which)
        state = torch.zeros((net.w32, 64 * 2), dtype=torch.int32, device="cuda")
        masks = torch.zeros((2, net.w32), dtype=torch.int32, device="cuda")
        edges = torch.full((2, 65), -1, dtype=torch.int32, device="cuda")
        t_hit = torch.full((2, 64), -1, dtype=torch.int64, device="cuda")
        tgt = np.arange(g, dtype=np.int32)
        goal = np.zeros(max(1, (1 << g) // 32), np.uint32)
        d = abi.PbnDraws(mode=abi.DRAW_PHILOX, seed=1, epoch=1)
        if replay:
            d.mode = abi.DRAW_REPLAY
        rc = lib.pbn_first_passage(net.handle, ptr(state), 64, env0, iters, t0, 0.01, ptr(masks), ptr(masks), K, ptr(edges), E,
                                   tgt.ctypes.data_as(C.c_void_p), g, None if null_goal else goal.ctypes.data_as(C.c_void_p),
                                   None if null_hit else ptr(t_hit), C.byref(d), None)
        torch.cuda.synchronize()
        return rc

    assert call() == 0 and call(g=12) == 0 and call(g=1) == 0
    assert call(g=13) == 1 and call(g=0) == 1  # PBN_ERR_ARG
    assert call(null_goal=True) == 1 and call(null_hit=True) == 1
    assert call(t0=-1) == 1 and call(iters=1 << 31) == 1
    assert call(env0=16) == 1
    assert call(K=0) == 1 and call(K=65536) == 1 and call(E=-1) == 1 and call(E=65) == 1
    assert call(replay=True) == 3  # PBN_ERR_UNSUPPORTED
    assert call("tt600", E=1) == 3 and call("tt600", E=0) == 0


def _tt_env(targets, values):
    """A 6-node truth-table target env: targets 3 and 4 copy node 1, node 1 copies node 2 (a coin flip) nine times in ten."""
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
    goal = {"target_nodes": targets, "intervene_on": [1], "target_node_values": values, "undesired_node_values": (),
            "horizon": 100}
    return PBNTargetEnv(base.Graph.from_spec(spec), goal)


def test_rank_pins_by_passage(eng):
    """With target node 3 and goal (1,), the pin 3 -> 1 is there at time 0 in every chain and ranks first; 3 -> 0 never
    gets there and ranks last; rank_edge_pins(measure="passage") runs and puts (2, 1) -> 1 ahead of (2, 1) -> 0."""
    from gym_PBN.utils import control

    env = _tt_env([3], ((1,),))
    res = control.rank_pins(env, iters=200, chains=512, seed=3, measure="passage")
    assert len(res["ranking"]) == 12
    assert all(a["change"] <= b["change"] for a, b in zip(res["ranking"], res["ranking"][1:]))
    best, worst = res["ranking"][0], res["ranking"][-1]
    assert (best["node"], best["value"]) == (3, 1) and best["mean_time"] == 0.0 and best["reached"] == 1.0
    assert (worst["node"], worst["value"]) == (3, 0) and worst["reached"] == 0.0 and worst["mean_time"] == 200.0
    assert res["unpinned"]["reached"] > 0.9 and best["change"] == -res["unpinned"]["mean_time"]
    res = control.rank_edge_pins(env, iters=200, chains=512, seed=3, measure="passage")
    assert len(res["ranking"]) == 2 * len(control.regulatory_edges(env))
    order = [(r["src"], r["dst"], r["value"]) for r in res["ranking"]]
    assert order.index((2, 1, 1)) < order.index((2, 1, 0)) and order[-1] in ((1, 3, 0), (2, 1, 0))
    assert "target_mass" not in res["ranking"][0] and "mean_time" in res["ranking"][0]
    # the default measure is unchanged
    assert "increase" in control.rank_pins(env, iters=50, chains=64)["ranking"][0]


def test_first_passage_api(eng):
    """Shapes, the source column of reset starts, explicit starts, and the distributed table (one rank)."""
    import gym_PBN
    from gym_PBN.utils import control

    env = gym_PBN.make("gym-PBN/Bittner-100-v0").unwrapped
    A = len(env.all_attractors)
    ids = env.graph.getIDs()
    pins = [{}, {ids[3]: 1}, {ids[5]: 0, control.regulatory_edges(env)[7]: 1}]
    res = control.first_passage(env, pins, 500, 100, seed=2)
    assert res["time"].shape == (3, 100) and res["time"].dtype == np.int64 and (res["time"] >= -1).all()
    assert res["source"].shape == (100,) and ((res["source"] >= 0) & (res["source"] < A)).all()
    dist = control.first_passage(env, pins, 500, 100, seed=2, distributed=True)
    assert np.array_equal(dist["time"], res["time"]) and np.array_equal(dist["source"], res["source"])
    start = np.zeros((100, env.network.n), np.uint8)
    own = control.first_passage(env, pins, 500, 100, start=start, seed=2)
    assert own["source"] is None and own["time"].shape == (3, 100)
    with pytest.raises(ValueError, match="start must be"):
        control.first_passage(env, pins, 10, 100, start=start[:5])
