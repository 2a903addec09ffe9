"""GPU: pbn_ssd_pinned (SSD estimates with genes pinned) against the oracle's orc_ssd_pinned bit for bit on every path of the
SSD loop, against pbn_ssd when nothing is pinned, against the exact stationary law of a small network, and through
gym_PBN.utils.control (pinned_ssd, rank_pins)."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402
import pinned_oracle as po  # noqa: E402
from golden_util import random_predictor_sets, random_tt_data  # noqa: E402
from pinned_util import exact_pinned_law  # noqa: E402


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


def _unpack(eng, planes, B, n):
    out = torch.empty((B, n), dtype=torch.uint8, device=planes.device)
    eng.abi.check(eng.abi.lib().pbn_unpack_state(C.c_void_p(planes.data_ptr()), B, n, C.c_void_p(out.data_ptr()),
                                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out.cpu().numpy()


def _run(eng, net, pins, chains, iters, p, tgt, seed, env0, care_value=None):
    """Device run from rand_state (epoch 0), the pinned SSD in epoch 1: (hist [K][2^g], final states [K][chains][N])."""
    K = len(pins)
    sim = eng.engine.Simulator(net, chains, seed=seed, env0=env0)
    sim.rand_state()
    state = sim.state.repeat(1, K)
    hist = torch.zeros((K, 1 << len(tgt)), dtype=torch.int64, device=sim.device)
    care, value = care_value if care_value is not None else _masks(pins, net.n)
    eng.engine.ssd_pinned(sim, state, iters, p, tgt, care, value, hist)
    return hist.cpu().numpy().astype(np.uint64), _unpack(eng, state, K * chains, net.n).reshape(K, chains, net.n)


def _pins(n, K, tgt, rng):
    """{} first, then K - 1 random pin sets of 1..6 nodes, every second one with a target gene among them."""
    out = [{}]
    for k in range(1, K):
        nodes = set(int(i) for i in rng.choice(n, size=int(rng.integers(1, 7)), replace=False))
        if k % 2:
            nodes.add(int(tgt[int(rng.integers(0, len(tgt)))]))
        out.append({i: int(rng.integers(0, 2)) for i in sorted(nodes)})
    return out


def _single_gene_pins(n):
    return [{}] + [{i: v} for i in range(n) for v in (0, 1)]


CASES = [  # which, chains, iters, p, targets, K
    ("pred20", 96, 41, 0.3, list(range(0, 7)), 3),              # static loop, several rounds per iteration
    ("pred256", 64 + 5, 40, 0.01, list(range(200, 207)), 3),    # 8-word states, a partial warp next to the static loop
    ("28_15_median", 160, 9, 0.01, [20, 21, 22, 23], 3),        # two-level threshold rows (TQ 4), odd iteration count
    ("100_5_kmeans", 96, 7, 1e-6, list(range(0, 7)), 201),      # every single-gene pin; rounds far apart
    ("100_5_kmeans", 3000, 400, 0.01, list(range(0, 7)), 3),    # the headline shape, smaller
    ("100_5_kmeans", 64, 10, 0.0, [3, 41, 69, 7], 3),           # no perturbation, scattered targets (generic loop)
    ("100_5_kmeans", 128, 10, 0.3, list(range(40, 53)), 3),     # g = 13: global-memory histogram
    ("100_5_kmeans", 32, 1, 0.01, list(range(0, 7)), 1),        # K = 1, one iteration (the generic tail only)
    ("tt70", 96, 9, 0.3, [1, 2, 3], 3),                          # truth table, threshold table in shared memory
    ("tt600", 70, 11, 0.01, [3, 41, 69, 7, 500], 3),             # truth table, threshold table in global memory
    ("tt1024", 64, 5, 0.3, list(range(1000, 1006)), 3),          # 32-word states
]


@pytest.mark.parametrize("which,chains,iters,p,tgt,K", CASES)
def test_pinned_ssd_matches_oracle(eng, which, chains, iters, p, tgt, K):
    net, onet = _nets(eng, which)
    tgt = np.array(tgt, np.int32)
    pins = _single_gene_pins(net.n) if K == 201 else _pins(net.n, K, tgt, np.random.default_rng(len(tgt) + K))
    seed, env0 = 17, 64
    hist, out = _run(eng, net, pins, chains, iters, p, tgt, seed, env0)
    ost = orc.rand_state(onet, chains, orc.Draws(seed=seed, epoch=0), env0=env0)
    ohist, oout = po.ssd_pinned(onet, ost, iters, p, pins, tgt, orc.Draws(seed=seed, epoch=1), env0=env0)
    assert (hist.sum(1) == chains * iters).all()
    assert np.array_equal(hist, ohist)
    assert np.array_equal(out, oout)


@pytest.mark.parametrize("K,chains,iters", [(1, 65536, 1000), (201, 4096, 200)])
def test_unpinned_row_is_pbn_ssd(eng, K, chains, iters):
    """Bittner-100, the seven targets, p = 0.01: the row without pins is pbn_ssd's estimate on the same draws, bit for bit
    (histogram and final states), alone and as row 0 of a 201-variant launch."""
    net, _ = _nets(eng, "100_5_kmeans")
    tgt = np.arange(7, dtype=np.int32)
    pins = [{}] if K == 1 else _single_gene_pins(net.n)
    hist, out = _run(eng, net, pins, chains, iters, 0.01, tgt, seed=3, env0=0)
    sim = eng.engine.Simulator(net, chains, seed=3)
    sim.rand_state()
    ref = sim.ssd(iters, 0.01, tgt).cpu().numpy().astype(np.uint64)
    assert np.array_equal(hist[0], ref)
    assert np.array_equal(out[0], sim.unpack().cpu().numpy())


@pytest.mark.parametrize("which", ["100_5_kmeans", "tt70"])
def test_pins_hold(eng, which):
    """p = 0.3: every final state carries its pins, and no counted state contradicts a pinned target gene."""
    net, _ = _nets(eng, which)
    tgt = np.array([1, 2, 3, 4, 5], np.int32)
    pins = [{2: 1}, {4: 0, 30: 1}, {1: 1, 3: 0, 5: 1, 60: 0}]
    hist, out = _run(eng, net, pins, 1000, 500, 0.3, tgt, seed=5, env0=0)
    for k, pin in enumerate(pins):
        for i, v in pin.items():
            assert (out[k][:, i] == v).all()
            if i in tgt:
                pos = len(tgt) - 1 - list(tgt).index(i)
                bad = [b for b in range(1 << len(tgt)) if (b >> pos) & 1 != v]
                assert hist[k][bad].sum() == 0 and hist[k].sum() == 1000 * 500


def test_value_bits_outside_care_are_ignored(eng):
    """Value bits of unpinned nodes, and care and value bits at or above N, change nothing."""
    tgt = np.arange(7, dtype=np.int32)
    pins = [{0: 1, 100: 0}, {255: 1}, {}]
    net, _ = _nets(eng, "pred256")
    care, value = _masks(pins, net.n)
    a = _run(eng, net, pins, 256, 60, 0.05, tgt, 9, 0, care_value=(care, value))
    b = _run(eng, net, pins, 256, 60, 0.05, tgt, 9, 0, care_value=(care, value | (~care & np.uint32(0xA5A5A5A5))))
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    net, _ = _nets(eng, "tt70")  # 26 unused bits in the last state word
    pins = [{0: 1, 60: 0}, {5: 1}, {}]
    care, value = _masks(pins, net.n)
    care2 = care.copy()
    care2[:, -1] |= np.uint32(0xFFFFFFFF) << np.uint32(70 & 31)
    a = _run(eng, net, pins, 128, 40, 0.05, tgt, 9, 0, care_value=(care, value))
    b = _run(eng, net, pins, 128, 40, 0.05, tgt, 9, 0, care_value=(care2, value | ~care))
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_exact_law(eng):
    """An 8-node truth-table network with two genes pinned: 16 independent batches of 8192 chains x 20 000 iterations (after
    a burn-in) are within 0.005 in total variation of the exact stationary law, and within 5 batch-means standard errors in
    every bucket."""
    data = random_tt_data(8, seed=12)
    net = eng.engine.Network(eng.compiler.compile_pbn_data(data))
    pin, p, tgt = {2: 1, 5: 0}, 0.05, np.array([1, 2, 4, 7], np.int32)
    exact = exact_pinned_law(data, pin, p, tgt)
    care, value = _masks([pin], net.n)
    batches = []
    for b in range(16):
        sim = eng.engine.Simulator(net, 8192, seed=21, env0=8192 * b)
        sim.rand_state()
        state = sim.state.clone()
        burn = torch.zeros((1, 16), dtype=torch.int64, device=sim.device)
        eng.engine.ssd_pinned(sim, state, 500, p, tgt, care, value, burn)
        hist = torch.zeros((1, 16), dtype=torch.int64, device=sim.device)
        eng.engine.ssd_pinned(sim, state, 20000, p, tgt, care, value, hist)
        h = hist.cpu().numpy()[0].astype(np.float64)
        batches.append(h / h.sum())
    batches = np.array(batches)
    est, se = batches.mean(0), batches.std(0, ddof=1) / np.sqrt(len(batches))
    assert 0.5 * np.abs(est - exact).sum() < 0.005
    assert (np.abs(est - exact) <= 5 * se + 1e-12).all()


def test_sharded_launches_sum_to_one(eng):
    """Chains 0..95 and 96..255 in two launches (env0 = 0 and 96) give the histogram and final states of one launch."""
    net, _ = _nets(eng, "100_5_kmeans")
    tgt = np.arange(7, dtype=np.int32)
    pins = _pins(net.n, 5, tgt, np.random.default_rng(2))
    full_h, full_s = _run(eng, net, pins, 256, 300, 0.01, tgt, 4, 0)
    h0, s0 = _run(eng, net, pins, 96, 300, 0.01, tgt, 4, 0)
    h1, s1 = _run(eng, net, pins, 160, 300, 0.01, tgt, 4, 96)
    assert np.array_equal(full_h, h0 + h1)
    assert np.array_equal(full_s, np.concatenate([s0, s1], axis=1))


def test_argument_errors(eng):
    net, _ = _nets(eng, "100_5_kmeans")
    lib, abi = eng.abi.lib(), eng.abi
    state = torch.zeros((net.w32, 64 * 65535), dtype=torch.int32, device="cuda")  # room for the largest K
    masks = torch.zeros((65535, net.w32), dtype=torch.int32, device="cuda")
    hist = torch.zeros((65535, 1 << 7), dtype=torch.int64, device="cuda")
    ptr = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    def call(K=2, env0=0, p=0.01, g=7, draws=None):
        tgt = np.arange(max(g, 1), dtype=np.int32)
        d = draws or abi.PbnDraws(mode=abi.DRAW_PHILOX, seed=1, epoch=1)
        return lib.pbn_ssd_pinned(net.handle, ptr(state), 64, env0, 10, p, ptr(masks), ptr(masks), K,
                                  tgt.ctypes.data_as(C.c_void_p), g, ptr(hist), C.byref(d), None)

    ints = torch.zeros((64, 1), dtype=torch.int32, device="cuda")
    dbls = torch.zeros((64, 1), dtype=torch.float64, device="cuda")
    replay = abi.PbnDraws(mode=abi.DRAW_REPLAY, ints=ptr(ints), dbls=ptr(dbls), int_stride=1, dbl_stride=1)
    assert call(draws=replay) == 3  # PBN_ERR_UNSUPPORTED
    for kw in ({"K": 0}, {"K": 65536}, {"env0": 5}, {"g": 0}, {"g": 25}):
        assert call(**kw) == 1, kw  # PBN_ERR_ARG
    assert call(env0=5, p=0.0) == 0  # the alignment is only needed with perturbations
    assert call(K=65535) == 0
    torch.cuda.synchronize()


def _tt_env():
    """A 6-node truth-table target env with an obvious best pin: targets 3 and 4 copy node 1, node 1 copies node 2 (a coin
    flip) most of the time; pinning node 1 at 1 puts the favourable pattern (1, 1) on about all of the mass (all but the
    ~5 % of the time each target spends flipped away, at p = 0.01 and one update in five for each node)."""
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


def test_rank_pins_finds_the_obvious_pin(eng):
    from gym_PBN.utils import control

    env = _tt_env()
    res = control.rank_pins(env, iters=4000, chains=2048, bit_flip_prob=0.01, seed=3)
    best = res["ranking"][0]
    assert (best["node"], best["value"]) == (1, 1)
    assert best["target_mass"] > 0.9 and best["undesired_mass"] < 0.01
    second = res["ranking"][1]  # node 2 -> 1: node 1 then follows it nine times in ten
    assert (second["node"], second["value"]) == (2, 1) and best["increase"] > second["increase"] + 0.1
    assert 0.3 < res["unpinned"]["target_mass"] < 0.7
    assert len(res["ranking"]) == 12
    assert all(a["increase"] >= b["increase"] for a, b in zip(res["ranking"], res["ranking"][1:]))
    worst = res["ranking"][-1]
    assert worst["value"] == 0 and worst["node"] in (1, 3, 4)
    # pinned_ssd by gene id on the same env: the rows of rank_pins' launch
    h = control.pinned_ssd(env, [{}, {1: 1}], 4000, 2048, seed=3)
    assert h.shape == (2, 4) and (h.sum(1) == 4000 * 2048).all()
    assert abs(h[1][3] / h[1].sum() - best["target_mass"]) < 1e-12
