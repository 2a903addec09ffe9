"""GPU: the CUDA path (through the C-ABI) against (a) golden traces recorded from the reference, replayed
draw for draw, and (b) the C oracle in Philox mode at larger sizes.  Everything here is bit-exact."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402
from golden_util import Traj, cubes_to_attractors, load, pbn_data_from, random_predictor_net, random_tt_data  # noqa: E402


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gym_PBN.b200 import abi, compiler, engine

    class E:
        pass

    e = E()
    e.abi, e.compiler, e.engine = abi, compiler, engine
    return e


def _state_np(sim):
    return sim.unpack().cpu().numpy()


def _replay(eng, ints, dbls):
    return eng.engine.Replay(np.asarray(ints, np.int32).reshape(1, -1), np.asarray(dbls, np.float64).reshape(1, -1), "cuda", B=1)


def _used(rp):
    return tuple(rp.used.cpu().numpy()[0])


# ------------------------------------------------------------------------------------------------ golden replays
@pytest.mark.parametrize("name", ["b28_graph_core.npz", "b100_graph_core.npz", "b200_graph_core.npz"])
def test_golden_graph_core(eng, name):
    z = load(name)
    net = eng.engine.Network(eng.compiler.load_bittner(str(z["pickle"])))
    for e in range(int(z["n_traj"])):
        tr = Traj(z, e)
        sim = eng.engine.Simulator(net, 1)
        rp = _replay(eng, *tr.draws(0))
        sim.rand_state(replay=rp)
        assert np.array_equal(_state_np(sim)[0], tr.state[0])
        # async segment in ONE launch per flip-free stretch would hide per-step states; go op by op
        for t in range(1, tr.T):
            ints, dbls = tr.draws(t)
            rp = _replay(eng, ints, dbls)
            if tr.op[t] == 0:
                a = int(tr.act[t, 0])
                if a >= 0:
                    sim.state[a >> 5, 0] ^= np.int32(np.uint32(1 << (a & 31)).view(np.int32))
                sim.rollout(1, replay=rp)
            else:
                sim.rollout(1, sync=True, replay=rp)
            assert _used(rp) == (len(ints), len(dbls))
            assert np.array_equal(_state_np(sim)[0], tr.state[t]), (name, e, t)


def test_golden_graph_core_multistep(eng):
    """400 async updates of the golden trace in a single launch (state stays on chip)."""
    z = load("b100_graph_core.npz")
    net = eng.engine.Network(eng.compiler.load_bittner(str(z["pickle"])))
    tr = Traj(z, 0)
    # stretches between flips: 5 steps each
    sim = eng.engine.Simulator(net, 1)
    sim.set_state(tr.state[0:1])
    t = 1
    while t < tr.T and tr.op[t] == 0:
        a = int(tr.act[t, 0])
        if a >= 0:
            sim.state[a >> 5, 0] ^= np.int32(np.uint32(1 << (a & 31)).view(np.int32))
        t1 = t + 1
        while t1 < tr.T and tr.op[t1] == 0 and tr.act[t1, 0] < 0:
            t1 += 1
        ints, dbls = tr.draws(t, t1)
        sim.rollout(t1 - t, replay=_replay(eng, ints, dbls))
        assert np.array_equal(_state_np(sim)[0], tr.state[t1 - 1]), t
        t = t1


def test_golden_tt_core(eng):
    z = load("tt40_core.npz")
    net = eng.engine.Network(eng.compiler.compile_pbn_data([(m, t, f"n{i}", False) for i, (m, t) in enumerate(pbn_data_from(z))]))
    tr = Traj(z, 0)
    sim = eng.engine.Simulator(net, 1)
    sim.set_state(tr.state[0:1])
    for t in range(1, tr.T):
        ints, dbls = tr.draws(t)
        rp = _replay(eng, ints, dbls)
        a = int(tr.act[t, 0])
        if a >= 0:
            sim.state[a >> 5, 0] ^= np.int32(np.uint32(1 << (a & 31)).view(np.int32))
        sim.rollout(1, replay=rp)
        assert _used(rp) == (len(ints), len(dbls))
        assert np.array_equal(_state_np(sim)[0], tr.state[t]), t


def _run_env_trace(eng, net, env, tr, K):
    sim = eng.engine.Simulator(net, 1)
    for t in range(tr.T):
        ints, dbls = tr.draws(t)
        rp = _replay(eng, ints, dbls)
        if tr.op[t] == 1:
            sim.env_reset(env, replay=rp)
            assert _used(rp) == (len(ints), len(dbls))
            assert np.array_equal(_state_np(sim)[0], tr.state[t]), ("reset", t)
            if tr.target_att[t] >= 0:
                assert int(sim.target_att[0]) == tr.target_att[t]
        else:
            sim.env_step(env, torch.from_numpy(tr.act[t:t + 1, :K].copy()), replay=rp)
            assert _used(rp) == (len(ints), len(dbls)), t
            assert np.array_equal(_state_np(sim)[0], tr.state[t]), ("state", t)
            assert np.array_equal(sim.unpack(sim.obs_state).cpu().numpy()[0], tr.obs[t]), ("obs", t)
            got = (int(sim.reward[0]), int(sim.terminated[0]), int(sim.truncated[0]))
            assert got == (tr.reward[t], tr.term[t], tr.trunc[t]), ("reward", t)


def test_golden_pbn_env_ex5(eng):
    z = load("ex5_pbnenv.npz")
    net = eng.engine.Network(eng.compiler.compile_pbn_data([(m, t, f"n{i}", False) for i, (m, t) in enumerate(pbn_data_from(z))]))
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = eng.engine.EnvImage(net, eng.abi.ENV_PBN, attractors=atts, targets=[tuple(t) for t in z["targets"]])
    for e in range(int(z["n_traj"])):
        _run_env_trace(eng, net, env, Traj(z, e), 1)


def test_golden_pbcn_and_sampled_data(eng):
    z = load("ex5_pbcn_sampled.npz")
    net = eng.engine.Network(eng.compiler.compile_pbn_data([(m, t, f"n{i}", False) for i, (m, t) in enumerate(pbn_data_from(z))]))
    kinds = [eng.abi.ENV_PBCN, eng.abi.ENV_PBCN_SD, eng.abi.ENV_PBN_SD]
    for e, kind in enumerate(kinds):
        atts = cubes_to_attractors(z[f"e{e}/att_cubes"], z[f"e{e}/att_off"])
        env = eng.engine.EnvImage(net, kind, attractors=atts, targets=[tuple(t) for t in z["targets"]],
                                  n_control=int(z[f"e{e}/M"]), successful_reward=int(z[f"e{e}/successful_reward"]),
                                  wrong_attractor_cost=int(z[f"e{e}/wrong_attractor_cost"]))
        _run_env_trace(eng, net, env, Traj(z, e), 1 if e == 0 else 2)


@pytest.mark.parametrize("fname", ["b28_target_env.npz", "b100_target_env.npz"])
def test_golden_target_env(eng, fname):
    z = load(fname)
    net = eng.engine.Network(eng.compiler.load_bittner(str(z["pickle"])))
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    for e in range(int(z["n_traj"])):
        env = eng.engine.EnvImage(net, eng.abi.ENV_TARGET, attractors=atts, horizon=int(z["horizon"]),
                                  max_inner=int(z["cap"]), force=bool(z[f"e{e}/force"]))
        _run_env_trace(eng, net, env, Traj(z, e), 1)


@pytest.mark.parametrize("fname", ["b28_multi_env.npz", "b100_multi_env.npz"])
def test_golden_multi_env(eng, fname):
    z = load(fname)
    net = eng.engine.Network(eng.compiler.load_bittner(str(z["pickle"])))
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    for e in range(int(z["n_traj"])):
        env = eng.engine.EnvImage(net, eng.abi.ENV_MULTI, attractors=atts, horizon=int(z["horizon"]),
                                  max_inner=int(z["cap"]), dedup=bool(z[f"e{e}/dedup"]))
        _run_env_trace(eng, net, env, Traj(z, e), 3)


def test_golden_ssd_replay(eng):
    z = load("b100_ssd_replay.npz")
    net = eng.engine.Network(eng.compiler.load_bittner(str(z["pickle"])))
    sim = eng.engine.Simulator(net, 2)
    sim.set_state(z["init"])
    rp = eng.engine.Replay(z["ints"], z["dbls"], "cuda")
    hist = sim.ssd(int(z["iters"]), float(z["p"]), z["tgt_nodes"], replay=rp)
    assert np.array_equal(hist.cpu().numpy(), z["hist"].sum(0))
    used = rp.used.cpu().numpy()
    assert np.array_equal(used[:, 0], [z["ints"].shape[1]] * 2) and np.array_equal(used[:, 1], [z["dbls"].shape[1]] * 2)


# ------------------------------------------------------------------------------------------------ Philox mode vs oracle
def _nets(eng, which):
    if which == "tt":
        pbn_data = random_tt_data(70, seed=5)
        return eng.engine.Network(eng.compiler.compile_pbn_data(pbn_data)), orc.net_from_pbn_data(pbn_data)
    sets, ids = orc.load_bittner(which)
    return eng.engine.Network(eng.compiler.load_bittner(which)), orc.net_from_predictor_sets(sets, ids)


@pytest.mark.parametrize("fmax", [1, 2, 5, 6, 9, 13, 17, 18, 23])
def test_threshold_row_layouts(eng, fmax):
    """Predictor selection for every threshold-row layout: one quad (<= 5 predictors), leading quad + 2..4 quads (6..17),
    flat rows (more): rollout (async, sync) and SSD against the oracle."""
    net, onet = random_predictor_net(eng, 40, fmax, seed=fmax)
    B, seed = 512, 77
    sim = eng.engine.Simulator(net, B, seed=seed, env0=64)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0), env0=64)
    sim.rollout(301)
    orc.rollout(onet, ost, 301, orc.Draws(seed=seed, epoch=1), env0=64)
    assert np.array_equal(_state_np(sim), ost)
    sim.rollout(5, sync=True)
    orc.rollout(onet, ost, 5, orc.Draws(seed=seed, epoch=2), env0=64, sync=True)
    assert np.array_equal(_state_np(sim), ost)
    tgt = np.arange(3, 9, dtype=np.int32)
    hist = sim.ssd(50, 0.02, tgt)
    ohist = orc.ssd(onet, None, ost, 50, 0.02, tgt, orc.Draws(seed=seed, epoch=3), env0=64)
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist) and np.array_equal(_state_np(sim), ost)


@pytest.mark.parametrize("n,fmax", [(200, 12), (250, 5), (33, 3), (129, 7)])
def test_fast_record_paths(eng, n, fmax):
    """The fast asynchronous paths read 16-byte predictor records from aligned state columns (1..8 words per column);
    networks whose records exceed 32 KB (200 nodes x 12 predictors) take the generic path.  Both against the oracle."""
    net, onet = random_predictor_net(eng, n, fmax, seed=n + fmax)
    B, seed = 300, 5
    sim = eng.engine.Simulator(net, B, seed=seed, env0=64)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0), env0=64)
    sim.rollout(400)
    orc.rollout(onet, ost, 400, orc.Draws(seed=seed, epoch=1), env0=64)
    assert np.array_equal(_state_np(sim), ost)
    tgt = np.arange(n - 8, n - 2, dtype=np.int32) if (n - 8) // 32 == (n - 3) // 32 else np.arange(0, 6, dtype=np.int32)
    hist = sim.ssd(41, 0.01, tgt)
    ohist = orc.ssd(onet, None, ost, 41, 0.01, tgt, orc.Draws(seed=seed, epoch=2), env0=64)
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist) and np.array_equal(_state_np(sim), ost)


@pytest.mark.parametrize("which", ["28_15_median", "100_5_kmeans", "200_5_kmeans", "70_5_kmeans", "tt"])
@pytest.mark.parametrize("sync", [False, True])
def test_philox_rollout_matches_oracle(eng, which, sync):
    net, onet = _nets(eng, which)
    B, steps, seed, env0 = 1000, (7 if sync else 300), 1234, 5_000_000_000
    sim = eng.engine.Simulator(net, B, seed=seed, env0=env0)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0, B=B), env0=env0)
    assert np.array_equal(_state_np(sim), ost)
    sim.rollout(steps, sync=sync)
    od = orc.Draws(seed=seed, epoch=1, B=B)
    orc.rollout(onet, ost, steps, od, sync=sync, env0=env0)
    assert np.array_equal(_state_np(sim), ost)


def test_philox_split_invariance(eng):
    """env e's stream is keyed by its global id: two half-ranges == one full range (the multi-GPU contract)."""
    net, _ = _nets(eng, "100_5_kmeans")
    full = eng.engine.Simulator(net, 512, seed=9, env0=100)
    full.rand_state(); full.rollout(200)
    halves = []
    for k in range(2):
        h = eng.engine.Simulator(net, 256, seed=9, env0=100 + 256 * k)
        h.rand_state(); h.rollout(200)
        halves.append(_state_np(h))
    assert np.array_equal(_state_np(full), np.concatenate(halves))


def _fixture_atts(n, rng, n_att=4, care=5):
    atts = []
    for a in range(n_att):
        cubes = []
        for _ in range(1 + a % 2):
            c = ["*"] * n
            for i in rng.choice(n, size=care, replace=False):
                c[i] = int(rng.integers(0, 2))
            cubes.append(tuple(c))
        atts.append(cubes)
    return atts


@pytest.mark.parametrize("kind", ["target", "target_force", "multi", "multi_list"])
def test_philox_env_step_matches_oracle(eng, kind):
    net, onet = _nets(eng, "100_5_kmeans")
    rng = np.random.default_rng(3)
    n, B, seed = net.n, 2048, 77
    atts = _fixture_atts(n, rng)
    ek = eng.abi.ENV_TARGET if kind.startswith("target") else eng.abi.ENV_MULTI
    kw = dict(attractors=atts, horizon=7, max_inner=200, force=(kind == "target_force"), dedup=(kind != "multi_list"))
    env = eng.engine.EnvImage(net, ek, **kw)
    oenv = orc.Env(orc.ENV_TARGET if kind.startswith("target") else orc.ENV_MULTI, n, attractors=atts, horizon=7,
                   max_inner=200, force=int(kind == "target_force"), dedup=int(kind != "multi_list"))
    sim = eng.engine.Simulator(net, B, seed=seed)
    ost = np.zeros((B, n), np.uint8)
    ons, ota = np.zeros(B, np.int32), np.zeros(B, np.int32)
    otgt = np.zeros((B, n), np.uint8)
    sim.env_reset(env)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0), target_state=otgt)
    assert np.array_equal(_state_np(sim), ost) and np.array_equal(sim.target_att.cpu().numpy(), ota)
    assert np.array_equal(sim.unpack(sim.target_state).cpu().numpy(), otgt)
    K = 1 if kind.startswith("target") else 3
    for t in range(12):
        act = rng.integers(0, n + 1, size=(B, K)).astype(np.int32)
        if K == 3:
            dup = rng.random(B) < 0.3
            act[dup, 2] = act[dup, 0]
        sim.env_step(env, torch.from_numpy(act))
        obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + 2 * t))
        assert np.array_equal(_state_np(sim), ost), t
        assert np.array_equal(sim.unpack(sim.obs_state).cpu().numpy(), obs), t
        assert np.array_equal(sim.reward.cpu().numpy(), rew) and np.array_equal(sim.terminated.cpu().numpy(), term)
        assert np.array_equal(sim.truncated.cpu().numpy(), trunc) and np.array_equal(sim.inner.cpu().numpy(), inner)
        done = (term | trunc).astype(np.uint8)
        sim.env_reset(env, mask=torch.from_numpy(done))
        orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=2 + 2 * t), mask=done)
        assert np.array_equal(_state_np(sim), ost) and np.array_equal(sim.n_steps.cpu().numpy(), ons)


@pytest.mark.parametrize("kind", ["pbn", "pbcn", "pbn_sd", "pbcn_sd", "pbcn_sd_write"])
def test_philox_tt_env_step_matches_oracle(eng, kind):
    net, onet = _nets(eng, "tt")
    rng = np.random.default_rng(4)
    n, B, seed = net.n, 1500, 5
    atts = [[tuple(int(v) for v in rng.integers(0, 2, n)) for _ in range(1 + a)] for a in range(3)]
    targets = [atts[2][0], tuple(int(v) for v in rng.integers(0, 2, n))]
    kmap = {"pbn": (eng.abi.ENV_PBN, orc.ENV_PBN), "pbcn": (eng.abi.ENV_PBCN, orc.ENV_PBCN),
            "pbn_sd": (eng.abi.ENV_PBN_SD, orc.ENV_PBN_SD), "pbcn_sd": (eng.abi.ENV_PBCN_SD, orc.ENV_PBCN_SD),
            "pbcn_sd_write": (eng.abi.ENV_PBCN_SD, orc.ENV_PBCN_SD)}
    M = 3
    cw = kind == "pbcn_sd_write"
    env = eng.engine.EnvImage(net, kmap[kind][0], attractors=atts, targets=targets, n_control=M, control_write=cw,
                              successful_reward=10, wrong_attractor_cost=2)
    oenv = orc.Env(kmap[kind][1], n, attractors=atts, targets=targets, n_control=M, control_write=int(cw),
                   successful_reward=10, wrong_attractor_cost=2)
    sim = eng.engine.Simulator(net, B, seed=seed)
    ost = np.zeros((B, n), np.uint8)
    ons, ota = np.zeros(B, np.int32), np.zeros(B, np.int32)
    sim.env_reset(env)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    assert np.array_equal(_state_np(sim), ost)
    # random states make rewards non-trivial: plant targets/attractor states into a third of the envs
    plant = rng.random(B) < 0.3
    ost[plant] = np.array(targets[0], np.uint8)
    sim.set_state(ost)
    for t in range(6):
        if kind in ("pbn", "pbcn"):
            act = rng.integers(0, n, size=(B, 1))
        elif kind == "pbn_sd":
            act = np.stack([rng.integers(0, n + 1, B), rng.integers(1, 20, B)], 1)
        else:
            act = np.concatenate([rng.integers(1, 20, (B, 1)), rng.integers(0, 2, (B, M))], 1)
        act = act.astype(np.int32)
        sim.env_step(env, torch.from_numpy(act))
        obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + t))
        assert np.array_equal(_state_np(sim), ost), t
        assert np.array_equal(sim.reward.cpu().numpy(), rew) and np.array_equal(sim.terminated.cpu().numpy(), term)
        assert np.array_equal(sim.inner.cpu().numpy(), inner)


@pytest.mark.parametrize("which,p", [("100_5_kmeans", 0.01), ("28_15_median", 0.05), ("200_5_kmeans", 0.0), ("tt", 1.0),
                                     # the static loop at its extremes: several rounds of the perturbation process per
                                     # iteration, and rounds thousands of iterations apart (applied event slots stay stale)
                                     ("100_5_kmeans", 0.3), ("100_5_kmeans", 1e-5), ("100_5_kmeans", 1e-6)])
def test_philox_ssd_matches_oracle(eng, which, p):
    net, onet = _nets(eng, which)
    B, iters, seed = 3000, 400, 99
    tgt = np.array([0, 1, 2, 3, 4, 5, 6], np.int32) if which != "tt" else np.array([3, 41, 69, 7], np.int32)
    sim = eng.engine.Simulator(net, B, seed=seed, env0=64)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0), env0=64)
    hist = sim.ssd(iters, p, tgt)
    ohist = orc.ssd(onet, None, ost, iters, p, tgt, orc.Draws(seed=seed, epoch=1), env0=64)
    assert hist.sum().item() == B * iters
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist)
    assert np.array_equal(_state_np(sim), ost)


@pytest.mark.parametrize("which,B,iters,tgt", [
    ("100_5_kmeans", 64, 1, [0, 1, 2, 3, 4, 5, 6]),       # odd tail only (no static pair)
    ("100_5_kmeans", 96, 7, [0, 1, 2, 3, 4, 5, 6]),       # three static pairs + one tail iteration
    ("100_5_kmeans", 64 + 5, 8, [0, 1, 2, 3, 4, 5, 6]),   # last warp not full: generic path next to the static one
    ("100_5_kmeans", 128, 10, [3, 41, 69, 7]),             # scattered targets: generic bucket, generic static path
    ("100_5_kmeans", 128, 10, list(range(30, 37))),        # consecutive targets straddling a word boundary
    ("100_5_kmeans", 128, 10, list(range(40, 53))),        # 13 targets: global-memory histogram
    ("28_15_median", 160, 9, [20, 21, 22, 23]),            # four threshold quads per node
    ("200_5_kmeans", 96, 6, [64, 65, 66]),                 # targets in the third state word
    ("tt", 96, 9, [1, 2, 3]),                              # truth-table network: generic static path
])
def test_philox_ssd_loop_variants(eng, which, B, iters, tgt):
    """Every branch of the SSD loop (static update stream for full warps, specialised predictor path, generic tail)
    gives the oracle's histogram and final states; the update stream is two words per update, the perturbation gaps
    come from the env's second Philox stream."""
    net, onet = _nets(eng, which)
    seed, tgt = 5, np.array(tgt, np.int32)
    sim = eng.engine.Simulator(net, B, seed=seed, env0=32)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0), env0=32)
    hist = sim.ssd(iters, 0.02, tgt)
    ohist = orc.ssd(onet, None, ost, iters, 0.02, tgt, orc.Draws(seed=seed, epoch=1), env0=32)
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist)
    assert np.array_equal(_state_np(sim), ost)
    # a rollout continues from the same states: odd and even step counts of the static update stream
    for steps in (1, 4, 5):
        sim.rollout(steps)
        orc.rollout(onet, ost, steps, orc.Draws(seed=seed, epoch=sim.epoch - 1), env0=32)
        assert np.array_equal(_state_np(sim), ost), steps


def test_philox_ssd_with_attractor_loop(eng):
    net, onet = _nets(eng, "28_15_median")
    rng = np.random.default_rng(8)
    atts = _fixture_atts(net.n, rng, care=3)
    env = eng.engine.EnvImage(net, eng.abi.ENV_TARGET, attractors=atts, max_inner=50)
    oenv = orc.Env(orc.ENV_TARGET, net.n, attractors=atts, max_inner=50)
    B, iters, seed = 1024, 100, 3
    tgt = np.arange(9, dtype=np.int32)
    sim = eng.engine.Simulator(net, B, seed=seed)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0))
    hist = sim.ssd(iters, 0.01, tgt, env=env)
    ohist = orc.ssd(onet, oenv, ost, iters, 0.01, tgt, orc.Draws(seed=seed, epoch=1))
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist)
    assert np.array_equal(_state_np(sim), ost)


def test_flip_probability_below_the_gap_cap_is_refused(eng):
    """Gaps are capped at 2^25 (the 64 summed gaps of a round must fit 32 bits); the cap would bite below p = 1e-6."""
    net, _ = _nets(eng, "100_5_kmeans")
    sim = eng.engine.Simulator(net, 64, seed=1)
    sim.rand_state()
    with pytest.raises(eng.abi.PbnError):
        sim.ssd(4, 5e-7, np.arange(7, dtype=np.int32))


def test_large_g_uses_global_histogram(eng):
    net, onet = _nets(eng, "100_5_kmeans")
    B, iters, seed = 512, 64, 21
    tgt = np.arange(14, dtype=np.int32)
    sim = eng.engine.Simulator(net, B, seed=seed)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0))
    hist = sim.ssd(iters, 0.01, tgt)
    ohist = orc.ssd(onet, None, ost, iters, 0.01, tgt, orc.Draws(seed=seed, epoch=1))
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist)


def test_replay_lockstep_256_envs(eng):
    """256 envs x 1000 async updates under synthetic replayed draws: CUDA (float64 compares) == oracle."""
    net, onet = _nets(eng, "28_15_median")
    rng = np.random.default_rng(2)
    B, steps, n = 256, 1000, net.n
    ints = rng.integers(0, n, size=(B, steps)).astype(np.int32)
    dbls = rng.random((B, steps))
    st0 = rng.integers(0, 2, size=(B, n)).astype(np.uint8)
    sim = eng.engine.Simulator(net, B)
    sim.set_state(st0)
    sim.rollout(steps, replay=eng.engine.Replay(ints, dbls, "cuda"))
    ost = st0.copy()
    orc.rollout(onet, ost, steps, orc.Draws(ints=ints, dbls=dbls))
    assert np.array_equal(_state_np(sim), ost)


def test_pack_unpack_roundtrip(eng):
    net, _ = _nets(eng, "200_5_kmeans")
    rng = np.random.default_rng(0)
    bits = rng.integers(0, 2, size=(777, net.n)).astype(np.uint8)
    sim = eng.engine.Simulator(net, 777)
    sim.set_state(bits)
    assert np.array_equal(_state_np(sim), bits)


# ------------------------------------------------------------------------------------------------ statistics (Philox mode)
def _tv(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return 0.5 * np.abs(a / a.sum() - b / b.sum()).sum()


@pytest.mark.parametrize("p,T", [(0.01, 50), (0.3, 5)])
def test_philox_flip_rate_gpu(eng, p, T):
    """Identity dynamics: only the perturbation changes bits, so P(bit = 1 after T) = (1 - (1-2p)^T) / 2."""
    n, B = 100, 50000
    data = []
    for i in range(n):
        mask = np.zeros(n, bool)
        mask[i] = True
        data.append((mask, np.array([0.0, 1.0]), f"n{i}", False))
    net = eng.engine.Network(eng.compiler.compile_pbn_data(data))
    sim = eng.engine.Simulator(net, B, seed=3)
    hist = sim.ssd(T, p, np.arange(3, dtype=np.int32))
    assert int(hist.sum()) == B * T
    st = _state_np(sim)
    expect = (1 - (1 - 2 * p) ** T) / 2
    sigma = np.sqrt(expect * (1 - expect) / (B * n))
    assert abs(st.mean() - expect) <= 5 * sigma
    assert np.abs(st.mean(0) - expect).max() <= 6 * np.sqrt(expect * (1 - expect) / B)


def test_ssd_total_variation_vs_reference_gpu(eng):
    """Independent RNG: TV(GPU estimate, reference estimate) <= 3 x TV between two reference runs, at the reference's
    default budget (1.2 M iterations over 300 chains).  A 100x larger GPU estimate must sit within the same bound."""
    z = load("b100_ssd_long.npz")
    ref_a, ref_b = z["ssd"]
    floor = _tv(ref_a, ref_b)
    net = eng.engine.Network(eng.compiler.load_bittner(str(z["pickle"])))
    tgt = np.arange(7, dtype=np.int32)
    chains, iters = int(z["resets"]), int(z["iters"]) // int(z["resets"])
    sim = eng.engine.Simulator(net, chains, seed=5)
    sim.rand_state()
    hist = sim.ssd(iters, float(z["p"]), tgt).cpu().numpy()
    assert _tv(hist, ref_a) <= 3 * floor and _tv(hist, ref_b) <= 3 * floor
    big = eng.engine.Simulator(net, 30000, seed=6)
    big.rand_state()
    hb = big.ssd(iters, float(z["p"]), tgt).cpu().numpy()
    pooled = ref_a + ref_b
    assert _tv(hb, pooled) <= 3 * floor
    print("TV floor", floor, "gpu-vs-refA", _tv(hist, ref_a), "gpu(big)-vs-pooled", _tv(hb, pooled))


def _batch_se(batches):
    """Per-bucket standard error of the pooled estimate from independent batch estimates."""
    p = batches / batches.sum(1, keepdims=True)
    return p.std(0, ddof=1) / np.sqrt(len(batches))


def test_ssd_tight_tolerance_vs_literal_reference_algorithm(eng):
    """The product's SSD (geometric-skip flips, 31-bit integer thresholds, Philox) against 1.024e9 iterations of the
    reference's LITERAL algorithm — N Bernoulli(p) draws per iteration with float64 compares, `u*CODsum < cum` predictor
    picks — run through the oracle's replay path on NumPy draws (oracle/make_ssd_literal_golden.py; that path is pinned to
    traces of the unmodified reference).  Same chain length (4 000, the reference's default), 1.05e9 GPU iterations.
    Tolerance: total variation <= 0.005 over the 128 buckets (measured: 0.0009; round 1 accepted 0.094), and no bucket further
    than 5 standard errors (batch means on both sides) from the literal estimate."""
    z = load("b100_ssd_literal.npz")
    lit = z["hist"].astype(np.float64)
    iters = int(z["iters"])
    net = eng.engine.Network(eng.compiler.load_bittner(str(z["pickle"])))
    tgt = z["tgt_nodes"].astype(np.int32)
    runs = []
    for k in range(8):
        sim = eng.engine.Simulator(net, 1 << 15, seed=100 + k)
        sim.rand_state()
        runs.append(sim.ssd(iters, float(z["p"]), tgt).cpu().numpy().astype(np.float64))
    gpu = np.array(runs)
    assert gpu.sum() == 8 * (1 << 15) * iters
    tv = _tv(gpu.sum(0), lit.sum(0))
    p_lit, p_gpu = lit.sum(0) / lit.sum(), gpu.sum(0) / gpu.sum()
    se = np.sqrt(_batch_se(lit) ** 2 + _batch_se(gpu) ** 2)
    zmax = float(np.max(np.abs(p_gpu - p_lit)[p_lit > 1e-3] / se[p_lit > 1e-3]))
    print("TV(gpu 1.05e9, literal 1.02e9) =", tv, "max |z| =", zmax)
    assert tv <= 0.005
    assert zmax <= 5.0


def test_ssd_split_invariance(eng):
    """Shards cut at multiples of 32 chains reproduce the one-launch estimate exactly (the multi-GPU contract: groups of
    32 consecutive global chain ids share one perturbation stream)."""
    net, _ = _nets(eng, "100_5_kmeans")
    tgt = np.arange(7, dtype=np.int32)
    full = eng.engine.Simulator(net, 1000, seed=4, env0=96)
    full.rand_state()
    hf = full.ssd(300, 0.02, tgt).cpu().numpy()
    parts, states = np.zeros_like(hf), []
    for start, stop in ((0, 352), (352, 704), (704, 1000)):
        s = eng.engine.Simulator(net, stop - start, seed=4, env0=96 + start)
        s.rand_state()
        parts += s.ssd(300, 0.02, tgt).cpu().numpy()
        states.append(_state_np(s))
    assert np.array_equal(parts, hf)
    assert np.array_equal(np.concatenate(states), _state_np(full))
    bad = eng.engine.Simulator(net, 64, seed=4, env0=5)
    with pytest.raises(ValueError):
        bad.ssd(10, 0.02, tgt)


def test_golden_ssd_policy_branch(eng):
    """The `model` branch of _ssd_run replayed through the C-ABI: pbn_bucket_hist + pbn_env_step per iteration."""
    z = load("b28_ssd_policy.npz")
    net = eng.engine.Network(eng.compiler.load_bittner(str(z["pickle"])))
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = eng.engine.EnvImage(net, eng.abi.ENV_TARGET, attractors=atts, horizon=10**9, max_inner=int(z["cap"]))
    sim = eng.engine.Simulator(net, 1)
    sim.set_state(z["init"].reshape(1, -1))
    sim.target_att[0] = int(z["target_att"])
    tgt = z["tgt_nodes"]
    hist = torch.zeros(1 << len(tgt), dtype=torch.int64, device="cuda")
    for t, a in enumerate(z["actions"]):
        eng.engine.bucket_hist(sim, tgt, hist)
        rp = _replay(eng, z["ints"][z["int_off"][t]:z["int_off"][t + 1]], z["dbls"][z["dbl_off"][t]:z["dbl_off"][t + 1]])
        sim.env_step(env, torch.tensor([[int(a)]], dtype=torch.int32), replay=rp)
    assert np.array_equal(hist.cpu().numpy(), z["hist"])
    assert np.array_equal(_state_np(sim)[0], z["final"])


def test_bucket_hist_large_batch(eng):
    net, _ = _nets(eng, "100_5_kmeans")
    sim = eng.engine.Simulator(net, 100_000, seed=2)
    sim.rand_state()
    for tgt in (np.array([0, 1, 2, 3, 4, 5, 6], np.int32), np.array([99, 3, 64, 31, 32], np.int32), np.arange(14, dtype=np.int32)):
        hist = torch.zeros(1 << len(tgt), dtype=torch.int64, device="cuda")
        eng.engine.bucket_hist(sim, tgt, hist)
        bits = _state_np(sim)[:, tgt].astype(np.int64)
        idx = (bits * (1 << np.arange(len(tgt) - 1, -1, -1))).sum(1)
        assert np.array_equal(hist.cpu().numpy(), np.bincount(idx, minlength=1 << len(tgt)))


# ------------------------------------------------------------------------------------------------ edge cases
@pytest.mark.parametrize("n", [2, 31, 32, 33, 64, 65])
@pytest.mark.parametrize("B", [1, 31, 33, 257])
def test_word_boundaries_and_ragged_batches(eng, n, B):
    """State widths around the 32-bit word boundary, batches around the warp / block boundary; nodes without inputs."""
    rng = np.random.default_rng(n * 1000 + B)
    data = []
    for i in range(n):
        k = int(rng.integers(0, min(4, n) + 1)) if i % 5 else 0
        mask = np.zeros(n, bool)
        mask[rng.choice(n, size=k, replace=False)] = True
        table = rng.choice([0.0, 1.0, 0.25, 0.5], size=2**k).reshape([2] * k) if k else np.array(float(rng.integers(0, 2)))
        data.append((mask, table, f"g{i}", k == 0))
    net = eng.engine.Network(eng.compiler.compile_pbn_data(data))
    onet = orc.net_from_pbn_data(data)
    sim = eng.engine.Simulator(net, B, seed=n, env0=32 * B)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=n, epoch=0), env0=32 * B)
    assert np.array_equal(_state_np(sim), ost)
    sim.rollout(37)
    orc.rollout(onet, ost, 37, orc.Draws(seed=n, epoch=1), env0=32 * B)
    assert np.array_equal(_state_np(sim), ost)
    sim.rollout(2, sync=True)
    orc.rollout(onet, ost, 2, orc.Draws(seed=n, epoch=2), env0=32 * B, sync=True)
    assert np.array_equal(_state_np(sim), ost)
    tgt = np.array([n - 1, 0], np.int32)
    hist = sim.ssd(9, 0.2, tgt)
    ohist = orc.ssd(onet, None, ost, 9, 0.2, tgt, orc.Draws(seed=n, epoch=3), env0=32 * B)
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist) and np.array_equal(_state_np(sim), ost)


def test_empty_inputs_are_no_ops(eng):
    net, _ = _nets(eng, "28_15_median")
    sim = eng.engine.Simulator(net, 8, seed=1)
    sim.rand_state()
    before = _state_np(sim)
    sim.rollout(0)                       # zero steps
    hist = sim.ssd(0, 0.01, np.array([0, 1], np.int32))  # zero iterations
    assert int(hist.sum()) == 0 and np.array_equal(_state_np(sim), before)
    import ctypes as C
    lib = eng.abi.lib()
    d = eng.abi.PbnDraws(mode=eng.abi.DRAW_PHILOX, seed=1, epoch=0)
    assert lib.pbn_rollout(net.handle, C.c_void_p(sim.state.data_ptr()), 0, 0, 5, 0, C.byref(d), None) == 0  # B = 0
    assert lib.pbn_rand_state(net.handle, C.c_void_p(sim.state.data_ptr()), 0, 0, C.byref(d), None) == 0
    assert lib.pbn_rollout(None, None, 1, 0, 1, 0, C.byref(d), None) == 1  # PBN_ERR_ARG, nothing thrown across the ABI
    assert b"bad argument" in lib.pbn_last_error()


def test_full_size_properties(eng):
    """configs[2] at its full per-GPU width (2^20 chains): every iteration is histogrammed, the estimate is a pure function
    of (seed, epoch), shards cut at multiples of 32 chains add up to the whole, and the law agrees with a smaller oracle run."""
    net, onet = _nets(eng, "100_5_kmeans")
    tgt = np.arange(7, dtype=np.int32)
    B, iters = 1 << 20, 96

    def run(lo, hi):
        s = eng.engine.Simulator(net, hi - lo, seed=42, env0=lo)
        s.rand_state()
        return s.ssd(iters, 0.01, tgt).cpu().numpy()

    full = run(0, B)
    assert int(full.sum()) == B * iters
    assert np.array_equal(run(0, B), full)                                   # deterministic
    cut = 32 * 12345
    assert np.array_equal(run(0, cut) + run(cut, B), full)                   # shard additivity (the multi-GPU contract)
    ob = 1 << 14
    ost = orc.rand_state(onet, ob, orc.Draws(seed=42, epoch=0))
    ohist = orc.ssd(onet, None, ost, iters, 0.01, tgt, orc.Draws(seed=42, epoch=1))
    assert np.array_equal(run(0, ob).astype(np.uint64), ohist)               # the first 2^14 chains, bit for bit
    assert _tv(full, ohist) < 0.06  # and the same law at 64x the width (noise floor of 2^14 short chains over 128 buckets ~0.04)


@pytest.mark.parametrize("which,B", [("100_5_kmeans", 4096), ("200_5_kmeans", 1000), ("70_5_kmeans", 33), ("150_5_kmeans", 2049)])
def test_sync_sliced_matches_oracle(eng, which, B):
    """Bit-sliced synchronous kernel (32 envs per word, bit-serial threshold compare, mux-tree LUTs) == its restatement."""
    net, onet = _nets(eng, which)
    seed, env0 = 5, 96
    sim = eng.engine.Simulator(net, B, seed=seed, env0=env0)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0), env0=env0)
    sim.rollout(9, sync="sliced")
    orc.rollout_sync_sliced(onet, ost, 9, orc.Draws(seed=seed, epoch=1), env0=env0)
    assert np.array_equal(_state_np(sim), ost)
    sim.rollout(1, sync="sliced")
    orc.rollout_sync_sliced(onet, ost, 1, orc.Draws(seed=seed, epoch=2), env0=env0)
    assert np.array_equal(_state_np(sim), ost)


def test_sync_sliced_split_invariance_and_errors(eng):
    net, _ = _nets(eng, "100_5_kmeans")
    full = eng.engine.Simulator(net, 640, seed=8, env0=0)
    full.rand_state(); full.rollout(5, sync="sliced")
    parts = []
    for lo, hi in ((0, 320), (320, 640)):
        s = eng.engine.Simulator(net, hi - lo, seed=8, env0=lo)
        s.rand_state(); s.rollout(5, sync="sliced")
        parts.append(_state_np(s))
    assert np.array_equal(np.concatenate(parts), _state_np(full))
    with pytest.raises(ValueError):
        eng.engine.Simulator(net, 64, seed=8, env0=7).rollout(1, sync="sliced")
    net28, _ = _nets(eng, "28_15_median")  # 15 predictors per node: not supported by the sliced kernel
    with pytest.raises(eng.abi.PbnError):
        eng.engine.Simulator(net28, 64, seed=8).rollout(1, sync="sliced")


@pytest.mark.parametrize("p", [0.01, 0.02, 0.001, 0.3, 1e-5])
def test_gap_shortcut_is_exact(eng, p):
    """The lg2.approx shortcut of the SSD gap draw against the defining polynomial on ALL 2^23 inputs: no disagreement where
    it is taken; on for the usual flip probabilities (few inputs fall back), off when the margin would be too wide."""
    import ctypes as C

    delta, bad, fb = C.c_float(), C.c_uint32(), C.c_uint32()
    eng.abi.check(eng.abi.lib().pbn_geom_shortcut_check(p, C.byref(delta), C.byref(bad), C.byref(fb)))
    assert bad.value == 0
    if p >= 0.001:
        assert delta.value < 0.05 and fb.value < 0.1 * 2**23
    if p == 1e-5:
        assert delta.value == 1.0


def test_ssd_histogram_host_matches_oracle(eng):
    """ssd_histogram_host (the end-to-end call bench.py times; host states in, host histogram out) on several waves of
    blocks: the histogram equals the oracle's, from pinned and from pageable start states."""
    from gym_PBN.utils.eval import ssd_histogram_host

    net, onet = _nets(eng, "100_5_kmeans")
    wave = torch.cuda.get_device_properties(0).multi_processor_count * 4 * 256
    chains, iters, seed, env0 = 2 * wave + 4096, 3, 17, 64
    rng = np.random.default_rng(0)
    st = rng.integers(0, 2, size=(chains, 100)).astype(np.uint8)
    tgt = np.arange(7, dtype=np.int32)
    h_pinned = ssd_histogram_host(net, torch.from_numpy(st).pin_memory(), iters, 0.01, tgt, seed=seed, env0=env0)
    h_plain = ssd_histogram_host(net, st, iters, 0.01, tgt, seed=seed, env0=env0)
    ost = st.copy()
    ohist = orc.ssd(onet, None, ost, iters, 0.01, tgt, orc.Draws(seed=seed, epoch=0), env0=env0)
    assert np.array_equal(h_pinned.astype(np.uint64), ohist) and np.array_equal(h_plain, h_pinned)
    assert int(h_pinned.sum()) == chains * iters
