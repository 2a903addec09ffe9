"""GPU: the BASELINE.json configurations as parity cases at (or near) their full sizes, CUDA vs oracle, Philox mode."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402
from golden_util import cubes_to_attractors, hittable_cubes, load, synthetic_pbcn  # noqa: E402


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


def test_config2_bittner28_65536_lockstep_envs(eng):
    z = load("b28_target_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    net = eng.engine.Network(eng.compiler.load_bittner("28_15_median"))
    sets, ids = orc.load_bittner("28_15_median")
    onet = orc.net_from_predictor_sets(sets, ids)
    B, seed = 65536, 2
    env = eng.engine.EnvImage(net, eng.abi.ENV_TARGET, attractors=atts, horizon=100, max_inner=256)
    oenv = orc.Env(orc.ENV_TARGET, 28, attractors=atts, horizon=100, max_inner=256)
    sim = eng.engine.Simulator(net, B, seed=seed)
    ost, ons, ota = np.zeros((B, 28), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
    sim.env_reset(env)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    rng = np.random.default_rng(2)
    for t in range(6):
        act = rng.integers(0, 29, size=(B, 1)).astype(np.int32)
        sim.env_step(env, torch.from_numpy(act))
        obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + t))
        assert np.array_equal(sim.unpack().cpu().numpy(), ost)
        assert np.array_equal(sim.reward.cpu().numpy(), rew) and np.array_equal(sim.inner.cpu().numpy(), inner)
        assert np.array_equal(sim.terminated.cpu().numpy(), term)


def test_config4_bittner200_multi_attractor_path(eng):
    net = eng.engine.Network(eng.compiler.load_bittner("200_5_kmeans"))
    sets, ids = orc.load_bittner("200_5_kmeans")
    onet = orc.net_from_predictor_sets(sets, ids)
    n, B, seed = net.n, 8192, 4
    assert n == 199
    rng = np.random.default_rng(4)
    atts = []
    for a in range(4):
        c = ["*"] * n
        for i in rng.choice(n, size=4, replace=False):
            c[i] = int(rng.integers(0, 2))
        atts.append([tuple(c)])
    env = eng.engine.EnvImage(net, eng.abi.ENV_MULTI, attractors=atts, horizon=100, max_inner=4096, dedup=True)
    oenv = orc.Env(orc.ENV_MULTI, n, attractors=atts, horizon=100, max_inner=4096, dedup=1)
    sim = eng.engine.Simulator(net, B, seed=seed)
    ost, ons, ota = np.zeros((B, n), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
    sim.env_reset(env)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    assert np.array_equal(sim.unpack().cpu().numpy(), ost)
    for t in range(4):
        act = rng.integers(0, n + 1, size=(B, 3)).astype(np.int32)
        act[rng.random(B) < 0.25, 1] = 0
        sim.env_step(env, torch.from_numpy(act))
        obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + t))
        assert np.array_equal(sim.unpack().cpu().numpy(), ost)
        assert np.array_equal(sim.unpack(sim.obs_state).cpu().numpy(), obs)
        assert np.array_equal(sim.reward.cpu().numpy(), rew) and np.array_equal(sim.inner.cpu().numpy(), inner)
    assert inner.max() > 1  # the step-until-attractor loop actually ran


@pytest.mark.parametrize("control_write", [False, True])
def test_config5_synthetic_pbcn_1024_variable_durations(eng, control_write):
    data = synthetic_pbcn()
    net = eng.engine.Network(eng.compiler.compile_pbn_data(data))
    onet = orc.net_from_pbn_data(data)
    n, M, B, seed = 1024, 8, 2048, 9
    assert net.w32 == 32
    rng = np.random.default_rng(1)
    targets = [tuple(int(v) for v in rng.integers(0, 2, n)) for _ in range(4)]
    atts = [[t] for t in targets]
    env = eng.engine.EnvImage(net, eng.abi.ENV_PBCN_SD, attractors=atts, targets=targets[:2], n_control=M,
                              control_write=control_write, successful_reward=10, wrong_attractor_cost=2)
    oenv = orc.Env(orc.ENV_PBCN_SD, n, attractors=atts, targets=targets[:2], n_control=M, control_write=int(control_write),
                   successful_reward=10, wrong_attractor_cost=2)
    st0 = rng.integers(0, 2, size=(B, n)).astype(np.uint8)
    st0[:, 0] = 0
    sim = eng.engine.Simulator(net, B, seed=seed)
    sim.set_state(st0)
    ost, ons, ota = st0.copy(), np.zeros(B, np.int32), np.zeros(B, np.int32)
    for t in range(3):
        act = np.concatenate([rng.integers(1, 65, (B, 1)), rng.integers(0, 2, (B, M))], 1).astype(np.int32)  # interval ~ U{1..64}
        sim.env_step(env, torch.from_numpy(act))
        obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=t))
        assert np.array_equal(sim.unpack().cpu().numpy(), ost)
        assert np.array_equal(sim.reward.cpu().numpy(), rew) and np.array_equal(sim.inner.cpu().numpy(), act[:, 0])
    if control_write:
        # node 0 is never updated (randint(1, N-1)), so it holds the control bit written before the last update;
        # control nodes 1..M-1 can be picked for update and then fall to 0 (their table is P = 0)
        assert np.array_equal(ost[:, 0], act[:, 1].astype(np.uint8))


def test_large_truth_table_rollout_and_sync(eng):
    data = synthetic_pbcn(n=1024, m=8, seed=3)
    net = eng.engine.Network(eng.compiler.compile_pbn_data(data))
    onet = orc.net_from_pbn_data(data)
    B, seed = 777, 5
    sim = eng.engine.Simulator(net, B, seed=seed)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0))
    sim.rollout(500)
    orc.rollout(onet, ost, 500, orc.Draws(seed=seed, epoch=1))
    assert np.array_equal(sim.unpack().cpu().numpy(), ost)
    sim.rollout(2, sync=True)
    orc.rollout(onet, ost, 2, orc.Draws(seed=seed, epoch=2), sync=True)
    assert np.array_equal(sim.unpack().cpu().numpy(), ost)


def _target_case(eng, name, kind, n_act, B, seed, max_inner, care=4, full_care=False):
    """A step-until-attractor env on a shipped predictor set with a cube fixture, product + oracle side by side."""
    net = eng.engine.Network(eng.compiler.load_bittner(name))
    sets, ids = orc.load_bittner(name)
    onet = orc.net_from_predictor_sets(sets, ids)
    n = net.n
    rng = np.random.default_rng(seed)
    atts = []
    for a in range(5):
        c = ["*"] * n
        for i in rng.choice(n, size=n if full_care and a == 0 else care, replace=False):
            c[i] = int(rng.integers(0, 2))
        atts.append([tuple(c)] if a else [tuple(c), tuple(1 - v if v != "*" else v for v in c)])
    multi = kind == "multi"
    env = eng.engine.EnvImage(net, eng.abi.ENV_MULTI if multi else eng.abi.ENV_TARGET, attractors=atts, horizon=100,
                              max_inner=max_inner, dedup=True)
    oenv = orc.Env(orc.ENV_MULTI if multi else orc.ENV_TARGET, n, attractors=atts, horizon=100, max_inner=max_inner, dedup=1)
    sim = eng.engine.Simulator(net, B, seed=seed)
    ost, ons, ota = np.zeros((B, n), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
    sim.env_reset(env)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    acts = [rng.integers(0, n + 1, size=(B, n_act)).astype(np.int32) for _ in range(3)]
    return net, onet, env, oenv, sim, (ost, ons, ota), acts


@pytest.mark.parametrize("name,kind,n_act,care", [("28_15_median", "target", 1, 5), ("100_5_kmeans", "target", 1, 6),
                                                  ("200_5_kmeans", "multi", 3, 5), ("28_15_median", "multi", 2, 6)])
@pytest.mark.parametrize("budgets", [(32, 0), (1, 7, 64, 0), (2, 2, 500, 3, 0), (5000,)])
def test_step_plan_split_invariance(eng, name, kind, n_act, care, budgets):
    """A step split over budgeted launches (first pass: a lane per env; resume passes: groups of lanes, global queue) equals
    the oracle's unsplit step bit for bit: states, observations, rewards, flags, update counts."""
    if kind == "multi" and budgets[0] == 1:
        budgets = (2,) + budgets[1:]
    B, seed = 3000, 11
    net, onet, env, oenv, sim, (ost, ons, ota), acts = _target_case(eng, name, kind, n_act, B, seed, max_inner=700, care=care)
    for t, act in enumerate(acts):
        sim.env_step(env, torch.from_numpy(act), budget=budgets[0])
        parked = [int(sim.running.sum())]
        for b in budgets[1:]:
            sim.env_step_resume(env, budget=b)
            parked.append(int(sim.running.sum()))
        assert parked[-1] == 0, parked
        obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + t))
        assert np.array_equal(sim.unpack().cpu().numpy(), ost)
        assert np.array_equal(sim.unpack(sim.obs_state).cpu().numpy(), obs)
        assert np.array_equal(sim.reward.cpu().numpy(), rew) and np.array_equal(sim.inner.cpu().numpy(), inner)
        assert np.array_equal(sim.terminated.cpu().numpy(), term) and np.array_equal(sim.truncated.cpu().numpy(), trunc)
        assert np.array_equal(sim.n_steps.cpu().numpy(), ons)
        if len(budgets) > 1:
            assert parked[0] > 0 and inner.max() > budgets[0]  # the split actually happened


@pytest.mark.parametrize("name,kind,n_act,n_cubes", [
    pytest.param("200_5_kmeans", "multi", 3, 2, id="200_5_kmeans-multi-3"),
    pytest.param("28_15_median", "target", 1, 2, id="28_15_median-target-1"),
    # three and four cubes: the lanes of a two-lane group test cube sub + 2 as well (the TWO branch at g = 2)
    pytest.param("28_15_median", "target", 1, 3, id="28_15_median-target-1-3cubes"),
    pytest.param("200_5_kmeans", "multi", 3, 4, id="200_5_kmeans-multi-3-4cubes"),
])
def test_step_plan_two_lane_groups(eng, name, kind, n_act, n_cubes):
    """A resume pass whose list exceeds 8 envs per warp over the whole grid runs 16 envs per warp in groups of TWO lanes (envs
    with at most four cubes): same words, same result as the oracle's unsplit step."""
    net = eng.engine.Network(eng.compiler.load_bittner(name))
    sets, ids = orc.load_bittner(name)
    onet = orc.net_from_predictor_sets(sets, ids)
    n, B, seed = net.n, 80000, 23
    rng = np.random.default_rng(seed)
    atts = []
    for a in range(2):  # two single-cube attractors; cubes that care about many nodes: an intervention often leaves them
        c = ["*"] * n
        for i in rng.choice(n, size=n // 2 if n < 64 else 40, replace=False):
            c[i] = int(rng.integers(0, 2))
        atts.append([tuple(c)])
    if n_cubes > 2:  # cubes 2 (and 3) are reachable ones (golden_util.hittable_cubes), in the second attractor
        atts[1] += hittable_cubes(onet, n_cubes - 2, seed, care=5)
    multi = kind == "multi"
    env = eng.engine.EnvImage(net, eng.abi.ENV_MULTI if multi else eng.abi.ENV_TARGET, attractors=atts, horizon=100, max_inner=400, dedup=True)
    oenv = orc.Env(orc.ENV_MULTI if multi else orc.ENV_TARGET, n, attractors=atts, horizon=100, max_inner=400, dedup=1)
    sim = eng.engine.Simulator(net, B, seed=seed)
    ost, ons, ota = np.zeros((B, n), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
    sim.env_reset(env)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    cubes = np.array([[2 if v == "*" else v for v in c] for a in atts for c in a], np.int8)
    for t in range(2):
        act = rng.integers(0, n + 1, size=(B, n_act)).astype(np.int32)
        sim.env_step(env, torch.from_numpy(act), budget=2)
        assert int(sim.running.sum()) > 148 * 2 * 8 * 8  # longer than 8 envs per warp on every SM: the wide pass
        sim.env_step_resume(env, budget=0)
        assert int(sim.running.sum()) == 0
        obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + t))
        assert np.array_equal(sim.unpack().cpu().numpy(), ost)
        assert np.array_equal(sim.unpack(sim.obs_state).cpu().numpy(), obs)
        assert np.array_equal(sim.reward.cpu().numpy(), rew) and np.array_equal(sim.inner.cpu().numpy(), inner)
        assert np.array_equal(sim.terminated.cpu().numpy(), term) and np.array_equal(sim.truncated.cpu().numpy(), trunc)
        assert inner.max() == 400  # cap hits included
        if n_cubes > 2:  # envs stopped by the loop on cube 2 or 3 alone: only the lanes' second cubes test those
            stopped = (inner > 2) & (inner < 400)
            match = [((obs[stopped] == c) | (c == 2)).all(1) for c in cubes]
            assert (~match[0] & ~match[1] & (match[2] | match[-1])).sum() > 100


def test_step_plan_matches_single_launch(eng):
    """The two-pass default of Simulator.env_step against the one-launch kernel (plan_budgets = ()), cap hits included."""
    B, seed = 20000, 5
    res = []
    for p1 in ((32, 256), (), (4,), (2, 2, 2, 100), "auto"):
        net, onet, env, oenv, sim, _, acts = _target_case(eng, "28_15_median", "target", 1, B, seed, max_inner=300, care=28,
                                                          full_care=True)
        sim.plan_budgets = p1
        out = []
        for act in acts:
            sim.env_step(env, torch.from_numpy(act))
            out.append((sim.unpack().cpu().numpy().copy(), sim.reward.cpu().numpy().copy(), sim.inner.cpu().numpy().copy(),
                        sim.terminated.cpu().numpy().copy()))
        res.append(out)
        assert out[-1][2].max() == 300  # envs that hit the cap exist
    for other in res[1:]:
        for a, b in zip(res[0], other):
            assert all(np.array_equal(x, y) for x, y in zip(a, b))


def test_step_plan_errors(eng):
    net, onet, env, oenv, sim, _, acts = _target_case(eng, "28_15_median", "multi", 2, 64, 3, max_inner=50)
    with pytest.raises(ValueError):
        sim.env_step(env, torch.from_numpy(acts[0]), budget=1)  # MULTI needs two updates before it can park
    with pytest.raises(eng.abi.PbnError):
        eng.engine.Simulator(net, 8).env_step_resume(env)
