"""GPU: the drop-in gymnasium surface (gym_PBN.make / env classes) and the batched PBNVectorEnv.

Single-env classes are checked for API shape, return types and — by driving the same kernels with the oracle in
Philox mode from the same seed/epoch — for exact values.  The VectorEnv is checked against the oracle step by step."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402
from golden_util import cubes_to_attractors, load  # noqa: E402

EX5 = (["u", "x1", "x2", "x3", "x4"],
       [[], [("not x2 and not x4", 1)], [("not x4 and not u and (x2 or x3)", 1)],
        [("not x2 and not x4 and x1", 0.7), ("False", 0.3)], [("not x2 and not x3", 1)]])
GOAL = {"target_nodes": {(0, 0, 0, 0, 1)}, "target": {(0, 0, 0, 0, 1)},
        "all_attractors": [{(0, 0, 1, 0, 0)}, {(0, 0, 0, 0, 1)}]}


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def test_make_pbn_v0_example_network():
    import gym_PBN

    env = gym_PBN.make("gym-PBN/PBN-v0", logic_func_data=EX5, goal_config=dict(GOAL))
    # attractors of the example network (SURVEY.md §4): computed exhaustively in the constructor
    assert sorted(map(sorted, env.all_attractors)) == [[(0, 0, 0, 0, 1)], [(0, 0, 1, 0, 0)]]
    obs, info = env.reset(seed=0)
    assert obs.dtype == bool and obs.shape == (5,) and tuple(obs) in env.attracting_states
    assert info["observation_idx"] == int("".join(str(int(b)) for b in obs), 2)
    seen_term = False
    for t in range(300):
        a = t % 5
        obs, r, term, trunc, info = env.step(a)
        assert isinstance(r, int) and isinstance(term, bool) and trunc is False and obs[0] == 0
        hit = tuple(int(b) for b in obs) in env.target_nodes
        assert term == hit and r == (20 if hit else -4 - (a != 0))
        if term:
            seen_term = True
            obs, info = env.reset()
    assert seen_term
    with pytest.raises(Exception):
        env.step(5)


def test_readme_style_pbcn_example_runs():
    """example.py:19-44 (`gym.make("gym-PBN/PBCN-v0", ...)` with README-style goal_config and action [1]) fails in the
    reference with KeyError('target_nodes'); here it runs."""
    import gym_PBN

    env = gym_PBN.make("gym-PBN/PBCN-v0", logic_func_data=EX5,
                       goal_config={"all_attractors": [{(0, 0, 0, 0, 1)}, {(0, 0, 1, 0, 0)}], "target": {(0, 0, 0, 0, 1)}})
    assert env.PBN.M == 1 and env.action_space.n == 1 and env.discrete_action_space.n == 2
    env.reset(seed=3)
    for _ in range(10):
        obs, r, term, trunc, info = env.step([1])
        assert r in (env.successful_reward, -env.wrong_attractor_cost, 0)
        if term:
            break


def test_sampled_data_env_variable_intervals():
    import gym_PBN

    env = gym_PBN.make("gym-PBN/PBCN-sampled-data-v0", logic_func_data=EX5, goal_config=dict(GOAL), T=8)
    env.reset(seed=1)
    obs, r, term, trunc, info = env.step(([True], 5))
    assert info["interval"] == 5 and isinstance(r, int)
    obs, r, term, trunc, info = env.step(2 * 3 + 1)  # flat index -> ([True], 4)
    assert info["interval"] == 4 and info["control_action"] == [True]
    with pytest.raises(Exception):
        env.step(([True], 9))
    env2 = gym_PBN.make("gym-PBN/PBN-sampled-data-v0", logic_func_data=EX5, goal_config=dict(GOAL), T=8)
    env2.reset(seed=1)
    obs, r, term, trunc, info = env2.step((2, 3))
    assert info["interval"] == 2


def test_self_triggering_envs_run():
    import gym_PBN

    env = gym_PBN.make("gym-PBN/PBN-self-triggering-v0", logic_func_data=EX5, goal_config=dict(GOAL), T=6)
    env.reset(seed=2)
    obs, r, term, trunc, info = env.step((1, 3))
    assert 1 <= info["interval"] <= 6
    env = gym_PBN.make("gym-PBN/PBCN-self-triggering-v0", logic_func_data=EX5, goal_config=dict(GOAL), T=6)
    env.reset(seed=2)
    obs, r, term, trunc, info = env.step(([False], 10))
    assert info["interval"] == 1  # prob 10/10 stops after the first primitive step


def test_graph_api_matches_oracle_stream():
    """Graph.step on the device == oracle in Philox mode with the graph's (seed, epoch) stream."""
    from gym_PBN.envs.bittner import utils

    g = utils.spawn(total_genes=28, seed=123)
    sets, ids = orc.load_bittner("28_15_median")
    onet = orc.net_from_predictor_sets(sets, ids)
    assert g.getIDs() == ids and g.N == 28
    st0 = [(i * 7) % 2 for i in range(28)]
    g.setState(st0)
    assert tuple(g.getState()) == tuple(st0) and g.getState()[ids[3]] == st0[3] and g.nodes[5].value == st0[5]
    g.flipNode(4)
    ost = np.array([st0], np.uint8)
    ost[0, 4] ^= 1
    s = g.step()
    orc.rollout(onet, ost, 1, orc.Draws(seed=123, epoch=g.sim.epoch - 1))
    assert tuple(s) == tuple(ost[0])
    g.step(steps=500)
    orc.rollout(onet, ost, 500, orc.Draws(seed=123, epoch=g.sim.epoch - 1))
    assert tuple(g.getState()) == tuple(ost[0])
    g.synch_step()
    orc.rollout(onet, ost, 1, orc.Draws(seed=123, epoch=g.sim.epoch - 1), sync=True)
    assert tuple(g.getState()) == tuple(ost[0])
    with pytest.raises(ValueError):
        g.flipNode(28)


def test_bittner28_env_with_fixture_attractors():
    import gym_PBN

    z = load("b28_target_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts, max_inner_steps=64, seed=5)
    core = env.unwrapped
    (state, target), info = env.reset(seed=5)
    assert len(state) == 28 and core.is_attracting_state(state) and core.target in atts
    sets, ids = orc.load_bittner("28_15_median")
    onet = orc.net_from_predictor_sets(sets, ids)
    oenv = orc.Env(orc.ENV_TARGET, 28, attractors=atts, horizon=100, max_inner=64)
    ost = np.array([state], np.uint8)
    ons, ota = np.zeros(1, np.int32), np.array([atts.index(core.target)], np.int32)
    for t in range(40):
        a = (t * 5) % 29
        epoch = core.sim.epoch
        obs, r, term, trunc, info = env.step(a)
        oobs, orew, oterm, otrunc, oin = orc.env_step(onet, oenv, ost, ons, ota, np.array([[a]], np.int32),
                                                      orc.Draws(seed=5, epoch=epoch))
        assert np.array_equal(obs, oobs[0]) and (r, term) == (int(orew[0]), bool(oterm[0]))
        assert info["inner_steps"] == int(oin[0]) and core.n_steps == int(ons[0])
        assert core.getTargetIdx() == int("".join(str(int(obs[ids.index(g)])) for g in core.target_nodes), 2)
        assert r == (20 if core.in_target(obs) else -5)
        if term or trunc:
            break


def test_make_bittner_100_and_200_default_attractors():
    import gym_PBN

    env = gym_PBN.make("gym-PBN/Bittner-100-v0", seed=1)
    core = env.unwrapped
    # no CABEAN here: the sampled + verified route (closed cube sets; Bittner-100: exact terminal SCCs inside 19- and 21-wildcard
    # trap spaces, found by the exhaustive device search on the restricted network)
    assert core.graph.N == 100 and len(core.all_attractors) >= 2 and core.horizon == 69 and core.attractor_source == "verified"
    from gym_PBN.b200 import attractors as att_tools

    model = att_tools.SuccessorModel(core.network.spec)
    assert all(att_tools.cubes_closed(model, a) for a in core.all_attractors)
    (state, target), info = env.reset(seed=1)
    for _ in range(5):
        obs, r, term, trunc, info = env.step(0)
        assert obs.shape == (100,) and r in (20, -5)
    env = gym_PBN.make("gym-PBN/Bittner-200-v0", seed=1)  # example.py:53; the shipped 200-gene set has 199 nodes
    assert env.unwrapped.graph.N == 199
    env.reset(seed=2)
    env.step(0)
    # sizes upstream ships no set for are fitted on the GPU (tests/test_gpu_fit.py); naming a set that does not exist raises
    with pytest.raises(FileNotFoundError):
        gym_PBN.make("gym-PBN/Bittner-100-v0", predictor_set="100_9_median")


def test_multi_env_list_and_tensor_actions():
    import gym_PBN

    z = load("b28_multi_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/BittnerMulti-28-v0", all_attractors=atts, max_inner_steps=64, seed=9)
    core = env.unwrapped
    (state, target), info = env.reset(seed=9)
    assert core.target is atts[-1] or core.target == atts[-1]
    sets, ids = orc.load_bittner("28_15_median")
    onet = orc.net_from_predictor_sets(sets, ids)
    oenv = orc.Env(orc.ENV_MULTI, 28, attractors=atts, horizon=100, max_inner=64, dedup=0)
    ost = np.array([state], np.uint8)
    ons, ota = np.zeros(1, np.int32), np.array([len(atts) - 1], np.int32)
    for t in range(30):
        acts = [(3 * t) % 29, (7 * t + 1) % 29, (3 * t) % 29 if t % 2 else 0]
        epoch = core.sim.epoch
        if t % 3 == 0:
            obs, r, term, trunc, info = env.step(torch.tensor(acts))
            eff = sorted(set(acts))
        else:
            obs, r, term, trunc, info = env.step(list(acts))
            eff = acts
        oobs, orew, oterm, otrunc, oin = orc.env_step(onet, oenv, ost, ons, ota, np.array([eff], np.int32),
                                                      orc.Draws(seed=9, epoch=epoch))
        assert tuple(obs) == tuple(oobs[0]) and (r, term, trunc) == (int(orew[0]), bool(oterm[0]), bool(otrunc[0]))
        if term or trunc:
            break


@pytest.mark.parametrize("plan", [None, (3, 8)])
def test_vector_env_matches_oracle(plan):
    import gym_PBN
    from gym_PBN.b200.vector_env import PBNVectorEnv

    z = load("b28_target_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts, max_inner_steps=32)
    B, seed = 4096, 17
    vec = PBNVectorEnv(env, B, seed=seed)
    if plan is not None:  # planned step: three passes + the masked reset launch (Simulator.vec_step)
        vec.sim.plan_budgets = plan
    obs, info = vec.reset()
    sets, ids = orc.load_bittner("28_15_median")
    onet = orc.net_from_predictor_sets(sets, ids)
    oenv = orc.Env(orc.ENV_TARGET, 28, attractors=atts, horizon=100, max_inner=32)
    ost = np.zeros((B, 28), np.uint8)
    ons, ota = np.zeros(B, np.int32), np.zeros(B, np.int32)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    assert np.array_equal(obs.cpu().numpy(), ost)
    rng = np.random.default_rng(0)
    episodes = 0
    for t in range(25):
        act = rng.integers(0, 29, size=(B, 1)).astype(np.int32)
        obs, rew, term, trunc, info = vec.step(torch.from_numpy(act))
        oobs, orew, oterm, otrunc, oin = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + 2 * t))
        assert np.array_equal(rew.cpu().numpy(), orew) and np.array_equal(term.cpu().numpy(), oterm.astype(bool))
        assert np.array_equal(vec.sim.unpack(info["final_obs_packed"]).cpu().numpy(), oobs)
        done = (oterm | otrunc).astype(np.uint8)
        episodes += int(done.sum())
        orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=2 + 2 * t), mask=done)
        assert np.array_equal(obs.cpu().numpy(), ost)  # auto-reset envs observe their new state
    red = vec.stats.reduced()
    assert red["episodes"] == episodes and red["env_steps"] == 25 * B and episodes > 0
    sd = vec.state_dict()
    vec2 = PBNVectorEnv(env, B, seed=0)
    vec2.load_state_dict(sd)
    act = rng.integers(0, 29, size=(B, 1)).astype(np.int32)
    o1 = vec.step(torch.from_numpy(act))[0].clone()
    o2 = vec2.step(torch.from_numpy(act))[0]
    assert torch.equal(o1, o2)


def test_vector_env_pbn_family_and_host_step():
    import gym_PBN
    from gym_PBN.b200.vector_env import PBNVectorEnv

    env = gym_PBN.make("gym-PBN/PBN-v0", logic_func_data=EX5, goal_config=dict(GOAL))
    vec = PBNVectorEnv(env, 1000, seed=4)
    obs, _ = vec.reset()
    assert obs.shape == (1000, 5) and int(obs[:, 0].sum()) == 0
    o, r, te, tr = vec.step_host(np.random.default_rng(1).integers(0, 5, size=(1000, 1)))
    assert o.shape == (1000, 5) and set(np.unique(r)) <= {20, -4, -5} and not tr.any()


def test_compute_ssd_hist_drop_in():
    import gym_PBN
    from gym_PBN.utils.eval import compute_ssd_hist, total_variation

    env = gym_PBN.make("gym-PBN/Bittner-100-v0", all_attractors=[[("*",) * 100], [("*",) * 100]], seed=3)
    df, fig = compute_ssd_hist(env.unwrapped, iters=1_200_000, resets=300, bit_flip_prob=0.01, seed=3)
    vals = np.asarray(df["Value"])
    assert vals.shape == (128,) and abs(vals.sum() - 1.0) < 1e-9 and list(df.index[:2]) == ["0000000", "0000001"]
    z = load("b100_ssd_long.npz")
    floor = total_variation(z["ssd"][0], z["ssd"][1])
    assert total_variation(vals, z["ssd"][0]) <= 3 * floor


def test_abi_error_paths():
    """Errors are status codes at the C boundary and the reference's exception types above it."""
    from gym_PBN.b200 import abi, compiler, engine

    net = engine.Network(compiler.load_bittner("28_15_median"))
    sim = engine.Simulator(net, 64, seed=1)
    with pytest.raises(ValueError):  # target node out of range
        sim.ssd(10, 0.01, np.array([0, 99], np.int32))
    with pytest.raises(ValueError):  # invalid bit flip probability (utils/eval.py:31-33)
        sim.ssd(10, 1.5, np.array([0, 1], np.int32))
    with pytest.raises(ValueError):  # TARGET reset needs two attractors (random.sample(..., 2))
        img = engine.EnvImage(net, abi.ENV_TARGET, attractors=[[("*",) * 28]])
        sim.env_reset(img)
    with pytest.raises(ValueError):  # cube of the wrong length
        engine.EnvImage(net, abi.ENV_TARGET, attractors=[[(0, 1)]])
    with pytest.raises(ValueError):  # sampled-data action width
        tt = engine.Network(compiler.compile_pbn_data([(np.array([False, True]), np.array([0.2, 0.9]), "a", False),
                                                       (np.array([True, False]), np.array([0.5, 0.5]), "b", False)]))
        s2 = engine.Simulator(tt, 4)
        s2.env_step(engine.EnvImage(tt, abi.ENV_PBN_SD, attractors=[[(0, 0)]], targets=[(0, 1)]), torch.zeros((4, 1), dtype=torch.int32))
    assert b"" == b"" and abi.lib().pbn_last_error() is not None
    with pytest.raises(ValueError):  # a negative COD would make a cumulative row descend
        spec = compiler.load_bittner("28_15_median")
        spec.arrays["pr_cum"] = spec.arrays["pr_cum"].copy()
        spec.arrays["pr_cum"][1] = spec.arrays["pr_cum"][0] - 0.5
        engine.Network(spec)
    with pytest.raises(abi.PbnError):  # predictor networks are limited to 256 nodes
        spec = compiler.load_bittner("28_15_median")
        spec.n = 300
        engine.Network(spec)


def test_compute_ssd_hist_with_model():
    """compute_ssd_hist(env, model=...) — the policy branch of the reference (utils/eval.py:97-101) on the GPU path."""
    import gym_PBN
    from gym_PBN.utils.eval import compute_ssd_hist

    z = load("b28_target_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts, max_inner_steps=64).unwrapped
    tgt_idx = env.target_node_indices

    class RefStyle:  # the reference protocol: predict(state, target, deterministic) -> (action, _)
        def predict(self, state, target, deterministic=True):
            for i in tgt_idx:
                if int(state[i]) == 0:
                    return (i + 1, None)
            return (0, None)

    class Batched:  # device-side protocol
        def predict_batch(self, obs):
            sub = obs[:, tgt_idx]
            zero = (sub == 0)
            first = torch.argmax(zero.to(torch.int32), dim=1)
            idx = torch.tensor(tgt_idx, device=obs.device)[first] + 1
            return torch.where(zero.any(1), idx, torch.zeros_like(idx)).to(torch.int32)

    a, _ = compute_ssd_hist(env, model=RefStyle(), iters=64 * 40, resets=64, seed=5)
    b, _ = compute_ssd_hist(env, model=Batched(), iters=64 * 40, resets=64, seed=5)
    va, vb = np.asarray(a["Value"]), np.asarray(b["Value"])
    assert abs(va.sum() - 1.0) < 1e-12 and np.array_equal(va, vb)
    assert va[-1] > 0.3  # the policy drives the target genes to all-ones


def test_eval_increase():
    import gym_PBN
    from gym_PBN.utils.eval import eval_increase

    z = load("b28_target_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts, max_inner_steps=64).unwrapped
    env.target_node_values = ((1, 1, 1, 1, 1, 1, 1),)
    tgt_idx = env.target_node_indices

    class Policy:
        def predict_batch(self, obs):
            zero = obs[:, tgt_idx] == 0
            first = torch.argmax(zero.to(torch.int32), dim=1)
            idx = torch.tensor(tgt_idx, device=obs.device)[first] + 1
            return torch.where(zero.any(1), idx, torch.zeros_like(idx)).to(torch.int32)

    inc = eval_increase(env, Policy(), iters=128 * 30, resets=128)
    assert 0.0 < inc <= 1.0  # steering every target gene to 1 raises the mass of the all-ones pattern


def test_exact_attractors_on_gpu_match_host_and_reference():
    """Terminal SCCs of the exhaustive async STG computed on the device == the host search == the reference's
    compute_attractors (recorded for five random networks and the example network)."""
    from gym_PBN.b200 import attractors, compiler, engine
    from gym_PBN.envs.common.node import Node
    from gym_PBN.envs.common.pbn import PBN

    z = load("tt_attractors.npz")
    for k in range(int(z["n_nets"])):
        masks, tables = z[f"n{k}/masks"], z[f"n{k}/tables"]
        n = len(masks)
        data = [(masks[i], tables[i, : 2 ** int(masks[i].sum())], f"g{i}", False) for i in range(n)]
        net = engine.Network(compiler.compile_pbn_data(data))
        got = sorted(sorted(a) for a in attractors.attractor_state_sets(net))
        states = [tuple(int(v) for v in s) for s in z[f"n{k}/att_states"]]
        want, pos = [], 0
        for sz in z[f"n{k}/att_sizes"]:
            want.append(sorted(states[pos:pos + sz]))
            pos += sz
        assert got == sorted(want), k
    # larger random networks against the host search
    rng = np.random.default_rng(3)
    for n in (11, 14, 16):
        data = []
        for i in range(n):
            kin = int(rng.integers(1, 4))
            mask = np.zeros(n, bool)
            mask[rng.choice(n, size=kin, replace=False)] = True
            table = rng.choice([0.0, 1.0, 1.0, 0.0, 0.4], size=2**kin)
            data.append((mask, table, f"g{i}", False))
        net = engine.Network(compiler.compile_pbn_data(data))
        pbn = PBN.__new__(PBN)
        pbn.N = n
        pbn.nodes = np.empty(n, dtype=object)
        for i, (m, t, *_r) in enumerate(data):
            pbn.nodes[i] = Node(m, t, i)
        host = sorted(sorted(a) for a in pbn.attractors_host())
        dev = sorted(sorted(a) for a in attractors.attractor_state_sets(net, list_limit=1 << 20))
        assert dev == host, n


def test_exact_attractors_predictor_graph_28():
    """The shipped 28-gene predictor graph: every reported attractor is closed under the dynamics (no change mask leads out)."""
    from gym_PBN.b200 import attractors, compiler, engine

    net = engine.Network(compiler.load_bittner("28_15_median"))
    found = attractors.exact_attractors(net, list_limit=4096)
    assert found and sum(a["size"] for a in found) >= 1
    stg = attractors.StateTransitionGraph(net)
    for a in found[:3]:
        bits = a["bits"] if a["bits"] is not None else stg.single(int(a["states"][0]))
        fwd = stg.reach(bits, 0)
        assert torch.equal(fwd, bits)  # closed: nothing outside is reachable
    print("Bittner-28 attractors:", [a["size"] for a in found][:10], "count", len(found))


def test_bittner28_default_attractors_are_exact():
    """gym.make("gym-PBN/Bittner-28-v0") without an attractor list: exact terminal SCCs of the async STG, as cubes."""
    import gym_PBN
    from gym_PBN.b200 import attractors

    env = gym_PBN.make("gym-PBN/Bittner-28-v0", seed=3)
    core = env.unwrapped
    assert core.attractor_source == "exact" and len(core.all_attractors) >= 2
    sizes = sorted(sum(2 ** sum(v == "*" for v in c) for c in a) for a in core.all_attractors)
    found = attractors.exact_attractors(core.network, list_limit=1 << 17)
    assert sizes == sorted(a["size"] for a in found)
    small = min(found, key=lambda a: a["size"])
    cubes = next(a for a in core.all_attractors if sum(2 ** sum(v == "*" for v in c) for c in a) == small["size"])
    listed = {tuple((int(s) >> i) & 1 for i in range(28)) for s in small["states"]}
    assert {t for c in cubes for t in attractors.expand_cube(c)} == listed
    for t in list(listed)[:20]:
        assert core.is_attracting_state(t)
    (state, target), _ = env.reset(seed=3)
    assert core.is_attracting_state(state)
    for a in (0, 5, 0, 17, 0):
        obs, r, term, trunc, info = env.step(a)
        assert core.is_attracting_state(obs) or info["inner_cap_hit"]


def test_vector_env_multi_matches_oracle():
    """PBNVectorEnv over PBNTargetMultiEnv (K = 3 action slots, tensor semantics = duplicates dropped), fused step + reset."""
    import gym_PBN
    from gym_PBN.b200.vector_env import PBNVectorEnv

    z = load("b28_multi_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/BittnerMulti-28-v0", all_attractors=atts, max_inner_steps=48, horizon=9)
    B, seed = 2048, 23
    vec = PBNVectorEnv(env, B, seed=seed, action_slots=3, dedup=True)
    obs, info = vec.reset()
    sets, ids = orc.load_bittner("28_15_median")
    onet = orc.net_from_predictor_sets(sets, ids)
    oenv = orc.Env(orc.ENV_MULTI, 28, attractors=atts, horizon=9, max_inner=48, dedup=1)
    ost = np.zeros((B, 28), np.uint8)
    ons, ota = np.zeros(B, np.int32), np.zeros(B, np.int32)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    assert np.array_equal(obs.cpu().numpy(), ost) and np.array_equal(info["target_attractor"].cpu().numpy(), ota)
    rng = np.random.default_rng(5)
    for t in range(15):
        act = rng.integers(0, 29, size=(B, 3)).astype(np.int32)
        dup = rng.random(B) < 0.3
        act[dup, 2] = act[dup, 0]
        obs, rew, term, trunc, info = vec.step(torch.from_numpy(act))
        oobs, orew, oterm, otrunc, oin = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + 2 * t))
        assert np.array_equal(rew.cpu().numpy(), orew) and np.array_equal(term.cpu().numpy(), oterm.astype(bool))
        assert np.array_equal(trunc.cpu().numpy(), otrunc.astype(bool)) and np.array_equal(info["inner_steps"].cpu().numpy(), oin)
        assert np.array_equal(vec.sim.unpack(info["final_obs_packed"]).cpu().numpy(), oobs)
        done = (oterm | otrunc).astype(np.uint8)
        orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=2 + 2 * t), mask=done)
        want = np.where(done[:, None].astype(bool), ost, oobs)  # reset envs observe their new state, the rest the step's obs
        assert np.array_equal(obs.cpu().numpy(), want)
    assert vec.stats.reduced()["env_steps"] == 15 * B


def test_eval_winrate_matches_single_env_loop():
    """eval_winrate (utils/eval.py:160-197, working version): lockstep GPU episodes == the reference's per-state loop run
    through the single-env API, for a deterministic network (no probabilistic node) and a fixed policy."""
    import itertools

    import gym_PBN
    from gym_PBN.utils.eval import eval_winrate

    det = (["a", "b", "c", "d"], [[("a", 1.0)], [("a or c", 1.0)], [("not d", 1.0)], [("b and c", 1.0)]])
    goal = {"target_nodes": {(0, 1, 1, 0)}, "target": {(0, 1, 1, 0)}, "all_attractors": [{(0, 1, 1, 0)}, {(0, 0, 0, 0)}]}

    class Policy:
        def predict(self, obs, target=None, deterministic=True):
            return (int(obs[2]) + 1, 2)  # flip node obs[2], hold for 2 steps

        def predict_batch(self, obs):
            return torch.stack([obs[:, 2].to(torch.int32) + 1, torch.full_like(obs[:, 2], 2, dtype=torch.int32)], dim=1)

    env = gym_PBN.make("gym-PBN/PBN-sampled-data-v0", logic_func_data=det, goal_config=dict(goal), T=4)
    rate, inter, steps = eval_winrate(env, Policy(), max_episode_steps=6)
    # the reference loop, one start state at a time; the update picks a random node, so compare the laws loosely and the
    # bookkeeping exactly where it is deterministic
    wins = n = 0
    lens = []
    for state in itertools.product([0, 1], repeat=4):
        if state in env.unwrapped.target_nodes:
            continue
        n += 1
        env.reset()
        env.unwrapped.set(np.array(state, dtype=bool))
        obs = np.array(state, dtype=bool)
        for j in range(1, 7):
            obs, _r, term, trunc, info = env.step(Policy().predict(obs))
            if term:
                wins += 1
            if term or j == 6:
                lens.append(j)
                break
    assert n == 16 - len(env.unwrapped.target_nodes) and 0.0 <= rate <= 1.0 and 1.0 <= inter <= 6.0
    assert abs(steps - inter) < 1e-9  # PBN-sampled-data reports interval - 1 = 1 per interaction
    assert abs(rate - wins / n) <= 0.5 and abs(inter - np.mean(lens)) <= 2.5
    with pytest.raises(ValueError):
        eval_winrate(env.unwrapped, Policy())  # no step limit anywhere


def test_rollout_buffer_and_training_example(monkeypatch, capsys):
    """Device-resident rollouts over the vector env, and the actor-critic example end to end (two small updates)."""
    import importlib.util
    import sys as _sys
    from pathlib import Path

    import gym_PBN
    from gym_PBN.b200.rollout import RolloutBuffer
    from gym_PBN.b200.vector_env import PBNVectorEnv

    z = load("b28_target_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts, max_inner_steps=32)
    vec = PBNVectorEnv(env, 256, seed=3)
    buf = RolloutBuffer(vec, horizon=5, gamma=0.9)

    def policy(obs):
        a = torch.randint(0, 29, (obs.shape[0], 1), device=obs.device, dtype=torch.int32)
        return a, None, torch.zeros(obs.shape[0], device=obs.device)

    last = buf.collect(policy)
    assert buf.t == 5 and buf.obs.shape == (6, 256, 28) and last.shape == (256, 28)
    assert set(buf.rewards.unique().tolist()) <= {20.0, -5.0}
    ret = buf.returns()
    adv, tgt = buf.gae(torch.zeros(256, device=vec.device))
    assert ret.shape == adv.shape == tgt.shape == (5, 256)
    assert torch.allclose(ret[-1], buf.rewards[-1])
    o, a, r, o2, te = buf.transitions()
    assert o.shape == (5 * 256, 28) and a.shape == (5 * 256, 1) and torch.equal(o2[:256], buf.obs[1])

    path = Path(__file__).resolve().parents[1] / "examples" / "train_vector_policy.py"
    spec = importlib.util.spec_from_file_location("train_vector_policy", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    monkeypatch.setattr(_sys, "argv", ["train_vector_policy.py", "--envs", "512", "--updates", "2", "--horizon", "4", "--max-inner", "32"])
    mod.main()
    out = capsys.readouterr().out
    assert "update   1" in out and "env-steps/s" in out


def test_graph_analysis_helpers_match_reference():
    """Host-side analysis surface of the Bittner graph (getStateProbs, getNextStates, forced-node step, genSTG,
    findAttractors, sync_getNextStates) against vectors recorded from the reference (oracle/make_analysis_golden.py)."""
    import random

    from gym_PBN.envs.bittner import base, utils

    z = load("graph_analysis.npz")
    g = utils.spawn(total_genes=28, seed=1)
    for k, s in enumerate(z["b28_states"]):
        g.setState(list(s))
        probs = np.array([node.getStateProbs(g.getState()) for node in g.nodes])
        assert np.allclose(probs, z["b28_probs"][k], rtol=0, atol=1e-12)
        d = g.getNextStates()
        lo, hi = z["b28_next_off"][k], z["b28_next_off"][k + 1]
        assert sorted(d) == [tuple(int(v) for v in r) for r in z["b28_next_states"][lo:hi]]
        assert np.allclose([d[key] for key in sorted(d)], z["b28_next_probs"][lo:hi], rtol=0, atol=1e-12)
        assert abs(sum(d.values()) - 1.0) < 1e-9
    g.setState(list(z["b28_states"][0]))
    random.seed(5)
    for k, want in enumerate(z["b28_forced_trace"]):
        assert list(g.step(i=(7 * k) % 28)) == list(want), k
    # labelled (ID-keyed) states work too
    assert g.nodes[3].getStateProbs(g.getLabeledState()) == g.nodes[3].getStateProbs(g.getState())

    n, F = z["s6_cod"].shape
    nodes = []
    for i in range(n):
        buf = np.empty((3, F), dtype=object)
        for f in range(F):
            buf[0, f], buf[1, f] = float(z["s6_cod"][i, f]), z["s6_A"][i, f].reshape(4, 1)
            buf[2, f] = np.array([int(z["s6_ids"][t]) for t in z["s6_inp"][i, f]])
        node = base.Node(i, i, f"g{i}", int(z["s6_ids"][i]))
        node.add_predictors(buf)
        nodes.append(node)
    g6 = base.Graph(2)
    g6.add_nodes(nodes)
    stg = g6.genSTG()
    assert sorted(u + v for u, v in stg.edges()) == [tuple(int(x) for x in r) for r in z["s6_edges"]]
    atts = sorted(sorted(a) for a in base.findAttractors(stg))
    want = [[tuple(int(x) for x in r) for r in z["s6_att_states"][z["s6_att_off"][a]:z["s6_att_off"][a + 1]]]
            for a in range(len(z["s6_att_off"]) - 1)]
    assert atts == want
    assert sorted(sorted(a) for a in g6.getAttractors()) == want  # the exhaustive device search agrees
    g6.setState([1, 0, 1, 1, 0, 0])
    d = g6.sync_getNextStates()
    assert sorted(d) == [tuple(int(x) for x in r) for r in z["s6_sync_states"]]
    assert np.allclose([d[k] for k in sorted(d)], z["s6_sync_probs"], rtol=0, atol=1e-12)
    assert g6.printGraph().number_of_nodes() == 6
    from gym_PBN.envs import PBNTargetEnv

    env6 = PBNTargetEnv(g6, {"target_nodes": [101], "intervene_on": [101], "target_node_values": ((0,),),
                             "undesired_node_values": tuple(), "horizon": 5}, "human")
    assert env6.render(mode="STG").number_of_edges() == len(z["s6_edges"]) and env6.render(mode="PBN").number_of_nodes() == 6


def test_env_reward_helpers():
    """_get_reward / compute_attractors / _to_map of the env classes give what env.step reports."""
    import gym_PBN

    env = gym_PBN.make("gym-PBN/PBN-v0", logic_func_data=EX5, goal_config=dict(GOAL)).unwrapped
    assert env._get_reward((0, 0, 0, 0, 1), 0) == (20, True, False)
    assert env._get_reward((0, 0, 1, 0, 0), 2) == (-5, False, False)
    assert env._get_reward((1, 1, 1, 1, 1), 0) == (-4, False, False)  # is_attracting_state is constant True (pbn_env.py:19-21)
    penv = gym_PBN.make("gym-PBN/PBCN-v0", logic_func_data=EX5, goal_config=dict(GOAL)).unwrapped
    assert penv._get_reward((0, 0, 0, 0, 1))[:2] == (penv.successful_reward, True)
    assert penv._get_reward((0, 0, 1, 0, 0))[0] == -penv.wrong_attractor_cost
    assert len(list(penv.PBN.control_actions)) == 2 ** penv.PBN.N
    assert penv.PBN._compute_next_states(np.array([0, 0, 1, 0, 0], bool)) == []  # a fixed point: no node can change
    assert all(len(t) == 3 for t in penv.PBN._async_compute_next_states(np.array([0, 1, 1, 1, 0], bool)))
    node = env.PBN.nodes[3]
    assert node.compute_next_value(np.array([0, 1, 0, 0, 0], bool)) in (True, False)
    assert all(len(t) == 3 for t in env.PBN._compute_next_states(np.array([0, 1, 0, 0, 0], bool)))

    z = load("b28_target_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    tenv = gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts, max_inner_steps=64, seed=5).unwrapped
    tenv.reset(seed=3)
    obs, r, term, trunc, _ = tenv.step(0)
    assert tenv._get_reward(tenv._to_map(obs), 0)[:2] == (r, term)
    assert tenv.dep_is_attracting_state(obs) is True
    with pytest.raises(ValueError):
        tenv.also_dep_is_attracting_state(obs)
    found = tenv.compute_attractors()
    assert sorted(len(a) for a in found) == [120, 49152]  # the two attractors of the 28-gene network (DESIGN.md §7)


@pytest.mark.parametrize("tag", ["pbn", "pbcn"])
def test_self_triggering_envs_replay_reference(tag):
    """PB(C)NSelfTriggeringEnv.step (one kernel launch per macro step) under replayed draws against traces recorded from
    the reference (oracle/make_st_golden.py): observation, discounted reward (exact float64), terminated, interval; and the
    same kernel in Philox mode against the oracle."""
    import gym_PBN
    from gym_PBN.b200 import abi, engine

    z = load("ex5_self_triggering.npz")
    T = 5 if tag == "pbn" else 7
    env_id = "gym-PBN/PBN-self-triggering-v0" if tag == "pbn" else "gym-PBN/PBCN-self-triggering-v0"
    env = gym_PBN.make(env_id, logic_func_data=EX5, goal_config=dict(GOAL), gamma=0.9, T=T).unwrapped
    env.reset(seed=1)
    for k in range(len(z[f"{tag}_interval"])):
        n = int(z[f"{tag}_interval"][k])
        env.set(z[f"{tag}_start"][k].astype(bool))
        env.replay_draws(z[f"{tag}_ints"][k][:n], z[f"{tag}_dbls"][k][:2 * n])  # per primitive step: node, value, stop
        a0, a1 = (int(v) for v in z[f"{tag}_action"][k])
        obs, r, term, trunc, info = env.step((a0, a1) if tag == "pbn" else ([bool(a0)], a1))
        assert info["interval"] == n, k
        assert np.array_equal(np.asarray(obs).astype(np.uint8), z[f"{tag}_obs"][k]), k
        assert r == z[f"{tag}_reward"][k] and term == bool(z[f"{tag}_term"][k]), (k, r, z[f"{tag}_reward"][k])

    # Philox mode, many envs: kernel == oracle (float64 rewards bit for bit)
    B, seed = 777, 21
    rng = np.random.default_rng(4)
    kind, okind = (abi.ENV_PBN_ST, orc.ENV_PBN_ST) if tag == "pbn" else (abi.ENV_PBCN_ST, orc.ENV_PBCN_ST)
    atts = [[(0, 0, 1, 0, 0)], [(0, 0, 0, 0, 1)]]
    common = dict(attractors=atts, targets=[(0, 0, 0, 0, 1)], n_control=1, successful_reward=1, wrong_attractor_cost=1,
                  gamma=0.97, max_interval=T)
    img = engine.EnvImage(env.network, kind, **common)
    oenv = orc.Env(okind, 5, **common)
    from gym_PBN.utils.converters import logic_funcs_to_PBN_data

    onet = orc.net_from_pbn_data(logic_funcs_to_PBN_data(*EX5))
    sim = engine.Simulator(env.network, B, seed=seed)
    st0 = rng.integers(0, 2, size=(B, 5)).astype(np.uint8)
    sim.set_state(st0)
    ost = st0.copy()
    for t in range(3):
        act = (np.stack([rng.integers(0, 6, B), rng.integers(1, 11, B)], 1) if tag == "pbn"
               else np.stack([rng.integers(1, 11, B), rng.integers(0, 2, B)], 1)).astype(np.int32)
        sim.env_step(img, torch.from_numpy(act))
        obs, rf, term, inner = orc.env_step_f64(onet, oenv, ost, act, orc.Draws(seed=seed, epoch=sim.epoch - 1))
        assert np.array_equal(sim.unpack().cpu().numpy(), ost), t
        assert np.array_equal(sim.reward_f64.cpu().numpy(), rf) and np.array_equal(sim.inner.cpu().numpy(), inner), t
        assert np.array_equal(sim.terminated.cpu().numpy(), term), t


def _class_level_replay(env, tr, K, step, on_reset):
    """Drives an env CLASS through a golden trace of the reference: reset ops restore the recorded state by hand, step ops
    queue the recorded draws (env.replay_draws) and call env.step."""
    for t in range(tr.T):
        ints, dbls = tr.draws(t)
        if tr.op[t] == 1:
            on_reset(t)
            continue
        env.replay_draws(ints, dbls)
        obs, r, term, trunc, _info = step(tr.act[t, :K])
        assert np.array_equal(np.asarray(obs).astype(np.uint8), tr.obs[t]), ("obs", t)
        assert (int(r), bool(term), bool(trunc)) == (int(tr.reward[t]), bool(tr.term[t]), bool(tr.trunc[t])), ("reward", t)


def test_env_classes_replay_reference_traces():
    """The drop-in env CLASSES (not only the engine) against traces recorded from the reference classes, draws replayed."""
    from golden_util import Traj, pbn_data_from

    import gym_PBN
    from gym_PBN.envs import PBNEnv, PBNTargetEnv, PBNTargetMultiEnv
    from gym_PBN.envs.bittner import utils

    z = load("ex5_pbnenv.npz")
    env = PBNEnv(logic_func_data=EX5, goal_config=dict(GOAL))
    for e in range(int(z["n_traj"])):
        tr = Traj(z, e)
        _class_level_replay(env, tr, 1, lambda a: env.step(int(a[0])), lambda t: env.set(tr.state[t].astype(bool)))

    for fname, cls, K in (("b28_target_env.npz", PBNTargetEnv, 1), ("b28_multi_env.npz", PBNTargetMultiEnv, 3)):
        z = load(fname)
        atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
        goal = {"target_nodes": [234237], "intervene_on": [234237], "target_node_values": ((0,),),
                "undesired_node_values": tuple(), "horizon": int(z["horizon"])}
        for e in range(int(z["n_traj"])):
            if f"e{e}/op" not in z.files:
                continue
            tr = Traj(z, e)
            env = cls(utils.spawn(total_genes=28), dict(goal), "human", all_attractors=atts, max_inner_steps=int(z["cap"]))
            force = bool(z[f"e{e}/force"]) if f"e{e}/force" in z.files else False
            as_list = f"e{e}/dedup" in z.files and not bool(z[f"e{e}/dedup"])

            def on_reset(t, env=env, tr=tr):
                env.graph.setState(list(tr.state[t]))
                env.n_steps = 0
                env.setTarget(env._all_attractors[int(tr.target_att[t])])

            def step(a, env=env, force=force, as_list=as_list):
                if K == 1:
                    return env.step(int(a[0]), force=force)
                acts = [int(v) for v in a if v >= 0]
                return env.step(acts if as_list else torch.tensor(acts))

            _class_level_replay(env, tr, K, step, on_reset)


@pytest.mark.parametrize("tag", ["pbn", "pbcn"])
def test_vector_env_self_triggering_matches_oracle(tag):
    """PBNVectorEnv over the self-triggering envs: macro step + masked auto-reset against the oracle (float64 rewards,
    intervals, observations, episode statistics), epoch for epoch."""
    import gym_PBN
    from gym_PBN.b200.vector_env import PBNVectorEnv
    from gym_PBN.utils.converters import logic_funcs_to_PBN_data

    T = 5 if tag == "pbn" else 7
    env_id = "gym-PBN/PBN-self-triggering-v0" if tag == "pbn" else "gym-PBN/PBCN-self-triggering-v0"
    env = gym_PBN.make(env_id, logic_func_data=EX5, goal_config=dict(GOAL), gamma=0.9, T=T).unwrapped
    B, seed = 1500, 9
    vec = PBNVectorEnv(env, B, seed=seed)
    assert vec.family == "st" and vec.action_width == 2
    okind = orc.ENV_PBN_ST if tag == "pbn" else orc.ENV_PBCN_ST
    atts = [sorted(a) for a in env.all_attractors]
    oenv = orc.Env(okind, 5, attractors=atts, targets=env._target_states(), n_control=getattr(env.PBN, "M", 0),
                   successful_reward=env.successful_reward, wrong_attractor_cost=env.wrong_attractor_cost, gamma=0.9,
                   max_interval=T)
    onet = orc.net_from_pbn_data(logic_funcs_to_PBN_data(*EX5))
    ost, ons, ota = np.zeros((B, 5), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
    obs, _ = vec.reset()
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    assert np.array_equal(obs.cpu().numpy(), ost)
    rng = np.random.default_rng(2)
    ep_ret, ep_len = np.zeros(B), np.zeros(B, np.int64)
    episodes = successes = 0
    ret_sum = 0.0
    for t in range(6):
        act = (np.stack([rng.integers(0, 6, B), rng.integers(1, 11, B)], 1) if tag == "pbn"
               else np.stack([rng.integers(1, 11, B), rng.integers(0, 2, B)], 1)).astype(np.int32)
        obs, r, te, tr, info = vec.step(torch.from_numpy(act))
        _o, rf, term, inner = orc.env_step_f64(onet, oenv, ost, act, orc.Draws(seed=seed, epoch=1 + 2 * t))
        assert np.array_equal(vec.final_obs.cpu().numpy()[0], (ost.astype(np.int32) << np.arange(5)).sum(1)), t  # before the reset
        done = term.astype(bool)
        orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=2 + 2 * t), mask=done)
        assert np.array_equal(obs.cpu().numpy(), ost), t
        assert np.array_equal(r.cpu().numpy(), rf) and r.dtype == torch.float64, t
        assert np.array_equal(te.cpu().numpy(), done) and not tr.any(), t
        assert np.array_equal(info["interval"].cpu().numpy(), inner), t
        ep_ret += rf
        ep_len += 1
        episodes += int(done.sum()); successes += int(done.sum())
        ret_sum += float((ep_ret * done).sum())
        ep_ret[done] = 0; ep_len[done] = 0
        assert np.array_equal(vec.ep_return.cpu().numpy(), ep_ret) and np.array_equal(vec.ep_len.cpu().numpy(), ep_len), t
    s = vec.stats.reduced()
    assert s["episodes"] == episodes and s["successes"] == successes and s["env_steps"] == 6 * B and episodes > 0
    assert abs(float(vec.return_sum_f64) - ret_sum) < 1e-9 * max(1.0, abs(ret_sum))


@pytest.mark.parametrize("plan", [None, (4, 16)])
def test_vector_env_out_of_range_actions_are_ignored_and_counted(plan):
    """A policy network can emit anything: an action outside [0, N] must not touch another env's state column or the staged
    network image; the intervention is dropped (the step equals action 0) and counted in the statistics.  The planned step
    counts it too for the envs its first pass parks (their intervention is not applied again when they resume)."""
    import gym_PBN
    from gym_PBN.b200.vector_env import PBNVectorEnv

    z = load("b28_target_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts, max_inner_steps=32)
    B, seed = 2048, 23
    vec_bad, vec_ok = PBNVectorEnv(env, B, seed=seed), PBNVectorEnv(env, B, seed=seed)
    if plan is not None:
        vec_bad.sim.plan_budgets = vec_ok.sim.plan_budgets = plan
    vec_bad.reset(), vec_ok.reset()
    rng = np.random.default_rng(3)
    n_bad = 0
    for t in range(6):
        act = rng.integers(0, 29, size=(B, 1)).astype(np.int32)
        wild = act.copy()
        sel = rng.random(B) < 0.2
        wild[sel, 0] = rng.choice([-7, 29, 1000, -2**31, 2**31 - 1, 4096 * 33], size=int(sel.sum()))
        act[sel, 0] = 0
        n_bad += int(sel.sum())
        ob, rb, tb, ub, _ = vec_bad.step(torch.from_numpy(wild))
        oo, ro, to, uo, _ = vec_ok.step(torch.from_numpy(act))
        assert torch.equal(ob, oo) and torch.equal(rb, ro) and torch.equal(tb, to) and torch.equal(ub, uo)
    assert vec_bad.stats.reduced()["invalid_actions"] == n_bad and vec_ok.stats.reduced()["invalid_actions"] == 0


def test_self_triggering_prob_is_clamped():
    """prob = 0 would give a stop threshold of 0: with no interval cap the macro step would never end (a GPU hang)."""
    import gym_PBN
    from gym_PBN.b200.vector_env import PBNVectorEnv

    env = gym_PBN.make("gym-PBN/PBN-self-triggering-v0", logic_func_data=EX5, goal_config=dict(GOAL))
    vec = PBNVectorEnv(env, 256, seed=1)
    vec.reset()
    act = np.zeros((256, 2), np.int32)
    act[:, 1] = np.random.default_rng(0).choice([0, -5, 11, 100], size=256)
    obs, rew, term, trunc, info = vec.step(torch.from_numpy(act))
    torch.cuda.synchronize()
    assert int(info["interval"].min()) >= 1 and int(info["interval"].max()) < 500


@pytest.mark.parametrize("sample_pair,plan", [(False, None), (True, None), (True, (4, 16))])
def test_vector_env_curriculum_matches_oracle(sample_pair, plan):
    """Device-side curriculum of PBNTargetMultiEnv (pbn_target_multi.py:159-181, 232-235): every env's own probability row is
    reworked when its episode ends and the reset draws the attractor pair from it — product (fused in the step launch) vs the
    oracle (step, then per finished env rework_probas + reset), bit for bit, float64 rows included."""
    import gym_PBN
    from gym_PBN.b200.vector_env import PBNVectorEnv

    rng = np.random.default_rng(8)
    n = 28
    atts = []
    for a in range(5):
        c = ["*"] * n
        for i in rng.choice(n, size=3, replace=False):
            c[i] = int(rng.integers(0, 2))
        atts.append([tuple(c)])
    env = gym_PBN.make("gym-PBN/BittnerMulti-28-v0", all_attractors=atts, max_inner_steps=40, horizon=25, sample_pair=sample_pair)
    B, seed = 1500, 31
    vec = PBNVectorEnv(env, B, seed=seed, curriculum=True, action_slots=2)
    if plan is not None:  # a step of several budgeted passes: finished envs are reset by ONE masked launch after the last pass
        vec.sim.plan_budgets = plan
    obs, info = vec.reset()
    sets, ids = orc.load_bittner("28_15_median")
    onet = orc.net_from_predictor_sets(sets, ids)
    oenv = orc.Env(orc.ENV_MULTI, n, attractors=atts, horizon=env.unwrapped.horizon if hasattr(env, "unwrapped") else 25, max_inner=40, dedup=1)
    ost, ons, ota = np.zeros((B, n), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
    prob = np.full((B, 5), 0.2)
    pair = np.zeros((B, 2), np.int32)
    orc.env_reset_cur(onet, oenv, ost, ons, ota, prob, pair, orc.Draws(seed=seed, epoch=0), sample_pair=sample_pair)
    assert np.array_equal(obs.cpu().numpy(), ost) and np.array_equal(vec.pair_ids.cpu().numpy(), pair)
    assert np.array_equal(vec.sim.target_att.cpu().numpy(), ota)
    ep_len = np.zeros(B, np.int64)
    ends = 0
    for t in range(60):
        act = rng.integers(0, n + 1, size=(B, 2)).astype(np.int32)
        obs, rew, term, trunc, info = vec.step(torch.from_numpy(act))
        oobs, orew, oterm, otrunc, oin = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + 2 * t))
        assert np.array_equal(rew.cpu().numpy(), orew) and np.array_equal(term.cpu().numpy(), oterm.astype(bool))
        ep_len += 1
        done = (oterm | otrunc).astype(np.uint8)
        for e in np.nonzero(done)[0]:
            orc.rework_probas(prob[e], pair[e, 0], pair[e, 1], int(ep_len[e]))
        ep_len[done.astype(bool)] = 0
        ends += int(done.sum())
        orc.env_reset_cur(onet, oenv, ost, ons, ota, prob, pair, orc.Draws(seed=seed, epoch=2 + 2 * t), sample_pair=sample_pair, mask=done)
        # MULTI observes the state captured before its last update (Q11); envs that were reset observe their new state
        assert np.array_equal(obs.cpu().numpy(), np.where(done[:, None].astype(bool), ost, oobs))
        assert np.array_equal(vec.sim.unpack().cpu().numpy(), ost)
        assert np.array_equal(vec.pair_ids.cpu().numpy(), pair) and np.array_equal(vec.sim.target_att.cpu().numpy(), ota)
        assert np.array_equal(vec.probabilities.cpu().numpy(), prob)  # float64, bit for bit
    assert ends > B and not np.allclose(prob, 0.2)  # episodes ended and the tables moved
    sd = vec.state_dict()
    vec2 = PBNVectorEnv(env, B, seed=0, curriculum=True, action_slots=2)
    vec2.load_state_dict(sd)
    act = torch.from_numpy(rng.integers(0, n + 1, size=(B, 2)).astype(np.int32))
    assert torch.equal(vec.step(act)[0].clone(), vec2.step(act)[0]) and torch.equal(vec.probabilities, vec2.probabilities)


@pytest.mark.parametrize("family", ["target", "multi"])
def test_vector_env_cuda_graph_step_is_bit_identical(family):
    """cuda_graph=True: step() replays one captured graph (the planned step launches + unpack + epoch increment, epoch in
    device memory) — same observations, rewards, flags and statistics as the eager env, resets and reloads in between."""
    import gym_PBN
    from gym_PBN.b200.vector_env import PBNVectorEnv

    z = load("b28_target_env.npz" if family == "target" else "b28_multi_env.npz")
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = gym_PBN.make("gym-PBN/Bittner-28-v0" if family == "target" else "gym-PBN/BittnerMulti-28-v0", all_attractors=atts,
                       max_inner_steps=200)
    B, seed = 3000, 5
    kw = dict(curriculum=True, action_slots=2) if family == "multi" else {}
    a, b = PBNVectorEnv(env, B, seed=seed, **kw), PBNVectorEnv(env, B, seed=seed, cuda_graph=True, **kw)
    oa, _ = a.reset()
    ob, _ = b.reset()
    assert torch.equal(oa, ob)
    rng = np.random.default_rng(1)
    width = a.action_width
    for t in range(12):
        act = torch.from_numpy(rng.integers(0, 29, size=(B, width)).astype(np.int32))
        ra, rb = a.step(act), b.step(act)
        for x, y in zip(ra[:4], rb[:4]):
            assert torch.equal(x, y), t
        assert torch.equal(ra[4]["inner_steps"], rb[4]["inner_steps"])
        if t == 5:  # epochs consumed outside the graph
            assert torch.equal(a.reset()[0], b.reset()[0])
        if t == 8:
            sd = a.state_dict()
            a.load_state_dict(sd), b.load_state_dict(sd)
    assert b._graph is not None and a.stats.reduced() == b.stats.reduced() and a.sim.epoch == b.sim.epoch
