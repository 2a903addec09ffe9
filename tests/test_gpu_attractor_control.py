"""GPU: pbn_env_attractor_index (engine.attractor_index) against the host's cube test, and gym_PBN.utils.control against
the oracle (bit for bit), against exact landing probabilities of the explicit state-transition graph, and — for
attractor_policy — against a Monte-Carlo run of the policy on the real vector env."""
import ctypes as C
import functools
import json

import numpy as np
import pytest

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

import control_util as cu  # noqa: E402
from golden_util import GOLD, random_tt_data  # noqa: E402

BATCHES = (1, 31, 257, 65536)


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gym_PBN.b200 import abi, compiler, engine

    return abi, compiler, engine


def _tt_env(pbn_data, atts, cap=1 << 20):
    """PBNTargetEnv on a truth-table network."""
    from gym_PBN.b200 import compiler
    from gym_PBN.envs.bittner import base
    from gym_PBN.envs.pbn_target import PBNTargetEnv

    spec = compiler.compile_pbn_data(pbn_data)
    spec.ids = list(range(spec.n))
    goal = {"target_nodes": [0], "intervene_on": [0], "target_node_values": ((0,),), "undesired_node_values": (), "horizon": 100}
    return PBNTargetEnv(base.Graph.from_spec(spec), goal, all_attractors=atts, max_inner_steps=cap)


# ------------------------------------------------------------------------------------------------ 1. classification
def _random_atts(n, sizes, care, seed):
    """Attractors of len(sizes) groups of random cubes; each cube cares about a fraction `care` of the nodes."""
    rng = np.random.default_rng(seed)
    out = []
    for k in sizes:
        out.append([tuple(int(v) if c else "*" for v, c in zip(rng.integers(0, 2, n), rng.random(n) < care)) for _ in range(k)])
    return out


def _states(atts, n, B, seed):
    """B states: a third drawn inside cubes, a third uniformly random, a third one bit away from a state inside a cube."""
    rng = np.random.default_rng(seed)
    cubes = [c for a in atts for c in a]
    care = np.array([[v != "*" for v in c] for c in cubes])
    val = np.array([[0 if v == "*" else int(v) for v in c] for c in cubes], np.uint8)
    st = rng.integers(0, 2, size=(B, n)).astype(np.uint8)
    inside = np.nonzero(rng.random(B) < 2 / 3)[0]
    pick = rng.integers(0, len(cubes), size=len(inside))
    st[inside] = np.where(care[pick], val[pick], st[inside])
    near = inside[::2]
    st[near, rng.integers(0, n, size=len(near))] ^= 1
    return st


CLASSIFY = {  # name: (network, attractors)
    "b28-exact": ("28_15_median", "b28"),
    "b200-verified": ("200_5_kmeans", "b200"),
    "tt31": (31, ([1, 1, 2], 0.6)),
    "tt32": (32, ([3, 1, 4, 2], 0.3)),
    "tt33": (33, ([1, 2], 0.05)),   # nearly all-wildcard cubes: most states match
    "tt65": (65, ([2, 2, 5, 1, 3], 0.1)),
    "tt1024": (1024, ([1, 3, 2], 0.01)),
    "tt1024-global": (1024, ([170, 130, 200], 0.02)),  # 500 cubes x 32 words: the image is read from global memory
}


@functools.lru_cache(maxsize=None)
def _classify_case(name):
    net, att = CLASSIFY[name]
    if att == "b28":
        atts = cu.b28_attractors()
    elif att == "b200":
        atts = [[tuple(c) for c in a] for a in json.loads((GOLD / "b200_verified_attractors.json").read_text())]
    else:
        atts = _random_atts(net, *att, seed=net)
    n = len(atts[0][0])
    st = _states(atts, n, max(BATCHES), seed=n + len(atts))
    return atts, st, cu.classify(st, atts)


@gpu
@pytest.mark.parametrize("name", sorted(CLASSIFY))
def test_attractor_index_matches_host(eng, name):
    abi, compiler, engine = eng
    from gym_PBN.b200 import attractors as att_tools

    atts, st, want = _classify_case(name)
    net_id = CLASSIFY[name][0]
    spec = compiler.load_bittner(net_id) if isinstance(net_id, str) else compiler.compile_pbn_data(random_tt_data(net_id, seed=1))
    net = engine.Network(spec)
    assert net.n == st.shape[1]
    for e in range(257):  # the vectorised host test is att_tools.cube_matches
        ref = next((a for a, att in enumerate(atts) if any(att_tools.cube_matches(c, st[e]) for c in att)), -1)
        assert ref == want[e], (name, e)
    assert (want >= 0).any() and (want < 0).any() and len(set(want[want >= 0].tolist())) == len(atts)
    image = engine.EnvImage(net, abi.ENV_TARGET, attractors=atts)
    for B in BATCHES:
        sim = engine.Simulator(net, B)
        sim.set_state(st[:B])
        got = engine.attractor_index(sim, image).cpu().numpy()
        assert np.array_equal(got, want[:B]), (name, B)
        out = torch.full((B,), 7, dtype=torch.int32, device=net.device)
        assert engine.attractor_index(sim.state, image, out=out) is out and np.array_equal(out.cpu().numpy(), want[:B])


@gpu
def test_attractor_index_errors(eng):
    abi, compiler, engine = eng
    net = engine.Network(compiler.compile_pbn_data(random_tt_data(33, seed=1)))
    sim = engine.Simulator(net, 5)
    bare = engine.EnvImage(net, abi.ENV_TARGET)
    out = torch.zeros(5, dtype=torch.int32, device=net.device)
    rc = abi.lib().pbn_env_attractor_index(bare.handle, C.c_void_p(sim.state.data_ptr()), 5, C.c_void_p(out.data_ptr()), None)
    assert rc == 1 and "attractor" in abi.lib().pbn_last_error().decode()
    with pytest.raises(ValueError):
        engine.attractor_index(sim, bare)
    image = engine.EnvImage(net, abi.ENV_TARGET, attractors=[[("*",) * 33]])
    assert abi.lib().pbn_env_attractor_index(image.handle, None, 5, C.c_void_p(out.data_ptr()), None) == 1
    assert abi.lib().pbn_env_attractor_index(image.handle, C.c_void_p(sim.state.data_ptr()), 0, None, None) == 1
    with pytest.raises(ValueError):
        engine.attractor_index(sim.state[:1], image)  # wrong plane count
    with pytest.raises(ValueError):
        engine.attractor_index(sim, image, out=torch.zeros(4, dtype=torch.int32, device=net.device))


# ------------------------------------------------------------------------------------------------ 2. against the oracle
def _cap_env(name):
    import gym_PBN

    ref, atts = cu.cap_case(name)
    if name == "b28":
        return gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts, max_inner_steps=cu.CAP)
    return _tt_env(ref[1], atts, cap=cu.CAP)


@gpu
@pytest.mark.parametrize("name", sorted(cu.CAP_CASES))
def test_transitions_equal_oracle(eng, name):
    from gym_PBN.utils.control import attractor_transitions

    want = cu.oracle_transitions(name, cu.CAP_SAMPLES[name], cu.CAP_SEED)
    got = attractor_transitions(_cap_env(name), cu.CAP_SAMPLES[name], seed=cu.CAP_SEED, num_envs=cu.CAP_CASES[name])
    assert got.dtype == np.int64 and got.shape == want.shape
    assert np.array_equal(got, want)


@gpu
def test_transitions_multi_env_deterministic_and_argument_errors(eng):
    import gym_PBN
    from gym_PBN.utils.control import attractor_transitions

    atts = cu.b28_attractors()
    kw = dict(all_attractors=atts, max_inner_steps=cu.CAP)
    env = gym_PBN.make("gym-PBN/Bittner-28-v0", **kw)
    a = attractor_transitions(env, 40, seed=3, num_envs=2048)
    assert np.array_equal(a, attractor_transitions(env.unwrapped, 40, seed=3, num_envs=2048))
    assert np.array_equal(a, attractor_transitions(gym_PBN.make("gym-PBN/BittnerMulti-28-v0", **kw), 40, seed=3, num_envs=2048))
    assert not np.array_equal(a, attractor_transitions(env, 40, seed=4, num_envs=2048))
    with pytest.raises(ValueError):
        attractor_transitions(env, 40, force=True)
    with pytest.raises(ValueError):
        attractor_transitions(gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts[:1]), 40)
    with pytest.raises(TypeError):
        attractor_transitions(object(), 40)


# ------------------------------------------------------------------------------------------------ 3. exact ground truth
def _within(counts, P, k=5.0):
    """Every cell of the estimate counts / row total within k standard errors of the exact probability P."""
    n = counts.sum(2, keepdims=True)
    est = counts / n
    se = np.sqrt(np.clip(P * (1 - P), 0, None) / n)  # exact 0/1 cells can round a hair outside [0, 1]
    bad = np.abs(est - P) > k * se + 1e-12
    assert not bad.any(), (np.argwhere(bad)[:5], est[bad][:5], P[bad][:5])


@gpu
def test_transitions_match_exact_landing_probabilities(eng):
    from gym_PBN.utils.control import attractor_transitions

    data, atts = cu.ground_truth_net()
    P = cu.exact_landing(cu.transition_matrix(data), atts, len(data))
    counts = attractor_transitions(_tt_env(data, atts), 100_000, seed=7)
    assert counts.sum(2).min() >= 100_000
    _within(counts, P)


# ------------------------------------------------------------------------------------------------ 4. policy evaluation
@gpu
def test_policy_prediction_matches_the_env(eng):
    from gym_PBN.utils.control import attractor_policy, attractor_transitions, evaluate_attractor_policy

    data, atts = cu.fixed_point_net()
    env = _tt_env(data, atts)
    counts = attractor_transitions(env, 1_000_000, seed=1)
    _within(counts, cu.exact_landing(cu.transition_matrix(data), atts, len(data)))
    H, target, episodes = 3, 0, 200_000
    action, success = attractor_policy(counts, target, H)
    P = counts / counts.sum(2, keepdims=True)
    predicted = success[H].mean()  # the reset's start attractor is uniform
    assert np.isclose(predicted, cu.markov_optimum(P, target, H), rtol=0, atol=1e-12)
    assert cu.stationary_optimum(P, target, H) <= predicted + 1e-12
    rate, mean_steps = evaluate_attractor_policy(env, action, target, episodes, seed=5)
    se = np.sqrt(predicted * (1 - predicted) / episodes)
    assert abs(rate - predicted) <= 5 * se, (rate, predicted, se)
    assert 0 < mean_steps < H
    # a worse table is measured as worse: never intervening from the start
    rate0, _ = evaluate_attractor_policy(env, np.zeros_like(action), target, episodes, seed=5)
    assert rate0 < rate - 10 * se
