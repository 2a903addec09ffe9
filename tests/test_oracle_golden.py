"""CPU: the C oracle (oracle/pbn_oracle.c) replayed against golden vectors recorded from the
unmodified reference (oracle/make_golden.py).  Bit-exact: states, observations, rewards, flags,
and the number of draws consumed."""
import numpy as np
import pytest

import oracle as orc
from golden_util import Traj, cubes_to_attractors, load, pbn_data_from


def _rd(ints, dbls):
    return orc.Draws(ints=np.asarray(ints, np.int32).reshape(1, -1) if len(ints) else np.zeros((1, 1), np.int32),
                     dbls=np.asarray(dbls, np.float64).reshape(1, -1) if len(dbls) else np.zeros((1, 1), np.float64))


def _check_used(d, ints, dbls):
    assert tuple(d.used[0]) == (len(ints), len(dbls))


def test_philox_kat():
    # Random123 known-answer vectors for philox4x32-10
    assert orc.philox([0, 0, 0, 0], [0, 0]) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert orc.philox([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2) == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    assert orc.philox([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0]) == [
        0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


@pytest.mark.parametrize("name", ["b28_graph_core.npz", "b100_graph_core.npz", "b200_graph_core.npz"])
def test_graph_core(name):
    z = load(name)
    sets, ids = orc.load_bittner(str(z["pickle"]))
    net = orc.net_from_predictor_sets(sets, ids)
    for e in range(int(z["n_traj"])):
        tr = Traj(z, e)
        # op 1 = genRandState: randint(0,1) per node
        ints, dbls = tr.draws(0)
        d = _rd(ints, dbls)
        st = orc.rand_state(net, 1, d)
        assert np.array_equal(st[0], tr.state[0])
        for t in range(1, tr.T):
            ints, dbls = tr.draws(t)
            d = _rd(ints, dbls)
            if tr.op[t] == 0:
                a = int(tr.act[t, 0])
                if a >= 0:
                    st[0, a] ^= 1  # Graph.flipNode
                orc.rollout(net, st, 1, d)
            else:
                orc.rollout(net, st, 1, d, sync=True)
            _check_used(d, ints, dbls)
            assert np.array_equal(st[0], tr.state[t]), (name, e, t)


def test_tt_core():
    z = load("tt40_core.npz")
    net = orc.net_from_pbn_data(pbn_data_from(z))
    tr = Traj(z, 0)
    st = tr.state[0:1].copy()
    for t in range(1, tr.T):
        ints, dbls = tr.draws(t)
        d = _rd(ints, dbls)
        a = int(tr.act[t, 0])
        if a >= 0:
            st[0, a] ^= 1  # PBN.flip
        orc.rollout(net, st, 1, d)
        _check_used(d, ints, dbls)
        assert np.array_equal(st[0], tr.state[t]), t


def _run_env_trace(net, env, tr, K, reset_kind=True):
    n = net.n
    st = np.zeros((1, n), np.uint8)
    n_steps = np.zeros(1, np.int32)
    tatt = np.zeros(1, np.int32)
    for t in range(tr.T):
        ints, dbls = tr.draws(t)
        d = _rd(ints, dbls)
        if tr.op[t] == 1:
            orc.env_reset(net, env, st, n_steps, tatt, d)
            _check_used(d, ints, dbls)
            assert np.array_equal(st[0], tr.state[t]), ("reset", t)
            if tr.target_att[t] >= 0:
                assert tatt[0] == tr.target_att[t]
        else:
            obs, rew, term, trunc, inner = orc.env_step(net, env, st, n_steps, tatt, tr.act[t:t + 1, :K], d)
            _check_used(d, ints, dbls)
            assert np.array_equal(st[0], tr.state[t]), ("state", t)
            assert np.array_equal(obs[0], tr.obs[t]), ("obs", t)
            assert (rew[0], term[0], trunc[0]) == (tr.reward[t], tr.term[t], tr.trunc[t]), ("reward", t)


def test_pbn_env_ex5():
    z = load("ex5_pbnenv.npz")
    net = orc.net_from_pbn_data(pbn_data_from(z))
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = orc.Env(orc.ENV_PBN, 5, attractors=atts, targets=[tuple(t) for t in z["targets"]])
    for e in range(int(z["n_traj"])):
        _run_env_trace(net, env, Traj(z, e), 1)


def test_pbcn_and_sampled_data_ex5():
    z = load("ex5_pbcn_sampled.npz")
    net = orc.net_from_pbn_data(pbn_data_from(z))
    kinds = [orc.ENV_PBCN, orc.ENV_PBCN_SD, orc.ENV_PBN_SD]
    for e, kind in enumerate(kinds):
        atts = cubes_to_attractors(z[f"e{e}/att_cubes"], z[f"e{e}/att_off"])
        env = orc.Env(kind, 5, attractors=atts, targets=[tuple(t) for t in z["targets"]],
                      n_control=int(z[f"e{e}/M"]), successful_reward=int(z[f"e{e}/successful_reward"]),
                      wrong_attractor_cost=int(z[f"e{e}/wrong_attractor_cost"]))
        _run_env_trace(net, env, Traj(z, e), 1 if e == 0 else 2)


@pytest.mark.parametrize("fname", ["b28_target_env.npz", "b100_target_env.npz"])
def test_target_env(fname):
    z = load(fname)
    sets, ids = orc.load_bittner(str(z["pickle"]))
    net = orc.net_from_predictor_sets(sets, ids)
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    for e in range(int(z["n_traj"])):
        env = orc.Env(orc.ENV_TARGET, net.n, attractors=atts, horizon=int(z["horizon"]), max_inner=int(z["cap"]),
                      force=int(z[f"e{e}/force"]))
        _run_env_trace(net, env, Traj(z, e), 1)


@pytest.mark.parametrize("fname", ["b28_multi_env.npz", "b100_multi_env.npz"])
def test_multi_env(fname):
    z = load(fname)
    sets, ids = orc.load_bittner(str(z["pickle"]))
    net = orc.net_from_predictor_sets(sets, ids)
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    for e in range(int(z["n_traj"])):
        env = orc.Env(orc.ENV_MULTI, net.n, attractors=atts, horizon=int(z["horizon"]), max_inner=int(z["cap"]),
                      dedup=int(z[f"e{e}/dedup"]))
        _run_env_trace(net, env, Traj(z, e), 3)


def test_ssd_replay_b100():
    z = load("b100_ssd_replay.npz")
    sets, ids = orc.load_bittner(str(z["pickle"]))
    net = orc.net_from_predictor_sets(sets, ids)
    env = orc.Env(orc.ENV_TARGET, net.n)  # all-attracting fixture: one update per iteration
    st = z["init"].copy()
    d = orc.Draws(ints=z["ints"], dbls=z["dbls"])
    hist = orc.ssd(net, env, st, int(z["iters"]), float(z["p"]), z["tgt_nodes"], d)
    assert np.array_equal(hist.astype(np.int64), z["hist"].sum(0))
    assert np.array_equal(d.used[:, 0], [z["ints"].shape[1]] * 2) and np.array_equal(d.used[:, 1], [z["dbls"].shape[1]] * 2)


def test_ssd_policy_branch_b28():
    """The `model` branch of _ssd_run (utils/eval.py:97-101): histogram -> model.predict -> env.step(action)."""
    z = load("b28_ssd_policy.npz")
    sets, ids = orc.load_bittner(str(z["pickle"]))
    net = orc.net_from_predictor_sets(sets, ids)
    atts = cubes_to_attractors(z["att_cubes"], z["att_off"])
    env = orc.Env(orc.ENV_TARGET, net.n, attractors=atts, horizon=10**9, max_inner=int(z["cap"]))
    st = z["init"].reshape(1, -1).copy()
    n_steps, tatt = np.zeros(1, np.int32), np.array([int(z["target_att"])], np.int32)
    tgt = z["tgt_nodes"]
    hist = np.zeros(1 << len(tgt), np.int64)
    for t, a in enumerate(z["actions"]):
        hist[int("".join(str(int(st[0, i])) for i in tgt), 2)] += 1
        # the policy's decision is a function of the state: first target gene that is 0
        zeros = [i for i in tgt if st[0, i] == 0]
        assert a == (zeros[0] + 1 if zeros else 0)
        d = _rd(z["ints"][z["int_off"][t]:z["int_off"][t + 1]], z["dbls"][z["dbl_off"][t]:z["dbl_off"][t + 1]])
        orc.env_step(net, env, st, n_steps, tatt, np.array([[a]], np.int32), d)
    assert np.array_equal(hist, z["hist"]) and np.array_equal(st[0], z["final"])


@pytest.mark.parametrize("tag", ["pbn", "pbcn"])
def test_oracle_self_triggering_envs(tag):
    """orc_env_step_f64 (PB(C)NSelfTriggeringEnv.step) against traces recorded from the reference
    (oracle/make_st_golden.py): observation, discounted float64 reward bit for bit, terminated, interval, draws consumed."""
    z = load("ex5_self_triggering.npz")
    ex5 = load("ex5_pbnenv.npz")
    pbn_data = [(m, t, f"n{i}", False) for i, (m, t) in enumerate(pbn_data_from(ex5))]
    net = orc.net_from_pbn_data(pbn_data)
    atts = [[(0, 0, 1, 0, 0)], [(0, 0, 0, 0, 1)]]
    kind = orc.ENV_PBN_ST if tag == "pbn" else orc.ENV_PBCN_ST
    env = orc.Env(kind, 5, attractors=atts, targets=[(0, 0, 0, 0, 1)], n_control=1, successful_reward=1, wrong_attractor_cost=1,
                  gamma=0.9, max_interval=5 if tag == "pbn" else 7)
    for k in range(len(z[f"{tag}_interval"])):
        n = int(z[f"{tag}_interval"][k])
        st = z[f"{tag}_start"][k:k + 1].copy()
        a0, a1 = (int(v) for v in z[f"{tag}_action"][k])
        act = [a0, a1] if tag == "pbn" else [a1, a0]
        d = orc.Draws(ints=z[f"{tag}_ints"][k:k + 1, :n], dbls=z[f"{tag}_dbls"][k:k + 1, :2 * n])
        obs, rf, term, inner = orc.env_step_f64(net, env, st, np.array([act], np.int32), d)
        assert int(inner[0]) == n and tuple(d.used[0]) == (n, 2 * n), k
        assert np.array_equal(obs[0], z[f"{tag}_obs"][k]) and bool(term[0]) == bool(z[f"{tag}_term"][k]), k
        assert rf[0] == z[f"{tag}_reward"][k], (k, rf[0], z[f"{tag}_reward"][k])


def test_curriculum_restatements_match_numpy_and_the_reference_arithmetic():
    """pbn_target_multi.py:232-235 — np.random.choice(range(A), size=2, replace=False, p) restated from its uniforms, checked
    against NumPy's own legacy generator (third-party arithmetic not under /root/reference, SURVEY.md §8c(i)); and
    rework_probas (:159-181) against the same float64 expressions written out in Python, the language of the reference."""
    rng = np.random.default_rng(0)
    for _ in range(2000):
        A = int(rng.integers(2, 9))
        p = rng.random(A)
        p[rng.random(A) < 0.2] *= 1e-3
        p /= p.sum()
        seed = int(rng.integers(0, 2**31))
        np.random.seed(seed)
        want = tuple(int(v) for v in np.random.choice(range(A), size=2, replace=False, p=p))
        np.random.seed(seed)
        u = list(np.random.random_sample(2)) + list(np.random.random_sample(1)) + list(np.random.random_sample(1))
        got, used = orc.sample_pair(p, u)
        assert got == want and used in (2, 3)

    def reference_rework(prob, s, t, episode_len):  # the reference's statements, one for one
        A = len(prob)
        proba_eps = 1 * 1 / A
        min_prob = 0.01 * 1 / A
        max_prob = 0.5
        if episode_len < 20:
            prob[s] -= proba_eps
            prob[t] -= proba_eps
            prob[s] = max(prob[s], min_prob)
            prob[t] = max(prob[t], min_prob)
        if episode_len >= 99:
            prob[s] += proba_eps
            prob[t] += proba_eps
            prob[s] = min(prob[s], max_prob)
            prob[t] = min(prob[t], max_prob)
        for i in range(len(prob)):
            prob[i] = max(min_prob, prob[i])
        total = sum(prob)
        for i in range(len(prob)):
            prob[i] /= total
        return prob

    for A in (2, 3, 7, 12):
        mine, ref = np.full(A, 1.0 / A), [1.0 / A] * A
        for _ in range(300):
            s, t = (int(v) for v in rng.choice(A, 2, replace=False))
            ln = int(rng.choice([3, 19, 20, 50, 98, 99, 100]))
            orc.rework_probas(mine, s, t, ln)
            ref = reference_rework(ref, s, t, ln)
            assert mine.tolist() == ref  # bit for bit
