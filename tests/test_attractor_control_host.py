"""CPU: value iteration of gym_PBN.utils.control.attractor_policy on hand-made count tables with known answers, and the
premises of the GPU cases in test_gpu_attractor_control.py shown on the host."""
import numpy as np
import pytest

pytest.importorskip("torch")

import control_util as cu  # noqa: E402
from gym_PBN.utils.control import attractor_policy  # noqa: E402


def _counts(rows):
    """{(a, i): {b: count}} -> int64 [A][N+1][A+1] for A = 3 attractors, 3 actions (column 3 = cap)."""
    c = np.zeros((3, 3, 4), np.int64)
    for (a, i), land in rows.items():
        for b, k in land.items():
            c[a, i, b] = k
    return c


def test_horizon_one():
    # from 1: action 1 reaches 0 w.p. 3/4, action 2 w.p. 1/2; from 2: only action 0 reaches 0, w.p. 1/4
    c = _counts({(1, 0): {1: 10}, (1, 1): {0: 3, 2: 1}, (1, 2): {0: 2, 1: 2}, (2, 0): {0: 1, 2: 3}, (2, 1): {2: 5}, (2, 2): {1: 5},
                 (0, 0): {0: 1}, (0, 1): {1: 1}, (0, 2): {2: 1}})
    action, success = attractor_policy(c, target=0, horizon=1)
    assert action.shape == success.shape == (2, 3)
    assert np.allclose(success[0], [1, 0, 0]) and np.allclose(success[1], [1, 0.75, 0.25])
    assert action[1].tolist() == [0, 1, 0]


def test_two_steps_go_through_an_intermediate_attractor():
    # 2 -> 1 surely (action 2), 1 -> 0 w.p. 1/2 (action 1); 2 -> 0 directly w.p. 0.3 (action 1)
    c = _counts({(1, 1): {0: 1, 1: 1}, (2, 1): {0: 3, 2: 7}, (2, 2): {1: 4}, (1, 0): {1: 1}, (1, 2): {1: 1}, (2, 0): {2: 1}})
    action, success = attractor_policy(c, target=0, horizon=2)
    assert np.allclose(success[1], [1, 0.5, 0.3]) and action[1].tolist() == [0, 1, 1]
    # two steps left in 2: direct (0.3 + 0.7 * 0.3 = 0.51) beats the detour (1 * 0.5)
    assert np.isclose(success[2, 2], 0.51) and action[2, 2] == 1
    assert np.isclose(success[2, 1], 0.75) and action[2, 1] == 1


def test_unreachable_target():
    c = _counts({(a, i): {a: 5} for a in (1, 2) for i in range(3)} | {(1, 1): {2: 5}, (2, 2): {1: 5}})
    action, success = attractor_policy(c, target=0, horizon=4)
    assert np.allclose(success[:, 1:], 0) and (success[:, 0] == 1).all()
    assert (action == 0).all()  # every action ties at 0: the lowest index


def test_cap_column_is_failure():
    # action 1 lands in 0 on half of its steps and hits the cap on the rest; action 2 never hits the cap but lands in 0
    # only w.p. 0.4 and stays in 1 otherwise
    c = _counts({(1, 1): {0: 50, 3: 50}, (1, 2): {0: 40, 1: 60}, (2, 0): {2: 1}})
    _, success = attractor_policy(c, target=0, horizon=1)
    assert np.isclose(success[1, 1], 0.5)
    action, success = attractor_policy(c, target=0, horizon=2)
    assert np.isclose(success[2, 1], 0.4 + 0.6 * 0.5) and action[2, 1] == 2 and action[1, 1] == 1


def test_ties_go_to_the_lowest_action():
    c = _counts({(1, 0): {1: 3}, (1, 1): {0: 1, 2: 1}, (1, 2): {0: 2, 1: 2}, (2, 1): {0: 7}, (2, 2): {0: 7}})
    action, success = attractor_policy(c, target=0, horizon=1)
    assert action[1].tolist() == [0, 1, 1] and np.allclose(success[1], [1, 0.5, 1])


def test_argument_errors():
    c = _counts({})
    with pytest.raises(ValueError):
        attractor_policy(c[:, :, :3], 0, 1)
    with pytest.raises(ValueError):
        attractor_policy(c, 3, 1)
    with pytest.raises(ValueError):
        attractor_policy(c, 0, -1)
    with pytest.raises(ValueError):
        attractor_policy(-1 - c, 0, 1)


def test_value_iteration_equals_exhaustive_search():
    rng = np.random.default_rng(3)
    c = rng.integers(0, 20, size=(3, 4, 4))
    c[..., 3] = rng.integers(0, 5, size=(3, 4))
    P = c / c.sum(2, keepdims=True)
    for H in (1, 2, 3):
        _, success = attractor_policy(c, target=2, horizon=H)
        assert np.isclose(success[H].mean(), cu.markov_optimum(P, 2, H))
        assert cu.stationary_optimum(P, 2, H) <= success[H].mean() + 1e-12


# ------------------------------------------------------------------------------------------------ premises of the GPU cases
def test_fixed_point_network_has_only_fixed_point_attractors():
    data, atts = cu.fixed_point_net()
    sccs = cu.terminal_sccs(cu.transition_matrix(data))
    assert len(sccs) == len(atts) == 3 and all(len(a) == 1 for a in sccs)
    T = cu.transition_matrix(data)
    for (s,) in sccs:
        assert T[s, s] == 1.0  # no update moves a fixed point
    P = cu.exact_landing(T, atts, 6)
    assert np.allclose(P.sum(2), 1) and (P[..., 3] == 0).all()
    opt = [cu.markov_optimum(P, 0, H) for H in (1, 2, 3)]
    assert 0.5 < opt[0] < opt[1] < opt[2] < 0.97  # a case where the horizon matters and success is not certain


def test_ground_truth_network_premise():
    data, atts = cu.ground_truth_net()
    assert len(data) <= 10 and len(atts) >= 3
    assert any("*" in c for a in atts for c in a)  # the reset draws wildcard bits
    P = cu.exact_landing(cu.transition_matrix(data), atts, len(data))
    assert np.allclose(P.sum(2), 1) and (P[..., -1] == 0).all()
    assert ((P[..., :-1] > 0) & (P[..., :-1] < 1)).any()


@pytest.mark.parametrize("name", sorted(cu.CAP_CASES))
def test_cap_cases_hit_the_cap_in_the_oracle(name):
    counts = cu.oracle_transitions(name, cu.CAP_SAMPLES[name], cu.CAP_SEED)
    A = counts.shape[0]
    assert counts.sum(2).min() >= cu.CAP_SAMPLES[name]
    assert counts[..., A].sum() > 0 and counts[..., :A].sum() > 0  # column A is non-empty, and steps also land
    if name == "b28":
        assert cu.CAP_CASES[name] > 8192  # Simulator.env_step plans a first pass and a resume pass above 8192 envs
