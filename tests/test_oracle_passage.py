"""CPU: the oracle's first-passage loop (orc_first_passage) against the pinned oracle it restates, and against the exact
first-passage law of small networks; and the host side of gym_PBN.utils.control's passage measure (goal words, ranking)."""
import numpy as np
import pytest

import edge_pin_oracle as eo
import oracle as orc
import passage_oracle as pao
from edge_pin_util import edge_rows, edges_of
from golden_util import random_predictor_sets, random_tt_data
from passage_util import exact_passage


def _bucket(st, tgt):
    b = np.zeros(st.shape[:-1], np.int64)
    for i in tgt:
        b = b * 2 + st[..., i]
    return b


@pytest.mark.parametrize("kind", ["pred", "tt"])
def test_oracle_is_the_pinned_oracle_stopped(kind):
    """Each chain's time is the first t at which orc_ssd_pinned_edges run for t iterations (same starts and draws) ends in
    a goal pattern, -1 when none of t = 0..T-1 does; 40 chains (a partial group), T = 50, node and edge pins."""
    if kind == "pred":
        sets, ids = random_predictor_sets(20, 3, seed=20)
        onet = orc.net_from_predictor_sets(sets, ids)
    else:
        onet = orc.net_from_pbn_data(random_tt_data(40, seed=3))
    chains, T, p, seed, env0 = 40, 50, 0.05, 8, 32
    tgt = np.array([1, 3, 4, 6], np.int32)
    goal = [0b0110]
    es = edges_of(onet)
    pins = [{}, {4: 1}, {7: 0, 11: 1}]
    edges = edge_rows([[], [es[3] + (1,)], [es[10] + (0,), es[20] + (1,)]])
    start = orc.rand_state(onet, chains, orc.Draws(seed=seed, epoch=0), env0=env0)
    got, _ = pao.first_passage(onet, start, T, p, pins, tgt, goal, orc.Draws(seed=seed, epoch=1), env0=env0, edges=edges)
    want = np.full((len(pins), chains), -1, np.int64)
    for t in range(T - 1, -1, -1):
        _, st = eo.ssd_pinned(onet, start, t, p, pins, tgt, orc.Draws(seed=seed, epoch=1), env0=env0, edges=edges)
        want[np.isin(_bucket(st, tgt), goal)] = t
    assert np.array_equal(got, want)
    assert ((got >= 0).mean(1) > 0.1).all() and ((got >= 0).mean(1) < 0.9).all()  # some chains arrive, some do not


def test_oracle_chunks_and_arrived_chains():
    """Two calls carrying t0 and t_hit give the one-call times; chains that arrived keep their entry and their state."""
    onet = orc.net_from_predictor_sets(*random_predictor_sets(20, 3, seed=20))
    tgt, goal, pins = np.array([2, 5, 9], np.int32), [0b101], [{}, {4: 1}]
    start = orc.rand_state(onet, 70, orc.Draws(seed=1, epoch=0))
    one, _ = pao.first_passage(onet, start, 60, 0.05, pins, tgt, goal, orc.Draws(seed=1, epoch=1))
    h1, s1 = pao.first_passage(onet, start, 30, 0.05, pins, tgt, goal, orc.Draws(seed=1, epoch=1))
    h2, s2 = pao.first_passage(onet, s1, 30, 0.05, pins, tgt, goal, orc.Draws(seed=1, epoch=2), t0=30, t_hit=h1)
    assert np.array_equal(h2[h1 >= 0], h1[h1 >= 0]) and np.array_equal(s2[h1 >= 0], s1[h1 >= 0])
    assert np.array_equal(h2 >= 0, (h1 >= 0) | (h2 >= 30))
    assert np.array_equal(np.where(one < 30, one, -1), h1)  # the first chunk is the same run


@pytest.mark.parametrize("kind", ["pred", "tt"])
def test_exact_law(kind):
    """8-node networks with a node pin and an edge pin, uniform starts: the oracle's P(tau < T) and restricted mean
    E[min(tau, T)] lie within 5 standard errors of the exact values (chains are independent: the perturbation positions of
    a group are an i.i.d. renewal process)."""
    if kind == "tt":
        onet = orc.net_from_pbn_data(random_tt_data(8, seed=12))
        pin, edges = {2: 1}, {(5, 1): 1}
    else:
        onet = orc.net_from_predictor_sets(*random_predictor_sets(8, 3, seed=5))
        pin, edges = {3: 0}, {(1, 7): 1}
    assert all(e in edges_of(onet) for e in edges)
    p, T, chains = 0.05, 20, 32768
    tgt, goal = np.array([1, 4, 6], np.int32), [0b111]
    reached, mean = exact_passage(onet, pin, edges, p, tgt, goal, T)
    assert 0.1 < reached < 0.9
    start = orc.rand_state(onet, chains, orc.Draws(seed=3, epoch=0))
    rows = edge_rows([[(s, d, c) for (s, d), c in edges.items()]])
    t, _ = pao.first_passage(onet, start, T, p, [pin], tgt, goal, orc.Draws(seed=3, epoch=1), edges=rows)
    r = (t[0] >= 0).astype(np.float64)
    m = np.where(t[0] >= 0, t[0], T).astype(np.float64)
    assert abs(r.mean() - reached) <= 5 * r.std(ddof=1) / np.sqrt(chains)
    assert abs(m.mean() - mean) <= 5 * m.std(ddof=1) / np.sqrt(chains)


def test_goal_words():
    pytest.importorskip("torch")
    from gym_PBN.utils.control import goal_words

    w = goal_words([(1, 1), (0, 1)], 2)
    assert w.dtype == np.uint32 and w.tolist() == [0b1010]
    w = goal_words([(1,) * 7, (0, 0, 0, 0, 0, 0, 1)], 7)
    assert w.shape == (4,) and w.tolist() == [0b10, 0, 0, 1 << 31]
    assert goal_words([], 12).shape == (128,) and not goal_words([], 12).any()
    with pytest.raises(ValueError, match="patterns of 2"):
        goal_words([(1, 0, 1)], 2)


def test_passage_ranking_order(monkeypatch):
    """rank_pins(measure="passage") on a hand-made time table: reached, the restricted mean (unreached = iters) and the
    change against row 0, fastest first."""
    pytest.importorskip("torch")
    from gym_PBN.utils import control

    class Env:  # rank_pins needs the network's size and gene ids only
        class network:
            n = 2

    table = np.array([[5, -1, 3, 8],     # unpinned: mean (5 + 10 + 3 + 8) / 4 = 6.5, reached 3/4
                      [0, 0, 0, 0],      # node 0 -> 0: mean 0
                      [-1, -1, -1, -1],  # node 0 -> 1: mean 10, reached 0
                      [12, 2, 4, -1],    # node 1 -> 0: times above iters count as iters: (10 + 2 + 4 + 10) / 4 = 6.5
                      [1, 2, 3, 4]])     # node 1 -> 1: 2.5
    seen = {}

    def fake(env, pins, iters, chains, bit_flip_prob=0.01, seed=0):
        seen.update(pins=pins, iters=iters, chains=chains)
        return {"time": table, "source": None}

    monkeypatch.setattr(control, "first_passage", fake)
    res = control.rank_pins(Env(), iters=10, chains=4, measure="passage")
    assert seen["pins"] == [{}, {0: 0}, {0: 1}, {1: 0}, {1: 1}] and seen["iters"] == 10
    assert res["unpinned"] == {"reached": 0.75, "mean_time": 6.5}
    order = [(r["node"], r["value"]) for r in res["ranking"]]
    assert order == [(0, 0), (1, 1), (1, 0), (0, 1)]
    best = res["ranking"][0]
    assert best["mean_time"] == 0.0 and best["change"] == -6.5 and best["reached"] == 1.0
    assert res["ranking"][2]["change"] == 0.0 and res["ranking"][3]["reached"] == 0.0
    with pytest.raises(ValueError, match="measure"):
        control.rank_pins(Env(), iters=10, chains=4, measure="mass")
