"""CPU: the oracle's SSD with edges pinned (orc_ssd_pinned_edges) — without edge pins it is the pinned oracle
(orc_ssd_pinned), pinning every out-edge of a node equals the pinned oracle's node pin, and on small networks its estimate
converges to the exact stationary law computed on the gather side; and the regulatory edges of the shipped Bittner sets."""
import numpy as np
import pytest

import edge_pin_oracle as eo
import oracle as orc
import pinned_oracle as po
from edge_pin_util import EMPTY, edge_rows, edges_of, entry, exact_edge_law
from golden_util import random_predictor_sets, random_tt_data


def _net(which):
    if which == "tt":
        return orc.net_from_pbn_data(random_tt_data(40, seed=3))
    return orc.net_from_predictor_sets(*orc.load_bittner(which))


@pytest.mark.parametrize("which", ["28_15_median", "tt"])
@pytest.mark.parametrize("p", [0.3, 0.01, 0.0])
def test_no_edges_is_the_pinned_oracle(which, p):
    """No edge slots, empty slots, and entries that name no edge (dst not below N, src not an input of dst) all give the
    pinned oracle's output, bit for bit."""
    onet = _net(which)
    chains, iters, seed, env0 = 45, 37, 4, 64
    tgt = np.array([2, 9, 5], np.int32)
    pins = [{}, {4: 1, 11: 0}, {2: 0, 20: 1}]
    non_edge = next((s, 7) for s in range(onet.n) if (s, 7) not in edges_of(onet))
    rows = [None, edge_rows([[], [], []], E=5), edge_rows([[entry(3, onet.n, 1), non_edge + (1,), EMPTY]] * 3)]
    st = orc.rand_state(onet, chains, orc.Draws(seed=seed, epoch=0), env0=env0)
    ref_h, ref_out = po.ssd_pinned(onet, st, iters, p, pins, tgt, orc.Draws(seed=seed, epoch=1), env0=env0)
    for edges in rows:
        h, out = eo.ssd_pinned(onet, st, iters, p, pins, tgt, orc.Draws(seed=seed, epoch=1), env0=env0, edges=edges)
        assert np.array_equal(h, ref_h) and np.array_equal(out, ref_out)


def out_edge_variant(onet, u, c):
    return [(u, v, c) for s, v in edges_of(onet) if s == u and v != u]


@pytest.mark.parametrize("which", ["28_15_median", "tt"])
@pytest.mark.parametrize("p", [0.3, 0.01, 0.0])
def test_out_edges_equal_the_node_pin(which, p):
    """For a node u outside the targets, pinning every out-edge (u, v), v != u, at c gives the histogram of the node pin
    {u: c} bit for bit: every other node reads c in both, and u's update and perturbation draws are consumed alike.  The
    final states differ in u's bit only."""
    onet = _net(which)
    chains, iters, seed = 70, 200, 6
    tgt = np.array([3, 4, 5, 6], np.int32)
    outdeg = {u: len(out_edge_variant(onet, u, 0)) for u in range(onet.n) if u not in tgt}
    busiest = sorted((u for u in outdeg if outdeg[u] <= 64), key=lambda u: -outdeg[u])
    for u, c in ((busiest[0], 1), (busiest[1], 0)):
        edges = out_edge_variant(onet, u, c)
        st = orc.rand_state(onet, chains, orc.Draws(seed=seed, epoch=0))
        hn, sn = po.ssd_pinned(onet, st, iters, p, [{u: c}], tgt, orc.Draws(seed=seed, epoch=1))
        he, se = eo.ssd_pinned(onet, st, iters, p, [{}], tgt, orc.Draws(seed=seed, epoch=1), edges=edge_rows([edges]))
        assert np.array_equal(hn, he)
        others = np.arange(onet.n) != u
        assert np.array_equal(sn[..., others], se[..., others])
        assert (sn[..., u] == c).all() and (p == 0 or not (se[..., u] == c).all())


def _exact_net(kind):
    if kind == "tt":
        return orc.net_from_pbn_data(random_tt_data(8, seed=12))
    return orc.net_from_predictor_sets(*random_predictor_sets(8, 3, seed=5))


def exact_cases():
    """(kind, edge pins): on an 8-node predictor and an 8-node truth-table network, the single edge pin that moves the exact
    law most, and that pin with a second one (the predictor network's: a self-input)."""
    out = []
    for kind in ("pred", "tt"):
        onet = _exact_net(kind)
        p, tgt = 0.05, np.array([1, 4, 6, 7], np.int32)
        base = exact_edge_law(onet, {}, p, tgt)
        moved = sorted(((e, c) for e in edges_of(onet) for c in (0, 1)),
                       key=lambda ec: -np.abs(exact_edge_law(onet, {ec[0]: ec[1]}, p, tgt) - base).sum())
        (e0, c0), second = moved[0], next(ec for ec in moved if ec[0][1] != moved[0][0][1] and (kind == "tt" or ec[0][0] == ec[0][1]))
        out += [(kind, {e0: c0}), (kind, {e0: c0, second[0]: second[1]})]
    return out


@pytest.mark.parametrize("kind,edges", exact_cases())
def test_exact_edge_law(kind, edges):
    """Independent batches of oracle chains (after a burn-in) agree with the exact law, within 0.01 in total variation and
    5 batch-means standard errors per bucket."""
    onet = _exact_net(kind)
    p, tgt = 0.05, np.array([1, 4, 6, 7], np.int32)
    exact = exact_edge_law(onet, edges, p, tgt)
    assert 0.5 * np.abs(exact - exact_edge_law(onet, {}, p, tgt)).sum() > 0.02  # the pins move the law
    rows = edge_rows([[(s, d, c) for (s, d), c in edges.items()]])
    batches = []
    for b in range(16):
        st = orc.rand_state(onet, 64, orc.Draws(seed=b, epoch=0), env0=64 * b)
        _, st = eo.ssd_pinned(onet, st, 300, p, [{}], tgt, orc.Draws(seed=b, epoch=1), env0=64 * b, edges=rows)
        h, _ = eo.ssd_pinned(onet, st[0], 3000, p, [{}], tgt, orc.Draws(seed=b, epoch=2), env0=64 * b, edges=rows)
        batches.append(h[0] / h[0].sum())
    batches = np.array(batches)
    est, se = batches.mean(0), batches.std(0, ddof=1) / np.sqrt(len(batches))
    assert 0.5 * np.abs(est - exact).sum() < 0.01
    assert (np.abs(est - exact) <= 5 * se + 1e-12).all()


@pytest.mark.parametrize("name,n,edges,self_inputs", [("28_15_median", 28, 420, 28), ("100_5_kmeans", 100, 960, 100),
                                                      ("200_5_kmeans", 199, 1950, 199)])
def test_regulatory_edges_of_bittner_sets(name, n, edges, self_inputs):
    from gym_PBN.b200 import compiler
    from gym_PBN.utils import control

    spec = compiler.load_bittner(name)
    got = control.regulatory_edges(spec)
    assert spec.n == n and len(got) == edges == len(set(got))
    assert sum(s == d for s, d in got) == self_inputs
    assert got == edges_of(orc.net_from_predictor_sets(*orc.load_bittner(name)))
    assert [d for _, d in got] == sorted(d for _, d in got)  # (dst, slot) order
