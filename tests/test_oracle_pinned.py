"""CPU: the oracle's pinned SSD (orc_ssd_pinned) — without pins it is orc_ssd, pinned nodes hold, and on a small network its
estimate converges to the exact stationary law of the pinned, perturbed chain."""
import numpy as np
import pytest

import oracle as orc
import pinned_oracle as po
from golden_util import random_tt_data
from pinned_util import exact_pinned_law


def _net(which):
    if which == "tt":
        return orc.net_from_pbn_data(random_tt_data(40, seed=3))
    return orc.net_from_predictor_sets(*orc.load_bittner(which))


@pytest.mark.parametrize("which", ["28_15_median", "tt"])
@pytest.mark.parametrize("p", [0.3, 0.01, 0.0])
def test_no_pins_is_orc_ssd(which, p):
    onet = _net(which)
    chains, iters, seed, env0 = 45, 37, 4, 64
    tgt = np.array([2, 9, 5], np.int32)
    st = orc.rand_state(onet, chains, orc.Draws(seed=seed, epoch=0), env0=env0)
    ref = st.copy()
    href = orc.ssd(onet, None, ref, iters, p, tgt, orc.Draws(seed=seed, epoch=1), env0=env0)
    hist, out = po.ssd_pinned(onet, st, iters, p, [{}, {}], tgt, orc.Draws(seed=seed, epoch=1), env0=env0)
    for k in range(2):
        assert np.array_equal(hist[k], href) and np.array_equal(out[k], ref)


@pytest.mark.parametrize("which", ["28_15_median", "tt"])
def test_pinned_nodes_hold(which):
    """p = 0.3: about one perturbation event per node every three iterations, yet no counted state and no final state
    contradicts a pin; a pin outside the targets still moves the histogram."""
    onet = _net(which)
    chains, iters, seed = 70, 300, 8
    tgt = np.array([3, 4, 5, 6], np.int32)
    pins = [{4: 1, 11: 0}, {3: 0, 6: 1, 20: 1}, {11: 1}, {}]
    st = orc.rand_state(onet, chains, orc.Draws(seed=seed, epoch=0))
    hist, out = po.ssd_pinned(onet, st, iters, 0.3, pins, tgt, orc.Draws(seed=seed, epoch=1))
    assert (hist.sum(1) == chains * iters).all()
    for k, pin in enumerate(pins):
        for i, v in pin.items():
            assert (out[k][:, i] == v).all()
            if i in tgt:
                pos = len(tgt) - 1 - list(tgt).index(i)  # first target = most significant bit
                bad = [b for b in range(1 << len(tgt)) if (b >> pos) & 1 != v]
                assert hist[k][bad].sum() == 0
    assert not np.array_equal(hist[2], hist[3])


def test_exact_pinned_law():
    """An 8-node truth-table network with two genes pinned: independent batches of oracle chains (after a burn-in) agree
    with the exact law, within 0.01 in total variation and 5 batch-means standard errors per bucket."""
    data = random_tt_data(8, seed=12)
    onet = orc.net_from_pbn_data(data)
    pin, p, tgt = {2: 1, 5: 0}, 0.05, np.array([1, 2, 4, 7], np.int32)
    exact = exact_pinned_law(data, pin, p, tgt)
    batches = []
    for b in range(16):
        st = orc.rand_state(onet, 64, orc.Draws(seed=b, epoch=0), env0=64 * b)
        _, st = po.ssd_pinned(onet, st, 300, p, [pin], tgt, orc.Draws(seed=b, epoch=1), env0=64 * b)
        h, _ = po.ssd_pinned(onet, st[0], 3000, p, [pin], tgt, orc.Draws(seed=b, epoch=2), env0=64 * b)
        batches.append(h[0] / h[0].sum())
    batches = np.array(batches)
    est, se = batches.mean(0), batches.std(0, ddof=1) / np.sqrt(len(batches))
    assert 0.5 * np.abs(est - exact).sum() < 0.01
    assert (np.abs(est - exact) <= 5 * se + 1e-12).all()
    assert exact[[b for b in range(16) if not (b >> 2) & 1]].sum() < 1e-12  # target 2 is pinned at 1 (bit 2 of the bucket)
