"""GPU: the static SSD loop against the C oracle on synthetic predictor networks whose windows (32 x nodes positions per
iteration) test its position arithmetic: an event's position becomes the iteration it is due in, the state word and the
bit, through a multiply by a reciprocal of the window.  256 nodes is the largest window the loop takes (eight state
words); 20 nodes is one word with fewer than 32 nodes.  p = 0.3 draws many rounds of events per iteration, p = 1e-6
leaves applied events in their slots for thousands of iterations."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402
from golden_util import random_predictor_net  # noqa: E402


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


@pytest.mark.parametrize("n,p", [(256, 0.3), (256, 0.01), (256, 1e-6), (20, 0.3), (20, 1e-6)])
def test_static_ssd_window_arithmetic_matches_oracle(eng, n, p):
    net, onet = random_predictor_net(eng, n, 5, seed=11)  # at most five predictors per node: one threshold quad
    B, iters, seed = 3000, 401, 99  # an odd count: the pending events go back to the generic loop for the last iteration
    tgt = np.arange(7, dtype=np.int32)  # consecutive targets in one word: the static loop
    sim = eng.engine.Simulator(net, B, seed=seed, env0=64)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0), env0=64)
    hist = sim.ssd(iters, p, tgt)
    ohist = orc.ssd(onet, None, ost, iters, p, tgt, orc.Draws(seed=seed, epoch=1), env0=64)
    assert hist.sum().item() == B * iters
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist)
    assert np.array_equal(sim.unpack().cpu().numpy(), ost)
