"""GPU: shared-memory capacity of k_ssd with an attractor env.  A launch whose layout needs more dynamic shared memory than a
block may have is refused with PBN_ERR_UNSUPPORTED before anything runs, and the refusal leaves no CUDA error behind for the
next call; a layout just inside the limit runs and matches the oracle bit for bit.

Bittner-100 (4 state words), 7 target genes, p = 0.01: the windowed attractor loop adds the flip masks and the straggler-mode
staging to the image, so an env of one attractor with ~5 600 full cubes passes pbn_env_create but not the SSD launch.  Each
full cube takes 32 bytes of the cube image (w32 * 8), which is how the near-limit case is sized from the refusal message."""
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import oracle as orc  # noqa: E402
from golden_util import hittable_cubes  # noqa: E402

NET, TGT, P, CUBE_BYTES, N_OVER = "100_5_kmeans", np.arange(7, dtype=np.int32), 0.01, 32, 5600


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gym_PBN.b200 import abi, compiler, engine

    class E:
        pass

    e = E()
    e.abi, e.engine = abi, engine
    e.net = engine.Network(compiler.load_bittner(NET))
    sets, ids = orc.load_bittner(NET)
    e.onet = orc.net_from_predictor_sets(sets, ids)
    return e


def _attractor(onet, n_cubes, n_hit=0, seed=5):
    """One attractor: random full states (practically never reached), then n_hit reachable cubes at the END of the list, so
    that a chain stops only after testing every cube before them (the last bytes of the staged cube image)."""
    rng = np.random.default_rng(seed)
    cubes = [tuple(int(v) for v in rng.integers(0, 2, onet.n)) for _ in range(n_cubes - n_hit)]
    return [cubes + (hittable_cubes(onet, n_hit, seed) if n_hit else [])]


def _refusal(eng, n_cubes):
    env = eng.engine.EnvImage(eng.net, eng.abi.ENV_TARGET, attractors=_attractor(eng.onet, n_cubes), max_inner=8)
    sim = eng.engine.Simulator(eng.net, 1024, seed=3)
    sim.rand_state()
    with pytest.raises(eng.abi.PbnError) as err:
        sim.ssd(4, P, TGT, env=env)
    return str(err.value)


def _ssd_matches_oracle(eng, B, iters, env=None, oenv=None, seed=11):
    sim = eng.engine.Simulator(eng.net, B, seed=seed)
    sim.rand_state()
    ost = orc.rand_state(eng.onet, B, orc.Draws(seed=seed, epoch=0))
    hist = sim.ssd(iters, P, TGT, env=env)
    ohist = orc.ssd(eng.onet, oenv, ost, iters, P, TGT, orc.Draws(seed=seed, epoch=1))
    assert hist.sum().item() == B * iters
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist)
    assert np.array_equal(sim.unpack().cpu().numpy(), ost)


def test_ssd_over_the_shared_memory_limit_is_refused_and_leaves_no_error(eng):
    msg = _refusal(eng, N_OVER)
    assert msg.startswith("pbn_b200 error 3: k_ssd needs "), msg  # PBN_ERR_UNSUPPORTED, not a failed CUDA call
    need, avail = map(int, re.search(r"needs (\d+) bytes.*allows (\d+)", msg).groups())
    assert need > avail
    _ssd_matches_oracle(eng, 1024, 50)  # the next call runs: the refusal left no CUDA error to pick up


def test_ssd_within_1kb_of_the_shared_memory_limit_matches_oracle(eng):
    need, avail = map(int, re.search(r"needs (\d+) bytes.*allows (\d+)", _refusal(eng, N_OVER)).groups())
    n_cubes = N_OVER - -(-(need - avail) // CUBE_BYTES)  # the most full cubes that fit
    footprint = need - (N_OVER - n_cubes) * CUBE_BYTES
    assert avail - 1024 < footprint <= avail
    atts = _attractor(eng.onet, n_cubes, n_hit=4)
    env = eng.engine.EnvImage(eng.net, eng.abi.ENV_TARGET, attractors=atts, max_inner=8)
    oenv = orc.Env(orc.ENV_TARGET, eng.onet.n, attractors=atts, max_inner=8)
    _ssd_matches_oracle(eng, 256, 16, env, oenv)
    # one cube more is refused: the case above sits at the limit
    assert "k_ssd needs" in _refusal(eng, n_cubes + 1)
