"""GPU: the step-until-attractor kernels (k_env_step_first, k_env_step_att, the windowed attractor loop of k_ssd) against the
oracle on every instantiation the dispatch picks: threshold layouts (one quad, leading quad + quads, flat rows), state widths
of 1..32 words, predictor records above and below 32 KB, truth-table networks, and attractor lists long enough that lane
groups test cubes beyond their first two (the EXTRA branch of pbn_coop.cuh).  Everything here is bit-exact.

The product reports nothing about which branch ran, so every case proves its premise from the oracle's outputs instead:
test_cases_reach_their_regime (CPU only) checks the network's width and threshold class, that some envs stop inside the loop
and some at the cap, and that some stop on a cube which only the intended branch tests."""
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

import oracle as orc  # noqa: E402
from golden_util import attractor_fixture, random_predictor_sets, random_tt_data, synthetic_pbcn  # noqa: E402

# name: (kind, n, max predictors per node) -> what the dispatch makes of it (threshold quads TQ, lockstep first pass):
#   p30q   w32 1, one quad          first<1,true>       att<PRED,PHILOX,1,true>
#   p32t   w32 1, lead + 2 quads    first<0,false>      att<…,0,true>   (two-level rows read at run time; node 31 = top bit)
#   p30f   w32 1, flat rows         first<0,false>      att<…,0,true>
#   p33q   w32 2, one quad          first<1,true>       att<…,1,false>  (one live bit in word 2)
#   p65t   w32 3, lead + 3 quads    first<0,false>      att<…,0,false>  (two-level at run time)
#   p100t  w32 4, lead + 4 quads    first<4,true>       att<…,4,false>
#   p200t  w32 7, lead + 4 quads    first<4,false>      att<…,4,false>  (records 200 x 14 x 16 B > 32 KB)
#   p100f  w32 4, flat rows         first<0,false>      att<…,0,false>  (records 100 x 23 x 16 B > 32 KB)
#   p256q  w32 8, one quad          first<1,true>       att<…,1,false>  (the widest predictor state)
#   tt31, tt70, tt1024              no first pass       att<TT,PHILOX,0,false> in lane mode (tt1024: threshold table in
#                                                        global memory)
NETS = {"p30q": ("pred", 30, 5), "p32t": ("pred", 32, 9), "p30f": ("pred", 30, 23), "p33q": ("pred", 33, 3),
        "p65t": ("pred", 65, 11), "p100t": ("pred", 100, 16), "p200t": ("pred", 200, 14), "p100f": ("pred", 100, 23),
        "p256q": ("pred", 256, 5), "tt31": ("tt", 31, 0), "tt70": ("tt", 70, 0), "tt1024": ("pbcn", 1024, 0)}
# (w32, threshold class, records above 32 KB) each network must have
SHAPE = {"p30q": (1, "quad", False), "p32t": (1, "two-level", False), "p30f": (1, "flat", False), "p33q": (2, "quad", False),
         "p65t": (3, "two-level", False), "p100t": (4, "two-level", False), "p200t": (7, "two-level", True),
         "p100f": (4, "flat", True), "p256q": (8, "quad", False), "tt31": (1, None, None), "tt70": (3, None, None),
         "tt1024": (32, None, None)}
# step plans: one launch; odd budgets (a resume pass starts at an odd update); the default-like (32, 256) split
PLANS = {"one": (), "odd": (2, 7, 0), "wide": (32, 256, 0)}
# a hit at cube index >= THRESH[fixture] can only be seen by the branch the fixture is there for (golden_util.FIXTURE_HITS)
THRESH = {1: 0, 2: 1, 7: 4, 14: 8, 72: 64}


def _seed(name):
    return sum(map(ord, name))


@functools.lru_cache(maxsize=None)
def _ref(name):
    """Reference form of a network: ("pred", sets, ids) or ("tt", pbn_data)."""
    kind, n, fmax = NETS[name]
    if kind == "pred":
        return ("pred",) + random_predictor_sets(n, fmax, seed=_seed(name))
    return ("tt", random_tt_data(n, seed=_seed(name)) if kind == "tt" else synthetic_pbcn(n=n, m=8, seed=3))


@functools.lru_cache(maxsize=None)
def _onet(name):
    r = _ref(name)
    return orc.net_from_predictor_sets(r[1], r[2]) if r[0] == "pred" else orc.net_from_pbn_data(r[1])


@functools.lru_cache(maxsize=None)
def _atts(name, n_cubes):
    return attractor_fixture(_onet(name), n_cubes, seed=_seed(name) + n_cubes)


class Case:
    """One env on one network with one fixture, stepped len(plans) times; the oracle's trajectory computed once per session
    and shared by the GPU test and the regime test."""

    def __init__(self, name, n_cubes, kind, plans=("one", "odd", "wide"), cap=300, B=2500, horizon=2):
        self.name, self.n_cubes, self.kind, self.plans, self.cap, self.B, self.horizon = name, n_cubes, kind, plans, cap, B, horizon
        self.multi = kind.startswith("multi")
        self.force = kind == "target_force"
        self.dedup = kind != "multi_list"
        self.seed = _seed(name) + 7 * n_cubes + cap + len(kind)

    @property
    def id(self):
        return f"{self.name}-{self.n_cubes}-{self.kind}-{'.'.join(self.plans)}-cap{self.cap}-B{self.B}"

    def env_kw(self):
        return dict(attractors=_atts(self.name, self.n_cubes), horizon=self.horizon, max_inner=self.cap, force=self.force,
                    dedup=self.dedup)

    @property
    def resets(self):  # TARGET's reset draws two different attractors
        return self.multi or len(_atts(self.name, self.n_cubes)) >= 2

    @functools.cached_property
    def traj(self):
        onet, n, B = _onet(self.name), _onet(self.name).n, self.B
        kw = self.env_kw()
        oenv = orc.Env(orc.ENV_MULTI if self.multi else orc.ENV_TARGET, n, attractors=kw["attractors"], horizon=self.horizon,
                       max_inner=self.cap, force=int(self.force), dedup=int(self.dedup))
        rng = np.random.default_rng(self.seed)
        ost, ons, ota = np.zeros((B, n), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
        out = {"st0": None, "reset0": None, "steps": []}
        epoch = 0
        if self.resets:
            orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=self.seed, epoch=epoch))
            epoch += 1
            out["reset0"] = (ost.copy(), ons.copy(), ota.copy())
        else:  # a single attractor: start from random states, target attractor 0
            ost[:] = rng.integers(0, 2, size=(B, n))
            if onet.first:
                ost[:, : onet.first] = 0
            out["st0"] = ost.copy()
        for t in range(len(self.plans)):
            if self.multi:
                act = rng.integers(0, n + 1, size=(B, 3)).astype(np.int32)
                dup = rng.random(B) < 0.3
                act[dup, 2] = act[dup, 0]
                act[rng.random(B) < 0.1, 1] = -1  # an empty slot
            else:
                act = rng.integers(0, n + 1, size=(B, 1)).astype(np.int32)
            ta = ota.copy()
            obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=self.seed, epoch=epoch))
            epoch += 1
            step = dict(act=act, ta=ta, obs=obs, rew=rew, term=term, trunc=trunc, inner=inner, state=ost.copy(), n_steps=ons.copy())
            if self.resets:
                done = (term | trunc).astype(np.uint8)
                orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=self.seed, epoch=epoch), mask=done)
                epoch += 1
                step.update(done=done, reset=(ost.copy(), ons.copy(), ota.copy()))
            out["steps"].append(step)
        return out


CASES = [Case(name, 72, kind, B=(2500 if i % 2 else 3072) if name != "tt1024" else 2048)
         for i, name in enumerate(NETS) for kind in ("target", "multi", "multi_list")]
CASES += [Case("p100t", 72, "target_force", plans=("one", "one"))]
CASES += [Case(name, 72, kind, cap=cap) for name, kind in (("p65t", "target"), ("p256q", "multi")) for cap in (64, 65)]
PLACEMENTS = [Case(name, nc, kind) for name in ("p30f", "p100t") for nc in (1, 2, 7, 14) for kind in ("target", "multi")]


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gym_PBN.b200 import abi, compiler, engine

    class E:
        pass

    e = E()
    e.abi, e.compiler, e.engine = abi, compiler, engine
    e.nets = {}
    return e


def _net(eng, name):
    if name not in eng.nets:
        r = _ref(name)
        spec = eng.compiler.compile_predictor_sets(r[1], r[2]) if r[0] == "pred" else eng.compiler.compile_pbn_data(r[1])
        eng.nets[name] = eng.engine.Network(spec)
    return eng.nets[name]


def _np(t):
    return t.cpu().numpy()


def _run(eng, case):
    tr = case.traj
    net = _net(eng, case.name)
    env = eng.engine.EnvImage(net, eng.abi.ENV_MULTI if case.multi else eng.abi.ENV_TARGET, **case.env_kw())
    sim = eng.engine.Simulator(net, case.B, seed=case.seed)
    sim.plan_budgets = ()
    if case.resets:
        sim.env_reset(env)
        st, ns, ta = tr["reset0"]
        assert np.array_equal(_np(sim.unpack()), st) and np.array_equal(_np(sim.target_att), ta)
    else:
        sim.set_state(tr["st0"])
    for t, (plan, s) in enumerate(zip(case.plans, tr["steps"])):
        act = torch.from_numpy(s["act"])
        budgets = PLANS[plan]
        if budgets:
            sim.env_step(env, act, budget=budgets[0])
            parked = int(sim.running.sum())
            for b in budgets[1:]:
                sim.env_step_resume(env, budget=b)
            assert parked > 0 and int(sim.running.sum()) == 0, (t, parked)  # the split happened and ended
        else:
            sim.env_step(env, act)
        where = (case.id, t)
        assert np.array_equal(_np(sim.unpack()), s["state"]), where
        assert np.array_equal(_np(sim.unpack(sim.obs_state)), s["obs"]), where
        assert np.array_equal(_np(sim.reward), s["rew"]), where
        assert np.array_equal(_np(sim.terminated), s["term"]) and np.array_equal(_np(sim.truncated), s["trunc"]), where
        assert np.array_equal(_np(sim.inner), s["inner"]), where
        assert np.array_equal(_np(sim.n_steps), s["n_steps"]), where
        if case.resets:
            sim.env_reset(env, mask=torch.from_numpy(s["done"]))
            st, ns, ta = s["reset"]
            assert np.array_equal(_np(sim.unpack()), st) and np.array_equal(_np(sim.n_steps), ns), where
            assert np.array_equal(_np(sim.target_att), ta), where


@gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_env_step_matches_oracle(eng, case):
    """Every network with the 72-cube fixture: TARGET, MULTI with duplicate actions (dedup on and off), TARGET force=True on
    one network, caps of 64 (lane mode) and 65 (group mode) on two multi-word networks; one launch and two step plans."""
    _run(eng, case)


@gpu
@pytest.mark.parametrize("case", PLACEMENTS, ids=lambda c: c.id)
def test_cube_placements_match_oracle(eng, case):
    """The hittable cubes at every position that selects another branch of the attractor test (1, 2, 7, 14 cubes; the 72-cube
    fixture is in test_env_step_matches_oracle) on a flat-row one-word and a two-level four-word network."""
    _run(eng, case)


# ------------------------------------------------------------------------------------------------ SSD with an attractor loop
@gpu
@pytest.mark.parametrize("name", ["p30f", "p100t", "p256q", "tt70"])
@pytest.mark.parametrize("B,iters,force", [(1024, 37, False), (1000, 37, False), (1024, 20, True)])
def test_ssd_with_attractor_loop_matches_oracle(eng, name, B, iters, force):
    """k_ssd with a TARGET env and the 72-cube fixture: the windowed loop (flip masks of 16 / w32 iterations, at least 2, drawn
    ahead; lane groups take over a warp's last chains inside the window) with a last window cut short (37 iterations), a
    partial last warp (B = 1000), and force=True (no attractor loop, no window).  Histogram and final states."""
    onet, net = _onet(name), _net(eng, name)
    atts = _atts(name, 72)
    env = eng.engine.EnvImage(net, eng.abi.ENV_TARGET, attractors=atts, max_inner=300, force=force)
    oenv = orc.Env(orc.ENV_TARGET, onet.n, attractors=atts, max_inner=300, force=int(force))
    seed = _seed(name) + B
    tgt = np.arange(onet.n - 7, onet.n, dtype=np.int32)
    sim = eng.engine.Simulator(net, B, seed=seed)
    sim.rand_state()
    ost = orc.rand_state(onet, B, orc.Draws(seed=seed, epoch=0))
    hist = sim.ssd(iters, 0.02, tgt, env=env)
    ohist = orc.ssd(onet, oenv, ost, iters, 0.02, tgt, orc.Draws(seed=seed, epoch=1))
    assert hist.sum().item() == B * iters
    assert np.array_equal(hist.cpu().numpy().astype(np.uint64), ohist)
    assert np.array_equal(_np(sim.unpack()), ost)


# ------------------------------------------------------------------------------------------------ replayed draws
REPLAY = [(name, kind) for name in ("p100f", "tt70") for kind in ("target", "multi")]


@functools.lru_cache(maxsize=None)
def _replay_traj(name, kind):
    onet = _onet(name)
    n, B, L, cap = onet.n, 256, 700, 300
    atts = _atts(name, 72)
    multi = kind == "multi"
    oenv = orc.Env(orc.ENV_MULTI if multi else orc.ENV_TARGET, n, attractors=atts, horizon=100, max_inner=cap)
    rng = np.random.default_rng(_seed(name) + 99)
    ost = rng.integers(0, 2, size=(B, n)).astype(np.uint8)
    ost[:, : onet.first] = 0
    ota = rng.integers(0, len(atts), B).astype(np.int32)
    out = {"st0": ost.copy(), "ta": ota.copy(), "steps": []}
    ons = np.zeros(B, np.int32)
    for t in range(2):
        act = rng.integers(0, n + 1, size=(B, 3 if multi else 1)).astype(np.int32)
        ints = rng.integers(onet.first, n, size=(B, L)).astype(np.int32)
        dbls = rng.random((B, L))
        d = orc.Draws(ints=ints, dbls=dbls)
        obs, rew, term, trunc, inner = orc.env_step(onet, oenv, ost, ons, ota, act, d)
        out["steps"].append(dict(act=act, ints=ints, dbls=dbls, used=d.used.copy(), obs=obs, rew=rew, term=term, trunc=trunc,
                                 inner=inner, state=ost.copy()))
    return out, atts, cap


@gpu
@pytest.mark.parametrize("name,kind", REPLAY)
def test_replay_draws_many_envs(eng, name, kind):
    """k_env_step_att with replayed draws (lane mode; int and float64 rows per env) for 256 envs against the oracle, and the
    number of draws each env used.  The kernel does not bounds-check its rows: the oracle must leave room in every row first."""
    tr, atts, cap = _replay_traj(name, kind)
    for s in tr["steps"]:
        assert (s["used"][:, 0] < s["ints"].shape[1]).all() and (s["used"][:, 1] < s["dbls"].shape[1]).all()
    net = _net(eng, name)
    multi = kind == "multi"
    env = eng.engine.EnvImage(net, eng.abi.ENV_MULTI if multi else eng.abi.ENV_TARGET, attractors=atts, horizon=100, max_inner=cap)
    sim = eng.engine.Simulator(net, 256)
    sim.set_state(tr["st0"])
    sim.target_att.copy_(torch.from_numpy(tr["ta"]))
    for t, s in enumerate(tr["steps"]):
        rp = eng.engine.Replay(s["ints"], s["dbls"], "cuda")
        sim.env_step(env, torch.from_numpy(s["act"]), replay=rp)
        assert np.array_equal(_np(sim.unpack()), s["state"]), t
        assert np.array_equal(_np(sim.unpack(sim.obs_state)), s["obs"]), t
        assert np.array_equal(_np(sim.reward), s["rew"]) and np.array_equal(_np(sim.terminated), s["term"]), t
        assert np.array_equal(_np(sim.inner), s["inner"]), t
        assert np.array_equal(_np(rp.used), s["used"]), t


# ------------------------------------------------------------------------------------------------ fused vector step
@gpu
@pytest.mark.parametrize("kind", ["target", "multi"])
@pytest.mark.parametrize("B", [2048, 20000])
def test_vec_step_matches_oracle(eng, kind, B):
    """Simulator.vec_step with autoreset on the four-word two-level network and the 72-cube fixture: one launch that resets
    inside att_finish (B = 2048), or budgeted passes and one masked reset launch (B = 20000).  Rewards, flags, update counts,
    final observations, observations after the reset, episode returns and lengths, and the statistics against the oracle."""
    name, n_cubes = "p100t", 72
    onet, net = _onet(name), _net(eng, name)
    n, multi, seed, cap = onet.n, kind == "multi", 41, 300
    atts = _atts(name, n_cubes)
    env = eng.engine.EnvImage(net, eng.abi.ENV_MULTI if multi else eng.abi.ENV_TARGET, attractors=atts, horizon=3, max_inner=cap)
    oenv = orc.Env(orc.ENV_MULTI if multi else orc.ENV_TARGET, n, attractors=atts, horizon=3, max_inner=cap)
    sim = eng.engine.Simulator(net, B, seed=seed)
    sim.plan_budgets = () if B <= 8192 else (32, 256)
    assert len(sim._passes(env)) == (1 if B <= 8192 else 3)
    ep_return = torch.zeros(B, dtype=torch.int64, device="cuda")
    ep_len = torch.zeros(B, dtype=torch.int32, device="cuda")
    stats = torch.zeros(8, dtype=torch.int64, device="cuda")
    final_obs = torch.zeros_like(sim.state)
    sim.env_reset(env)
    ost, ons, ota = np.zeros((B, n), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
    orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=0))
    assert np.array_equal(_np(sim.unpack()), ost)
    rng = np.random.default_rng(6)
    ret, length, want = np.zeros(B, np.int64), np.zeros(B, np.int32), np.zeros(8, np.int64)
    for t in range(4):
        act = rng.integers(0, n + 1, size=(B, 3 if multi else 1)).astype(np.int32)
        sim.vec_step(env, torch.from_numpy(act).cuda(), ep_return, ep_len, stats, final_obs=final_obs)
        oobs, orew, oterm, otrunc, oin = orc.env_step(onet, oenv, ost, ons, ota, act, orc.Draws(seed=seed, epoch=1 + 2 * t))
        done = (oterm | otrunc).astype(bool)
        orc.env_reset(onet, oenv, ost, ons, ota, orc.Draws(seed=seed, epoch=2 + 2 * t), mask=done.astype(np.uint8))
        assert np.array_equal(_np(sim.reward), orew) and np.array_equal(_np(sim.inner), oin), t
        assert np.array_equal(_np(sim.terminated), oterm) and np.array_equal(_np(sim.truncated), otrunc), t
        assert np.array_equal(_np(sim.unpack(final_obs)), oobs), t
        assert np.array_equal(_np(sim.unpack(sim.obs_state)), np.where(done[:, None], ost, oobs)), t
        assert np.array_equal(_np(sim.unpack()), ost) and np.array_equal(_np(sim.target_att), ota), t
        ret += orew
        length += 1
        want += np.array([done.sum(), ret[done].sum(), length[done].sum(), oterm.sum(), (oin >= cap).sum(), B, 0, 0], np.int64)
        ret[done], length[done] = 0, 0
        assert np.array_equal(_np(ep_return), ret) and np.array_equal(_np(ep_len), length), t
        assert np.array_equal(_np(stats), want), t
    assert want[0] > 0 and want[3] > 0 and want[4] > 0  # episodes ended, some in the target, some at the cap


# ------------------------------------------------------------------------------------------------ premises (CPU)
def _threshold_class(fmax):
    return "quad" if fmax <= 5 else ("two-level" if fmax <= 17 else "flat")


def _first_match(atts, states):
    """Index of the first cube each state matches (len(cubes) if none)."""
    cubes = np.array([[2 if v == "*" else int(v) for v in c] for a in atts for c in a], np.int8)
    care = cubes != 2
    first = np.full(len(states), len(cubes))
    for c in range(len(cubes) - 1, -1, -1):
        hit = ((states[:, care[c]] == cubes[c, care[c]]).all(1))
        first[hit] = c
    return first


@pytest.mark.parametrize("case", CASES + PLACEMENTS, ids=lambda c: c.id)
def test_cases_reach_their_regime(case):
    """What each GPU case above is there for, shown on the oracle's outputs (no GPU needed): the network's width and
    threshold class; envs that stop inside the loop and envs that stop at the cap; envs that stop on a cube no branch below
    the intended one tests; and, for planned steps, envs still running after the first budget."""
    kind, n, fmax = NETS[case.name]
    onet = _onet(case.name)
    w32, tcls, big = SHAPE[case.name]
    assert (onet.n + 31) // 32 == w32
    if kind == "pred":
        sets = _ref(case.name)[1]
        real_fmax = max(sum(c is not None for c in s[0]) for s in sets)
        assert real_fmax == fmax and _threshold_class(fmax) == tcls and (n * fmax * 16 > 32 * 1024) == big
    atts = _atts(case.name, case.n_cubes)
    assert sum(map(len, atts)) == case.n_cubes and all(1 <= len(a) <= 3 for a in atts)
    steps = case.traj["steps"]
    inner = np.concatenate([s["inner"] for s in steps])
    if case.force:
        assert (inner == 1).all()
        return
    assert ((inner > 1) & (inner < case.cap)).any() and (inner == case.cap).any()
    stop = np.concatenate([s["obs"] for s in steps])  # TARGET: the final state; MULTI: the observation the loop ended on
    first = _first_match(atts, stop)
    inside = (inner > 1) & (inner < case.cap)
    assert (first[inside] < case.n_cubes).all()  # the loop stopped on a cube (the oracle agrees with itself)
    assert (first[inside] >= THRESH[case.n_cubes]).any()
    for plan, s in zip(case.plans, steps):
        if PLANS[plan]:
            assert (s["inner"] > PLANS[plan][0]).any()  # the first pass parks envs
    rew = np.concatenate([s["rew"] for s in steps])
    if case.multi:  # the observation matched the first cube of the target attractor: 1000 - len(actions)
        assert (rew > 900).any() or case.n_cubes == 7  # (the 7-cube fixture's last attractor is a decoy)
    else:
        assert (rew == 20).any()
        if case.n_cubes >= 7:  # ... and at least once on the SECOND cube of the target attractor only
            off = np.cumsum([0] + [len(a) for a in atts])
            ta = np.concatenate([s["ta"] for s in steps])
            sizes = off[ta + 1] - off[ta]
            second = (rew == 20) & (sizes >= 2) & (first == off[ta] + 1)
            assert second.any()
