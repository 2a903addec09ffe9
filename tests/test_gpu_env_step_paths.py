"""GPU: k_env_step — the env.step kernel of PBNEnv, PBCNEnv, both sampled-data envs and both self-triggering envs, behind the
single-env classes and the fused PBNVectorEnv step of the "pbn" family — against the oracle on every path it takes.  Everything
here is bit-exact: state, observation, int32 reward, float64 reward, flags, update counts and the draws each env used.

Networks, and the path each one is here for:
  tt31          truth table, 1 word                        tt_micro_step_sa, threshold table staged in shared memory
  tt70          truth table, 3 words (26 unused bits)      multi-word cube tests (cube_match_sa, 1024-byte column stride)
  pbcn1024      synthetic PBCN, 32 words, 40 control nodes threshold table in global memory (thr_dev: table > 16 KB)
  p30q          predictor, 1 word, one threshold quad      micro_step<PRED, ...>
  p100t         predictor, 4 words, two-level rows         micro_step<PRED, ...> on a wider state
  28_15_median  the shipped 28-gene set (<= 15 predictors) micro_step<PRED, ...> on real data
Every network runs PBN, PBCN, PBN_SD, PBCN_SD (control_write 0 and 1), PBN_ST (T capped) and PBCN_ST (control_write 0 and 1,
T capped and T = None), with M in {3, 32, 40} where M < N: M = 32 is the all-ones mask of CtlWrite, M = 40 its per-node
branch.  Sampled-data intervals include 1, even and odd values and values of 64 and more (odd intervals hand the PBCN_SD pair
loop's last update back to the stream object).  The attractors overlap (PBCN's wrong_attractor_cost x m sees m >= 2) and a third
of the envs start on a target state, so every reward branch fires.  Draws are Philox everywhere (batches of 1, 257 and 1500,
one batch at env0 >= 2^32), replayed on two networks, and replayed once more for a PBCN_ST macro step of more than 2048
primitive steps with no cap (the gamma_pow[n_gamma - 1] reuse, which Philox draws practically never reach).

The product reports nothing about which branch ran, so test_cases_reach_their_regime (CPU only) shows each case's premise on
the oracle's outputs and the network data."""
import ctypes as C
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

import oracle as orc  # noqa: E402
from golden_util import random_predictor_sets, random_tt_data, synthetic_pbcn  # noqa: E402

# name: (kind, n, max predictors per node)
NETS = {"tt31": ("tt", 31, 0), "tt70": ("tt", 70, 0), "pbcn1024": ("pbcn", 1024, 0), "p30q": ("pred", 30, 5),
        "p100t": ("pred", 100, 16), "28_15_median": ("bittner", 28, 15)}
# (w32, threshold class of a predictor net, truth table above the 16 KB staged in shared memory)
SHAPE = {"tt31": (1, None, False), "tt70": (3, None, False), "pbcn1024": (32, None, True), "p30q": (1, "quad", None),
         "p100t": (4, "two-level", None), "28_15_median": (1, "two-level", None)}
TT_THR_SMEM_MAX = 16 * 1024  # PBN_TT_THR_SMEM_MAX in pbn_b200.cu
KINDS = ("pbn", "pbcn", "pbn_sd", "pbcn_sd", "pbn_st", "pbcn_st")
INTERVALS = np.array([1, 2, 3, 4, 7, 8, 64, 65, 77])
SUCCESS, WRONG = 10, 2  # successful_reward, wrong_attractor_cost
GAMMA = 0.97


def _seed(name):
    return sum(map(ord, name))


@functools.lru_cache(maxsize=None)
def _ref(name):
    """Reference form of a network: ("pred", sets, ids) or ("tt", pbn_data)."""
    kind, n, fmax = NETS[name]
    if kind == "pred":
        return ("pred",) + random_predictor_sets(n, fmax, seed=_seed(name))
    if kind == "bittner":
        return ("pred",) + orc.load_bittner(name)
    return ("tt", random_tt_data(n, seed=_seed(name)) if kind == "tt" else synthetic_pbcn(n=n, m=40, seed=5))


@functools.lru_cache(maxsize=None)
def _onet(name):
    r = _ref(name)
    return orc.net_from_predictor_sets(r[1], r[2]) if r[0] == "pred" else orc.net_from_pbn_data(r[1])


@functools.lru_cache(maxsize=None)
def _fixture(name):
    """(attractors, targets) of a network.  Four attractors: two one-cube attractors with two cared nodes each that overlap on
    one node, one of two broad cubes, and twelve decoy cubes (PBNEnv.reset redraws an attractor of more than 10 states).  The
    cared nodes are the last six, which every network updates and no control vector writes.  Targets: the reset states of the
    first two attractors (value bits, wildcards 0, node 0 cleared) and two random states."""
    n = _onet(name).n
    rng = np.random.default_rng(_seed(name) + 1)
    v = [int(x) for x in rng.integers(0, 2, 6)]

    def cube(care):
        c = ["*"] * n
        for i, x in care.items():
            c[i] = x
        return tuple(c)

    atts = [[cube({n - 1: v[0], n - 2: v[1]})], [cube({n - 2: v[1], n - 3: v[2]})],
            [cube({n - 4: v[3]}), cube({n - 5: v[4], n - 6: v[5]})],
            [tuple(int(x) for x in rng.integers(0, 2, n)) for _ in range(12)]]
    targets = [tuple(0 if x == "*" else x for x in a[0]) for a in atts[:2]]
    targets = [(0,) + t[1:] for t in targets]
    targets += [(0,) + tuple(int(x) for x in rng.integers(0, 2, n - 1)) for _ in range(2)]
    return atts, targets


@functools.lru_cache(maxsize=None)
def _state_fixture(name):
    """(attractors, targets) of whole states for the vector-env test, whose resets draw a state of an attractor (the
    reference's attractors are sets of states): s0 lies in the first two attractors (m = 2 there), s1 and s2 are targets, the
    last attractor has twelve states (redrawn by the reset)."""
    n = _onet(name).n
    rng = np.random.default_rng(_seed(name) + 2)
    s = [(0,) + tuple(int(x) for x in rng.integers(0, 2, n - 1)) for _ in range(16)]
    return [[s[0]], [s[0], s[1]], [s[2], s[3]], s[4:]], [s[1], s[2]]


def _m_of(name, states):
    """Number of attractors each state lies in (PBCNEnv._get_reward's m), from the cube lists."""
    atts, _ = _fixture(name)
    m = np.zeros(len(states), np.int64)
    for a in atts:
        hit = np.zeros(len(states), bool)
        for c in a:
            care = np.array([x != "*" for x in c])
            val = np.array([0 if x == "*" else x for x in c], np.uint8)
            hit |= (states[:, care] == val[care]).all(1)
        m += hit
    return m


def _in_target(name, states):
    _, targets = _fixture(name)
    return (states[:, None, :] == np.array(targets, np.uint8)[None]).all(2).any(1)


def _orc_step(onet, oenv, state, actions, draws, env0):
    """orc_env_step_f64 with every output kept: (obs, reward int32, reward float64, terminated, truncated, updates)."""
    B = state.shape[0]
    actions = np.ascontiguousarray(actions, np.int32)
    obs = np.zeros_like(state)
    rew, rf = np.zeros(B, np.int32), np.zeros(B, np.float64)
    term, trunc, inner = np.zeros(B, np.uint8), np.zeros(B, np.uint8), np.zeros(B, np.int32)
    ns, ta = np.zeros(B, np.int32), np.zeros(B, np.int32)
    p = orc._p
    orc.lib().orc_env_step_f64(C.byref(onet.c), C.byref(oenv.c), p(state), p(ns), p(ta), p(actions), C.c_int(actions.shape[1]),
                               p(obs), p(rew), p(rf), p(term), p(trunc), p(inner), C.c_int64(B), C.c_int64(env0), C.byref(draws.c))
    return obs, rew, rf, term, trunc, inner


class Case:
    """One env kind on one network, stepped `steps` times from planted start states; the oracle's trajectory is computed once
    per session and shared by the GPU test and the regime test."""

    def __init__(self, name, kind, cw=0, M=3, T=5, B=257, env0=0, steps=3, replay=False, long_st=False):
        self.name, self.kind, self.cw, self.M, self.T, self.B, self.env0 = name, kind, cw, M, T, B, env0
        self.steps, self.replay, self.long_st = steps, replay, long_st
        self.st = kind.endswith("_st")
        self.seed = _seed(name) + 11 * KINDS.index(kind) + 3 * cw + M + (T or 0) + B + (env0 >> 20) + 7 * replay

    @property
    def id(self):
        t = (f"-T{self.T}" if self.T else "-Tnone") if self.st else ""
        c = f"-cw{self.cw}-M{self.M}" if self.kind.startswith("pbcn_") else ""
        d = "-longreplay" if self.long_st else ("-replay" if self.replay else "")
        e = f"-env0_{self.env0:#x}" if self.env0 else ""
        return f"{self.name}-{self.kind}{c}{t}-B{self.B}{e}{d}"

    def env_kw(self):
        atts, targets = _fixture(self.name)
        kw = dict(attractors=atts, targets=targets, n_control=self.M, control_write=self.cw, successful_reward=SUCCESS,
                  wrong_attractor_cost=WRONG)
        if self.st:
            kw.update(gamma=GAMMA, max_interval=self.T)
        return kw

    def _actions(self, rng, planted, tgt):
        n, B, M = _onet(self.name).n, self.B, self.M
        a = rng.integers(0, n if self.kind in ("pbn", "pbcn") else n + 1, B)  # PBN/PBCN flip node a, the others node a - 1
        a[planted & (rng.random(B) < 0.7)] = 0
        pv = rng.integers(1, 11, B)
        iv = rng.choice(INTERVALS, B)
        ctl = rng.integers(0, 2, (B, M))
        if self.cw:  # a planted env is written its target's first M bits: the target stays reachable
            ctl[planted] = tgt[planted, :M]
        if self.kind in ("pbn", "pbcn"):
            act = a[:, None]
        elif self.kind == "pbn_sd":
            act = np.stack([a, iv], 1)
        elif self.kind == "pbn_st":
            act = np.stack([a, pv], 1)
        else:
            act = np.concatenate([(iv if self.kind == "pbcn_sd" else pv)[:, None], ctl], 1)
        if self.long_st:
            act[:, 0] = 1  # prob 0.1
        return act.astype(np.int32)

    def _draws(self, rng, t):
        """(oracle draws, ints, dbls): Philox (epoch t), or rows of replayed draws."""
        onet, B = _onet(self.name), self.B
        if not self.replay:
            return orc.Draws(seed=self.seed, epoch=t, B=B), None, None
        L = 2600 if self.long_st else 400
        ints = rng.integers(onet.first, onet.n, size=(B, L)).astype(np.int32)
        dbls = rng.random((B, 2 * L))
        if self.long_st:  # per primitive step: value, stop.  Stop draws above prob 0.1 up to a step past 2048 for most envs
            last = rng.integers(1990, 2560, B)
            for e in range(B):
                dbls[e, 1:2 * last[e]:2] = rng.uniform(0.11, 1.0, last[e])
                dbls[e, 2 * last[e] + 1] = 0.05
        return orc.Draws(ints=ints, dbls=dbls), ints, dbls

    @functools.cached_property
    def traj(self):
        onet = _onet(self.name)
        n, B = onet.n, self.B
        okind = getattr(orc, "ENV_" + self.kind.upper())
        oenv = orc.Env(okind, n, **self.env_kw())
        _, targets = _fixture(self.name)
        rng = np.random.default_rng(self.seed)
        ost = rng.integers(0, 2, size=(B, n)).astype(np.uint8)
        ost[:, : onet.first] = 0
        planted = rng.random(B) < 1 / 3
        tgt = np.array(targets, np.uint8)[rng.integers(0, len(targets), B)]
        ost[planted] = tgt[planted]
        out = {"st0": ost.copy(), "planted": planted, "steps": []}
        for t in range(self.steps):
            act = self._actions(rng, planted, tgt)
            d, ints, dbls = self._draws(rng, t)
            st_before = ost.copy()
            obs, rew, rf, term, trunc, inner = _orc_step(onet, oenv, ost, act, d, self.env0)
            out["steps"].append(dict(act=act, before=st_before, obs=obs, rew=rew, rf=rf, term=term, trunc=trunc, inner=inner,
                                     used=d.used.copy(), state=ost.copy(), ints=ints, dbls=dbls))
        return out


def _cases():
    out = []
    for i, name in enumerate(NETS):
        n = NETS[name][1]
        Ms = [M for M in (3, 32, 40) if M < n]
        B = (257, 1500)[i % 2] if name != "pbcn1024" else 257
        out += [Case(name, k, B=B) for k in ("pbn", "pbcn", "pbn_sd")]
        out += [Case(name, "pbcn_sd", cw=0, M=Ms[-1], B=B)] + [Case(name, "pbcn_sd", cw=1, M=M, B=B) for M in Ms]
        out += [Case(name, "pbn_st", T=7, B=B)]
        out += [Case(name, "pbcn_st", cw=cw, M=Ms[(cw + j) % len(Ms)], T=T, B=B) for cw in (0, 1) for j, T in enumerate((5, None))]
    return out


CASES = _cases()
# one env per launch, and env ids above 2^32 (the high counter word of the Philox stream)
EDGES = [Case("tt70", "pbcn_sd", cw=1, M=32, B=1), Case("p30q", "pbn_st", T=7, B=1), Case("p100t", "pbcn_st", cw=1, M=40, T=None, B=1),
         Case("tt70", "pbcn_sd", cw=1, M=40, B=257, env0=(1 << 32) + 5), Case("p100t", "pbn_sd", B=257, env0=(3 << 32) + 77)]
REPLAYS = [Case(name, k, cw=1, M=3, T=(5 if k == "pbn_st" else None), B=300, replay=True) for name in ("tt70", "p30q") for k in KINDS]
LONG_ST = [Case("tt70", "pbcn_st", cw=1, M=3, T=None, B=64, steps=1, replay=True, long_st=True)]
ALL = CASES + EDGES + REPLAYS + LONG_ST


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


def _env(eng, case):
    return eng.engine.EnvImage(_net(eng, case.name), getattr(eng.abi, "ENV_" + case.kind.upper()), **case.env_kw())


def _run(eng, case):
    tr = case.traj
    abi, E = eng.abi, eng.engine
    env = _env(eng, case)
    sim = E.Simulator(_net(eng, case.name), case.B, env0=case.env0)
    sim.set_state(tr["st0"])
    rf = torch.zeros(case.B, dtype=torch.float64, device="cuda")
    used = torch.zeros((case.B, 2), dtype=torch.int64, device="cuda")
    for t, s in enumerate(tr["steps"]):
        act = torch.from_numpy(s["act"]).cuda()
        if case.replay:
            rp = E.Replay(s["ints"], s["dbls"], "cuda")
            d, used = rp.struct(), rp.used
        else:
            used.fill_(-1)
            d = abi.PbnDraws(mode=abi.DRAW_PHILOX, seed=case.seed, epoch=t, used=E._ptr(used))
        sim.obs_state.zero_()
        head = (env.handle, E._ptr(sim.state), E._ptr(sim.n_steps), E._ptr(sim.target_att), E._ptr(act), act.shape[1],
                E._ptr(sim.obs_state), E._ptr(sim.reward))
        tail = (E._ptr(sim.terminated), E._ptr(sim.truncated), E._ptr(sim.inner), case.B, case.env0, C.byref(d), E._stream())
        if case.st:
            abi.check(abi.lib().pbn_env_step_f64(*head, E._ptr(rf), *tail))
        else:
            abi.check(abi.lib().pbn_env_step(*head, *tail))
        where = (case.id, t)
        assert np.array_equal(_np(sim.unpack()), s["state"]), where
        assert np.array_equal(_np(sim.unpack(sim.obs_state)), s["obs"]), where
        assert np.array_equal(_np(sim.reward), s["rew"]), where
        if case.st:
            assert np.array_equal(_np(rf), s["rf"]), where  # float64, bit for bit
        assert np.array_equal(_np(sim.terminated), s["term"]) and np.array_equal(_np(sim.truncated), s["trunc"]), where
        assert np.array_equal(_np(sim.inner), s["inner"]), where
        assert np.array_equal(_np(used), s["used"]), where


@gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c.id)
def test_env_step_matches_oracle(eng, case):
    """Every env kind k_env_step runs, on every network, Philox draws: three env.steps from planted start states."""
    _run(eng, case)


@gpu
@pytest.mark.parametrize("case", EDGES, ids=lambda c: c.id)
def test_env_step_edge_batches_match_oracle(eng, case):
    """A batch of one env, and env ids above 2^32."""
    _run(eng, case)


@gpu
@pytest.mark.parametrize("case", REPLAYS + LONG_ST, ids=lambda c: c.id)
def test_env_step_replay_matches_oracle(eng, case):
    """Replayed draws, a row of ints and one of float64s per env, and the number of each that every env used; the last case is
    a PBCN_ST macro step with no cap that runs past the 2048 tabulated powers of gamma.  The kernel does not bounds-check its
    rows: the oracle must leave room in every row first."""
    for s in case.traj["steps"]:
        assert (s["used"][:, 0] < s["ints"].shape[1]).all() and (s["used"][:, 1] < s["dbls"].shape[1]).all()
    _run(eng, case)


# ------------------------------------------------------------------------------------------------ fused vector step
@gpu
@pytest.mark.parametrize("kind", ["pbn", "pbcn", "pbn_sd", "pbcn_sd"])
@pytest.mark.parametrize("name", ["tt70", "p30q"])
def test_vec_step_matches_oracle(eng, name, kind):
    """Simulator.vec_step with autoreset (k_env_step, vec_finish and the PBN-family reset in one launch) against the oracle's
    env.step followed by a masked reset: rewards, flags, update counts, final observations, observations after the reset,
    episode returns and lengths, and the statistics.  One attractor has twelve cubes, so some resets redraw."""
    case = Case(name, kind, cw=1, M=3, B=1500)
    onet, net = _onet(name), _net(eng, name)
    n, B, seed = onet.n, case.B, case.seed
    atts, targets = _state_fixture(name)
    kw = dict(case.env_kw(), attractors=atts, targets=targets)
    env = eng.engine.EnvImage(net, getattr(eng.abi, "ENV_" + kind.upper()), **kw)
    oenv = orc.Env(getattr(orc, "ENV_" + kind.upper()), n, **kw)
    sim = eng.engine.Simulator(net, B, seed=seed)
    ep_return = torch.zeros(B, dtype=torch.int64, device="cuda")
    ep_len = torch.zeros(B, dtype=torch.int32, device="cuda")
    stats = torch.zeros(8, dtype=torch.int64, device="cuda")
    final_obs = torch.zeros_like(sim.state)
    sim.env_reset(env)
    ost, ons, ota = np.zeros((B, n), np.uint8), np.zeros(B, np.int32), np.zeros(B, np.int32)
    d = orc.Draws(seed=seed, epoch=0, B=B)
    orc.env_reset(onet, oenv, ost, ons, ota, d)
    redraws = int((d.used[:, 0] > 2).sum())
    assert np.array_equal(_np(sim.unpack()), ost)
    rng = np.random.default_rng(6)
    tgt = np.array(targets, np.uint8)[rng.integers(0, len(targets), B)]
    ret, length, want = np.zeros(B, np.int64), np.zeros(B, np.int32), np.zeros(8, np.int64)
    for t in range(6):
        act = case._actions(rng, rng.random(B) < 0.5, tgt)
        sim.vec_step(env, torch.from_numpy(act).cuda(), ep_return, ep_len, stats, final_obs=final_obs)
        oobs, orew, _rf, oterm, otrunc, oin = _orc_step(onet, oenv, ost, act, orc.Draws(seed=seed, epoch=1 + 2 * t), 0)
        done = (oterm | otrunc).astype(bool)
        d = orc.Draws(seed=seed, epoch=2 + 2 * t, B=B)
        orc.env_reset(onet, oenv, ost, ons, ota, d, mask=done.astype(np.uint8))
        redraws += int((d.used[:, 0] > 2).sum())
        assert np.array_equal(_np(sim.reward), orew) and np.array_equal(_np(sim.inner), oin), t
        assert np.array_equal(_np(sim.terminated), oterm) and np.array_equal(_np(sim.truncated), otrunc), t
        assert np.array_equal(_np(sim.unpack(final_obs)), oobs), t
        assert np.array_equal(_np(sim.unpack(sim.obs_state)), np.where(done[:, None], ost, oobs)), t
        assert np.array_equal(_np(sim.unpack()), ost), t
        ret += orew
        length += 1
        want += np.array([done.sum(), ret[done].sum(), length[done].sum(), oterm.sum(), 0, B, 0, 0], np.int64)
        ret[done], length[done] = 0, 0
        assert np.array_equal(_np(ep_return), ret) and np.array_equal(_np(ep_len), length), t
        assert np.array_equal(_np(stats), want), t
    assert want[0] > 0 and redraws > 0 and (ret != 0).any()  # episodes ended, resets redrew, episodes are still running


# ------------------------------------------------------------------------------------------------ ignored interventions
@gpu
@pytest.mark.parametrize("kind", ["pbn", "pbn_sd", "pbn_st", "multi"])
@pytest.mark.parametrize("name", ["tt70", "p30q"])
def test_out_of_range_interventions_are_free(eng, name, kind):
    """An intervention outside the network is ignored, and costs nothing: a vector env given out-of-range actions steps exactly
    like one given action 0 (MULTI: like one whose slot is absent) — states, observations, rewards, flags, update counts,
    episode returns and lengths, statistics — and counts those env.steps in stats[6]."""
    onet, net = _onet(name), _net(eng, name)
    n, B, seed = onet.n, 1024, 17
    atts, targets = _fixture(name)
    if kind == "multi":
        env = eng.engine.EnvImage(net, eng.abi.ENV_MULTI, attractors=atts, horizon=4, max_inner=40)
        K, empty = 3, -1
    else:
        st = kind == "pbn_st"
        env = eng.engine.EnvImage(net, getattr(eng.abi, "ENV_" + kind.upper()), attractors=atts, targets=targets,
                                  gamma=GAMMA if st else None, max_interval=5 if st else None)
        K, empty = (1 if kind == "pbn" else 2), 0
    st = kind == "pbn_st"
    sims = [eng.engine.Simulator(net, B, seed=seed) for _ in range(2)]
    bufs = []
    for sim in sims:
        sim.env_reset(env)
        bufs.append(dict(ret=torch.zeros(B, dtype=torch.float64 if st else torch.int64, device="cuda"),
                         len=torch.zeros(B, dtype=torch.int32, device="cuda"), stats=torch.zeros(8, dtype=torch.int64, device="cuda"),
                         fo=torch.zeros_like(sim.state), rs=torch.zeros(1, dtype=torch.float64, device="cuda")))
    # out of range: PBN flips node a, the others node a - 1; MULTI's negative slots are absent, not out of range
    lo_bad = [-7, -2**31] if kind != "multi" else []
    bad_vals = np.array(lo_bad + [n + 1, n + 7, 1000, 2**31 - 1] + ([n] if kind == "pbn" else []))
    rng = np.random.default_rng(5)
    n_bad = 0
    for t in range(5):
        act = rng.integers(0, n + (0 if kind == "pbn" else 1), size=(B, K)).astype(np.int32)
        if kind == "pbn_sd":
            act[:, 1] = rng.choice(INTERVALS[:6], B)
        if kind == "pbn_st":
            act[:, 1] = rng.integers(1, 11, B)
        slots = K if kind == "multi" else 1
        sel = rng.random((B, slots)) < 0.25
        wild = act.copy()
        wild[:, :slots][sel] = rng.choice(bad_vals, size=int(sel.sum()))
        act[:, :slots][sel] = empty
        n_bad += int(sel.any(1).sum())
        outs = []
        for sim, b, a in zip(sims, bufs, (wild, act)):
            sim.vec_step(env, torch.from_numpy(a).cuda(), b["ret"], b["len"], b["stats"], final_obs=b["fo"],
                         return_sum_f64=b["rs"] if st else None)
            outs.append([_np(sim.unpack()), _np(sim.unpack(sim.obs_state)), _np(sim.reward), _np(sim.terminated),
                         _np(sim.truncated), _np(sim.inner), _np(b["ret"]), _np(b["len"]), _np(b["fo"]), _np(sim.target_att)]
                        + ([_np(sim.reward_f64)] if st else []))
        for k, (x, y) in enumerate(zip(*outs)):
            assert np.array_equal(x, y), (t, k)
        if st:  # a float64 sum of atomic adds: its order, and so its last bits, vary from launch to launch
            x, y = (float(b["rs"]) for b in bufs)
            assert abs(x - y) <= 1e-12 * max(1.0, abs(y)), t
    s_bad, s_ok = _np(bufs[0]["stats"]), _np(bufs[1]["stats"])
    assert s_bad[6] == n_bad and s_ok[6] == 0 and np.array_equal(np.delete(s_bad, 6), np.delete(s_ok, 6))
    assert s_ok[0] > 0  # episodes ended (resets ran in both)


@gpu
def test_env_create_refuses_n_control_outside_the_network(eng):
    """control_write stores the control vector into nodes 0..M-1 of the env's own state column: M > N (or M < 0) is refused
    when the env is created, before any step could write past the column."""
    net = _net(eng, "tt70")
    atts, targets = _fixture("tt70")
    for kind in ("PBCN_SD", "PBCN_ST"):
        for M in (-1, 71, 100, 1 << 20):
            with pytest.raises(ValueError, match="n_control"):
                eng.engine.EnvImage(net, getattr(eng.abi, "ENV_" + kind), attractors=atts, targets=targets, n_control=M,
                                    control_write=True, gamma=0.9, max_interval=5)
            assert b"n_control must be in 0..n_nodes" in eng.abi.lib().pbn_last_error()
    eng.engine.EnvImage(net, eng.abi.ENV_PBCN_SD, attractors=atts, targets=targets, n_control=70, control_write=True)  # M = N


# ------------------------------------------------------------------------------------------------ premises (CPU)
def _threshold_class(fmax):
    return "quad" if fmax <= 5 else ("two-level" if fmax <= 17 else "flat")


@pytest.mark.parametrize("case", ALL, ids=lambda c: c.id)
def test_cases_reach_their_regime(case):
    """What each GPU case above is there for, shown on the oracle's outputs and the network data (no GPU needed): the
    network's width, threshold class and truth-table size; every reward branch of the env kind; the PBCN_SD overshoot penalty;
    m >= 2; self-triggering steps that stop on the draw and at T; the uncapped replay past 2048 primitive steps; control bits
    at node 32 and above in the final states when M = 40."""
    onet = _onet(case.name)
    n = onet.n
    w32, tcls, big = SHAPE[case.name]
    assert (n + 31) // 32 == w32 and case.M < n
    r = _ref(case.name)
    if r[0] == "pred":
        assert _threshold_class(max(sum(c is not None for c in s[0]) for s in r[1])) == tcls
    else:
        assert (4 * sum(t[1].size for t in r[1]) > TT_THR_SMEM_MAX) == big
    steps = case.traj["steps"]
    cat = {k: np.concatenate([s[k] for s in steps]) for k in ("act", "obs", "rew", "term", "inner", "used")}
    if case.long_st:
        assert (cat["inner"] > 2048).any() and (cat["inner"] < 2048).any()
        return
    if case.B == 1:
        return
    term, obs, act = cat["term"].astype(bool), cat["obs"], cat["act"]
    used = cat["used"]
    if not case.replay:  # Philox: two words per update, one more per self-triggering stop
        assert (used[:, 0] == (3 if case.st else 2) * cat["inner"]).all() and (used[:, 1] == 0).all()
    if case.kind.startswith("pbn"):  # last update: 20 in a target, -5 after an applied flip, -4 otherwise
        assert term.any() and (~term & (act[:, 0] != 0)).any() and (~term & (act[:, 0] == 0)).any()
        assert (term == _in_target(case.name, obs)).all()
    else:  # successful_reward in a target, -wrong_attractor_cost * m outside, m = 0, 1 and >= 2
        m = _m_of(case.name, obs)
        assert term.any() and (~term & (m == 0)).any() and (~term & (m == 1)).any() and (~term & (m >= 2)).any()
    if case.kind == "pbcn":
        assert set(np.unique(cat["rew"])) >= {SUCCESS, 0, -WRONG, -2 * WRONG}
    if case.kind.endswith("_sd"):
        iv = act[:, 1] if case.kind == "pbn_sd" else act[:, 0]
        assert (cat["inner"] == iv).all() and set(iv.tolist()) >= {1, 2, 3, 64, 65}
    if case.kind == "pbcn_sd":  # overshoot: the first update lands in a target and the interval goes on
        first = [s["before"].copy() for s in steps]
        hit = []
        oenv = orc.Env(orc.ENV_PBCN_SD, n, **case.env_kw())
        for t, s in enumerate(steps):
            a1 = s["act"].copy()
            a1[:, 0] = 1
            d = orc.Draws(ints=s["ints"], dbls=s["dbls"]) if case.replay else orc.Draws(seed=case.seed, epoch=t)
            _o, _r, _rf, t1, _tr, _in = _orc_step(onet, oenv, first[t], a1, d, case.env0)
            hit.append(t1.astype(bool) & (s["act"][:, 0] >= 2))
        assert np.concatenate(hit).any()
    if case.st:
        pv = act[:, 1] if case.kind == "pbn_st" else act[:, 0]
        assert set(pv.tolist()) == set(range(1, 11))
        if case.T:
            assert (cat["inner"] < case.T).any() and (cat["inner"] == case.T).any() and (cat["inner"] <= case.T).all()
    if case.kind.startswith("pbcn_") and case.cw and case.M > 32:
        assert obs[:, 32:case.M].any()
