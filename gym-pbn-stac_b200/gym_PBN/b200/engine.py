"""Device-side engine: owns the compiled network / env handles and the per-env state tensors, and
launches the kernels of libpbn_b200.so on the caller's current CUDA stream.  torch is used for device
memory and streams only.

State layout (HBM): int32 planes [W32][B]; node i of env e is bit (i & 31) of state[i >> 5, e].
Every launch gets a fresh Philox epoch; env e of a job uses stream (seed; epoch, env0 + e), so the
result of a job does not depend on how its envs are split over launches, ranks or GPUs.
"""
import ctypes as C

import numpy as np
import torch

from . import abi
from .compiler import NetworkSpec, compile_cubes


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class on_device:
    """`with on_device(dev):` — make dev current for the block and put the caller's device back afterwards; costs two integer
    compares when dev already is current (the hot paths call this per launch)."""

    __slots__ = ("dev", "prev")

    def __init__(self, device):
        self.dev = device.index

    def __enter__(self):
        self.prev = torch.cuda.current_device()
        if self.prev != self.dev:
            torch.cuda.set_device(self.dev)

    def __exit__(self, *exc):
        if self.prev != self.dev:
            torch.cuda.set_device(self.prev)
        return False


def require_cuda(device):
    device = torch.device(device if device is not None else "cuda")
    if device.type != "cuda" or not torch.cuda.is_available():
        raise abi.PbnError("gym_PBN (B200 build) needs a CUDA device; there is no CPU fallback")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


class Network:
    """Compiled network handle (immutable; shareable across streams)."""

    def __init__(self, spec: NetworkSpec, device=None):
        self.spec = spec
        self.device = require_cuda(device)
        self.n, self.w32, self.kind = spec.n, spec.w32, spec.kind
        a = spec.arrays
        d = abi.PbnNetDesc(kind=spec.kind, n_nodes=spec.n, first_updatable=spec.first_updatable)
        for k, v in a.items():
            setattr(d, k, _np_ptr(v))
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            abi.check(abi.lib().pbn_net_create(C.byref(d), C.byref(h)))
        self.handle = h

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                abi.lib().pbn_net_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class EnvImage:
    """Compiled env description (cubes, rewards, horizon) bound to a Network."""

    def __init__(self, net: Network, kind, attractors=(), targets=(), horizon=100, max_inner=1 << 20, force=False,
                 dedup=True, control_write=False, n_control=0, successful_reward=10, wrong_attractor_cost=2,
                 gamma=None, max_interval=None):
        self.net, self.kind = net, kind
        self.n_att = len(attractors)
        self.force = bool(force)
        self.max_inner = int(max_inner)
        cube, off, tgt_first, n_tgt = compile_cubes(net.n, attractors, targets)
        self._keep = (cube, off)
        d = abi.PbnEnvDesc(kind=kind, horizon=int(horizon), max_inner=int(max_inner), force=int(bool(force)),
                           dedup=int(bool(dedup)), control_write=int(bool(control_write)), n_control=int(n_control),
                           successful_reward=int(successful_reward), wrong_attractor_cost=int(wrong_attractor_cost),
                           n_att=self.n_att, att_off=_np_ptr(off), cube=_np_ptr(cube), tgt_first=tgt_first, n_tgt=n_tgt)
        if kind in (abi.ENV_PBN_ST, abi.ENV_PBCN_ST):
            # gamma**i exactly as the reference computes it (Python float pow, self_triggering.py:76,178); the kernel only
            # multiplies and adds.  With no cap (T = None) the interval is geometric with p >= 0.1: 2048 entries are plenty.
            n_gamma = int(max_interval) if max_interval else 2048
            self._gamma_pow = np.array([float(gamma) ** i for i in range(n_gamma)], np.float64)
            d.gamma_pow, d.n_gamma, d.max_interval = _np_ptr(self._gamma_pow), n_gamma, int(max_interval or 0)
        h = C.c_void_p()
        with torch.cuda.device(net.device):
            abi.check(abi.lib().pbn_env_create(net.handle, C.byref(d), C.byref(h)))
        self.handle = h

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                abi.lib().pbn_env_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class Replay:
    """Recorded draws (SURVEY.md §3.5) for B envs: ints int32 [B][Li], dbls float64 [B][Ld]."""

    def __init__(self, ints, dbls, device, B=None):
        ints = np.zeros((B or 1, 1), np.int32) if ints is None else np.asarray(ints, np.int32)
        dbls = np.zeros((B or 1, 1), np.float64) if dbls is None else np.asarray(dbls, np.float64)
        if ints.ndim == 1:
            ints = ints.reshape(1, -1)
        if dbls.ndim == 1:
            dbls = dbls.reshape(1, -1)
        if ints.shape[1] == 0:
            ints = np.zeros((ints.shape[0], 1), np.int32)
        if dbls.shape[1] == 0:
            dbls = np.zeros((dbls.shape[0], 1), np.float64)
        self.ints = torch.from_numpy(np.ascontiguousarray(ints)).to(device)
        self.dbls = torch.from_numpy(np.ascontiguousarray(dbls)).to(device)
        self.used = torch.zeros((self.ints.shape[0], 2), dtype=torch.int64, device=device)

    def struct(self):
        return abi.PbnDraws(mode=abi.DRAW_REPLAY, ints=_ptr(self.ints), dbls=_ptr(self.dbls),
                            int_stride=self.ints.shape[1], dbl_stride=self.dbls.shape[1], used=_ptr(self.used))


class Simulator:
    """B envs of one network on one GPU."""

    def __init__(self, net: Network, num_envs: int, seed: int = 0, env0: int = 0):
        self.net, self.B, self.env0 = net, int(num_envs), int(env0)
        self.device = net.device
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.epoch = 0
        self.state = torch.zeros((net.w32, self.B), dtype=torch.int32, device=self.device)
        self.n_steps = torch.zeros(self.B, dtype=torch.int32, device=self.device)
        self.target_att = torch.zeros(self.B, dtype=torch.int32, device=self.device)
        self.target_state = torch.zeros((net.w32, self.B), dtype=torch.int32, device=self.device)
        self.obs_state = torch.zeros((net.w32, self.B), dtype=torch.int32, device=self.device)
        self.reward = torch.zeros(self.B, dtype=torch.int32, device=self.device)
        self.terminated = torch.zeros(self.B, dtype=torch.bool, device=self.device)  # 1-byte 0/1, written by the kernels
        self.truncated = torch.zeros(self.B, dtype=torch.bool, device=self.device)
        self.inner = torch.zeros(self.B, dtype=torch.int32, device=self.device)
        self.launches = 0
        self._vec_cache = None
        self._unpack_out = None
        # step plan of the step-until-attractor envs (include/pbn_b200.h: PbnStepPlan): a full env.step is a first pass with
        # plan_budgets[0] updates per env (every lane owns an env; most envs finish there), resume passes with the further
        # budgets (the envs still outside every attractor, run by groups of lanes and spread over the whole GPU: each pass
        # sheds the envs that finish, so the next one runs fewer envs per warp in wider, faster groups) and a last pass to the
        # end; () = one launch does everything.  "auto" (default) sizes the first pass to the workload: (b, 8b) with b the
        # smallest of 32, 64, 128, 256 within which at least half of the envs finish their env.step — 32 when most envs need a
        # few updates (Bittner-28: median 6, however heavy the tail), 256 when they need hundreds (Bittner-200 on its real
        # attractor; the lockstep pass moves 2x the updates per instruction the lane groups do).  The counts come from the
        # previous steps' update counts, read back asynchronously every 16th step (no synchronisation; every plan gives the
        # same results)
        self.plan_budgets = "auto"
        self._auto = {"b": 32, "steps": 0, "host": None, "event": None}
        self.running = None   # bool [B]: envs whose env.step is unfinished (budgeted stepping)
        self._work = None     # int32 [2 * (B + 4)]: the two parking lists
        self._plan_phase = 0
        self._plan_draws = None

    # ---- draws
    def reseed(self, seed):
        self.seed, self.epoch = int(seed) & 0xFFFFFFFFFFFFFFFF, 0

    def _draws(self, replay=None):
        if replay is not None:
            return replay.struct()
        d = abi.PbnDraws(mode=abi.DRAW_PHILOX, seed=self.seed, epoch=self.epoch & 0xFFFFFFFF)
        self.epoch += 1
        return d

    # ---- state in / out
    def set_state(self, bits):
        """bits: uint8/bool [B][N] (host array or tensor)."""
        t = torch.as_tensor(np.ascontiguousarray(np.asarray(bits, dtype=np.uint8)) if not torch.is_tensor(bits) else bits)
        t = t.to(self.device, dtype=torch.uint8).reshape(self.B, self.net.n).contiguous()
        with torch.cuda.device(self.device):
            abi.check(abi.lib().pbn_pack_state(_ptr(t), self.B, self.net.n, _ptr(self.state), _stream()))
            self.launches += 1

    def unpack(self, planes=None, out=None):
        """uint8 [B][N] device tensor of the packed planes (default: the live state)."""
        planes = self.state if planes is None else planes
        if out is None:
            out = torch.empty((self.B, self.net.n), dtype=torch.uint8, device=self.device)
        with on_device(self.device):
            abi.check(abi.lib().pbn_unpack_state(_ptr(planes), self.B, self.net.n, _ptr(out), _stream()))
        self.launches += 1
        return out

    # ---- kernels
    def rand_state(self, replay=None):
        d = self._draws(replay)
        with torch.cuda.device(self.device):
            abi.check(abi.lib().pbn_rand_state(self.net.handle, _ptr(self.state), self.B, self.env0, C.byref(d), _stream()))
            self.launches += 1

    def rollout(self, steps, sync=False, replay=None):
        """sync: False = asynchronous updates, True = Graph.synch_step per env, "sliced" = the same law computed for 32 envs
        at a time on bit-sliced words (predictor networks with <= 5 predictors per node, Philox draws only)."""
        d = self._draws(replay)
        mode = 2 if sync == "sliced" else int(bool(sync))
        with torch.cuda.device(self.device):
            abi.check(abi.lib().pbn_rollout(self.net.handle, _ptr(self.state), self.B, self.env0, int(steps), mode,
                                            C.byref(d), _stream()))
            self.launches += 1

    def _plan_buffers(self):
        if self.running is None:
            self.running = torch.zeros(self.B, dtype=torch.bool, device=self.device)
            self._work = torch.zeros(2 * (self.B + 4), dtype=torch.int32, device=self.device)

    def _plan_call(self, env, actions, d, budget, resume, vec=None):
        self._plan_buffers()
        plan = abi.PbnStepPlan(running=_ptr(self.running), work=_ptr(self._work), budget=int(budget), resume=int(resume),
                               phase=self._plan_phase)
        self._plan_phase ^= 1  # the next call reads the list this one wrote
        with torch.cuda.device(self.device):
            abi.check(abi.lib().pbn_env_step_plan(
                env.handle, _ptr(self.state), _ptr(self.n_steps), _ptr(self.target_att), _ptr(actions), actions.shape[1],
                _ptr(self.obs_state), _ptr(self.reward), _ptr(self.terminated), _ptr(self.truncated), _ptr(self.inner),
                C.byref(vec) if vec is not None else None, C.byref(plan), self.B, self.env0, C.byref(d), _stream()))
            self.launches += 1

    def _plannable(self, env, replay):
        return (replay is None and env.kind in (abi.ENV_TARGET, abi.ENV_MULTI) and env.n_att > 0 and not env.force
                and len(self._passes(env)) > 1)

    def _auto_poll(self):
        a = self._auto
        if a["event"] is None or torch.cuda.is_current_stream_capturing():
            return
        if a["event"].query():  # a finished read-back: update the first-pass budget
            counts = a["host"].tolist()
            a["b"] = next((b for b, c in zip((32, 64, 128), counts) if 2 * c >= self.B), 256)
            a["event"] = None

    def _auto_sample(self):
        """Every 16th planned step: sum of the step's update counts -> pinned host memory, no synchronisation."""
        a = self._auto
        if not isinstance(self.plan_budgets, str):
            return
        a["steps"] += 1
        if a["steps"] % 16 != 1 or a["event"] is not None or torch.cuda.is_current_stream_capturing():
            return
        if a["host"] is None:
            a["host"] = torch.zeros(3, dtype=torch.int64).pin_memory()
            a["thr"] = torch.tensor([[32], [64], [128]], dtype=torch.int32, device=self.device)
        a["host"].copy_((self.inner.unsqueeze(0) <= a["thr"]).sum(1), non_blocking=True)  # envs done within 32 / 64 / 128 updates
        a["event"] = torch.cuda.Event()
        a["event"].record()

    def _passes(self, env):
        """Budgets of the passes of one full env.step: plan_budgets as far as the cap can exceed them, then 0 (to the end)."""
        out, spent = [], 0
        budgets = self.plan_budgets
        if isinstance(budgets, str):
            # a lockstep round costs ~1 us whatever the batch (a lane's update is a ~2000-cycle chain; the pass is efficient
            # only when the GPU is full of lanes), a group's update 0.03-0.07 us: small batches skip the lockstep pass (one
            # launch, group mode), medium ones keep it short
            if self.B <= 8192:
                budgets = ()
            else:
                self._auto_poll()
                b = self._auto["b"] if self.B >= 65536 else 32
                budgets = (b, 8 * b)
        for b in budgets:
            b = max(int(b), 2)
            if spent + b >= env.max_inner:
                break
            out.append(b)
            spent += b
        return out + [0]

    def env_step(self, env: EnvImage, actions, replay=None, budget=None):
        """actions: int32 device tensor [B] or [B][K].  Results land in self.reward / terminated / truncated / inner /
        obs_state (overwritten by the next call).

        budget (step-until-attractor envs, Philox draws): at most that many updates per env in this launch; envs still
        outside every attractor are parked (self.running) and go on with env_step_resume — any split gives the result of
        the unsplit step, bit for bit.  budget=None runs the step to its end."""
        actions = actions.to(self.device, dtype=torch.int32).reshape(self.B, -1).contiguous()
        d = self._draws(replay)
        if budget is not None or self._plannable(env, replay):
            self._plan_draws, self._plan_actions = d, actions
            if budget is not None:
                self._plan_call(env, actions, d, budget, 0)
            else:
                for k, b in enumerate(self._passes(env)):
                    self._plan_call(env, actions, d, b, int(k > 0))
                self._auto_sample()
            return
        if env.kind in (abi.ENV_PBN_ST, abi.ENV_PBCN_ST):  # discounted float64 reward (self.reward_f64), interval in self.inner
            if getattr(self, "reward_f64", None) is None:
                self.reward_f64 = torch.zeros(self.B, dtype=torch.float64, device=self.device)
            with torch.cuda.device(self.device):
                abi.check(abi.lib().pbn_env_step_f64(
                    env.handle, _ptr(self.state), _ptr(self.n_steps), _ptr(self.target_att), _ptr(actions), actions.shape[1],
                    _ptr(self.obs_state), _ptr(self.reward), _ptr(self.reward_f64), _ptr(self.terminated), _ptr(self.truncated),
                    _ptr(self.inner), self.B, self.env0, C.byref(d), _stream()))
                self.launches += 1
            return
        with torch.cuda.device(self.device):
            abi.check(abi.lib().pbn_env_step(env.handle, _ptr(self.state), _ptr(self.n_steps), _ptr(self.target_att),
                                             _ptr(actions), actions.shape[1], _ptr(self.obs_state), _ptr(self.reward),
                                             _ptr(self.terminated), _ptr(self.truncated), _ptr(self.inner), self.B,
                                             self.env0, C.byref(d), _stream()))
            self.launches += 1

    def env_step_resume(self, env: EnvImage, budget=0):
        """Continues the envs a budgeted env_step (or env_step_resume) left running; budget=0 runs them to the end."""
        if self._plan_draws is None:
            raise abi.PbnError("env_step_resume without a budgeted env_step")
        self._plan_call(env, self._plan_actions, self._plan_draws, budget, 1)

    def vec_step(self, env: EnvImage, actions, ep_return, ep_len, stats, final_obs=None, autoreset=True, curriculum=None,
                 epoch_dev=None, epoch_base=None, return_sum_f64=None):
        """Fused vector-env step (one launch): env.step for every env + episode bookkeeping + statistics + reset of the envs
        that finished.  Consumes two epochs (step, reset) exactly like env_step followed by a masked env_reset."""
        if actions.dtype != torch.int32 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(self.device, dtype=torch.int32).contiguous()
        K = actions.numel() // self.B
        key = (env.handle.value, ep_return.data_ptr(), final_obs.data_ptr() if final_obs is not None else 0, bool(autoreset),
               tuple(self._passes(env)), curriculum[0].data_ptr() if curriculum else 0)
        c = self._vec_cache
        if c is None or c["key"] != key:  # the buffers never move: build the argument block once
            d, rd = abi.PbnDraws(mode=abi.DRAW_PHILOX), abi.PbnDraws(mode=abi.DRAW_PHILOX)
            v = abi.PbnVecState(ep_return=_ptr(ep_return), ep_len=_ptr(ep_len), stats=_ptr(stats), final_obs=_ptr(final_obs),
                                target_state=_ptr(self.target_state), autoreset=int(bool(autoreset)))
            if env.kind in (abi.ENV_PBN_ST, abi.ENV_PBCN_ST):  # float64 reward / return (ep_return is a float64 tensor here)
                if getattr(self, "reward_f64", None) is None:
                    self.reward_f64 = torch.zeros(self.B, dtype=torch.float64, device=self.device)
                v.ep_return, v.ep_return_f64 = None, _ptr(ep_return)
                v.reward_f64, v.return_sum_f64 = _ptr(self.reward_f64), _ptr(return_sum_f64)
            if curriculum:  # (probabilities float64 [B][A], pair_ids int32 [B][2], sample_pair)
                v.probabilities, v.pair_ids, v.sample_pair = _ptr(curriculum[0]), _ptr(curriculum[1]), int(bool(curriculum[2]))
            head = (env.handle, _ptr(self.state), _ptr(self.n_steps), _ptr(self.target_att))
            tail = (_ptr(self.obs_state), _ptr(self.reward), _ptr(self.terminated), _ptr(self.truncated), _ptr(self.inner))
            c = self._vec_cache = {"key": key, "d": d, "v": v, "head": head, "tail": tail, "fn": abi.lib().pbn_vec_step}
            if self._plannable(env, None):  # budgeted start, resume passes (see env_step)
                self._plan_buffers()
                c["plans"] = [abi.PbnStepPlan(running=_ptr(self.running), work=_ptr(self._work), budget=b, resume=int(k > 0), phase=k & 1)
                              for k, b in enumerate(self._passes(env))]
                c["fn2"] = abi.lib().pbn_env_step_plan
                if autoreset and len(c["plans"]) > 1:
                    # A step of several passes resets its finished envs in ONE masked launch after the last pass instead of
                    # inside the passes: in group mode the lane that finishes an env would otherwise run the reset (pair
                    # sampling, wildcard bits, state write-back) alone while the other envs of its warp wait for it.
                    # Same draws (reset_draws, the step's second epoch), same result as the fused reset.
                    c["v_nr"] = abi.PbnVecState.from_buffer_copy(v)
                    c["v_nr"].autoreset = 0
                    c["rd"] = rd
                    c["mask"] = torch.zeros(self.B, dtype=torch.bool, device=self.device)
                    c["cur"] = curriculum
        d, v = c["d"], c["v"]
        d.seed = v.reset_draws.seed = self.seed
        v.reset_draws.mode = abi.DRAW_PHILOX
        if epoch_dev is not None:  # CUDA-graph capture: the epoch is epoch_base + a counter in device memory (int32 [1])
            d.epoch, v.reset_draws.epoch = epoch_base & 0xFFFFFFFF, (epoch_base + 1) & 0xFFFFFFFF
            d.epoch_dev = v.reset_draws.epoch_dev = _ptr(epoch_dev)
        else:
            d.epoch, v.reset_draws.epoch = self.epoch & 0xFFFFFFFF, (self.epoch + 1) & 0xFFFFFFFF
            d.epoch_dev = v.reset_draws.epoch_dev = None
        self.epoch += 2
        with on_device(self.device):
            stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            if "plans" in c:
                vv = c.get("v_nr", v)
                for plan in c["plans"]:
                    rc = c["fn2"](*c["head"], C.c_void_p(actions.data_ptr()), K, *c["tail"], C.byref(vv), C.byref(plan), self.B,
                                  self.env0, C.byref(d), stream)
                    if rc:
                        abi.check(rc)
                    self.launches += 1
                if "v_nr" in c:
                    rd, mask, cur = c["rd"], c["mask"], c["cur"]
                    rd.seed, rd.epoch, rd.epoch_dev = v.reset_draws.seed, v.reset_draws.epoch, v.reset_draws.epoch_dev
                    torch.bitwise_or(self.terminated, self.truncated, out=mask)
                    if cur:
                        rc = abi.lib().pbn_env_reset_cur(env.handle, _ptr(self.state), _ptr(self.n_steps), _ptr(self.target_att),
                                                         _ptr(self.target_state), _ptr(mask), _ptr(cur[0]), _ptr(cur[1]),
                                                         int(bool(cur[2])), self.B, self.env0, C.byref(rd), stream)
                    else:
                        rc = abi.lib().pbn_env_reset(env.handle, _ptr(self.state), _ptr(self.n_steps), _ptr(self.target_att),
                                                     _ptr(self.target_state), _ptr(mask), self.B, self.env0, C.byref(rd), stream)
                    if rc:
                        abi.check(rc)
                    torch.where(mask, self.state, self.obs_state, out=self.obs_state)  # reset envs observe their new state
                    self.launches += 1
                self._auto_sample()
                return
            rc = c["fn"](*c["head"], C.c_void_p(actions.data_ptr()), K, *c["tail"], C.byref(v), self.B, self.env0, C.byref(d), stream)
            if rc:
                abi.check(rc)
            self.launches += 1

    def env_reset(self, env: EnvImage, mask=None, replay=None, curriculum=None):
        """curriculum = (probabilities float64 [B][A], pair_ids int32 [B][2], sample_pair): PBNTargetMultiEnv draws its
        attractor pair from the env's own probability row (pbn_target_multi.py:232-235)."""
        if mask is not None:
            mask = mask.to(self.device, dtype=torch.uint8).contiguous()
        d = self._draws(replay)
        if curriculum:
            with torch.cuda.device(self.device):
                abi.check(abi.lib().pbn_env_reset_cur(env.handle, _ptr(self.state), _ptr(self.n_steps), _ptr(self.target_att),
                                                      _ptr(self.target_state), _ptr(mask), _ptr(curriculum[0]), _ptr(curriculum[1]),
                                                      int(bool(curriculum[2])), self.B, self.env0, C.byref(d), _stream()))
                self.launches += 1
            return
        with torch.cuda.device(self.device):
            abi.check(abi.lib().pbn_env_reset(env.handle, _ptr(self.state), _ptr(self.n_steps), _ptr(self.target_att),
                                              _ptr(self.target_state), _ptr(mask), self.B, self.env0, C.byref(d), _stream()))
            self.launches += 1

    def ssd(self, iters, bit_flip_prob, tgt_nodes, env: EnvImage = None, hist=None, replay=None):
        """Accumulates the visit histogram of B chains x iters iterations into hist (int64 [2^g], device)."""
        tgt = np.ascontiguousarray(tgt_nodes, np.int32)
        g = len(tgt)
        if hist is None:
            hist = torch.zeros(1 << g, dtype=torch.int64, device=self.device)
        d = self._draws(replay)
        with torch.cuda.device(self.device):
            abi.check(abi.lib().pbn_ssd(self.net.handle, env.handle if env is not None else None, _ptr(self.state), self.B,
                                        self.env0, int(iters), float(bit_flip_prob), _np_ptr(tgt), g, _ptr(hist),
                                        C.byref(d), _stream()))
            self.launches += 1
        return hist


def bucket_hist(sim: "Simulator", tgt_nodes, hist):
    """hist[bucket(state_e)] += 1 for every env of `sim` (target-node bits, first node most significant)."""
    tgt = np.ascontiguousarray(tgt_nodes, np.int32)
    with torch.cuda.device(sim.device):
        abi.check(abi.lib().pbn_bucket_hist(_ptr(sim.state), sim.B, sim.net.n, _np_ptr(tgt), len(tgt), _ptr(hist), _stream()))
        sim.launches += 1
    return hist


def attractor_index(sim_or_state, env_image: EnvImage, out=None):
    """int32 [B] device tensor: index of the first attractor of `env_image` with a cube containing each env's state, -1 if
    none.  sim_or_state: a Simulator (its live state) or packed state planes int32 [W32][B] on the image's device."""
    state = sim_or_state.state if isinstance(sim_or_state, Simulator) else sim_or_state
    net = env_image.net
    if state.dim() != 2 or state.shape[0] != net.w32 or state.dtype != torch.int32 or state.device != net.device:
        raise ValueError(f"state must be int32 planes [{net.w32}][B] on {net.device}")
    state = state.contiguous()
    B = state.shape[1]
    if out is None:
        out = torch.empty(B, dtype=torch.int32, device=net.device)
    elif out.shape != (B,) or out.dtype != torch.int32 or out.device != net.device or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous int32 tensor [{B}] on {net.device}")
    with on_device(net.device):
        abi.check(abi.lib().pbn_env_attractor_index(env_image.handle, _ptr(state), B, _ptr(out), _stream()))
    if isinstance(sim_or_state, Simulator):
        sim_or_state.launches += 1
    return out


def issue_peak(kind, iters=2000):
    """(ops/s) of the instruction-issue microbenchmarks: kind 0 = INT ALU ops, kind 1 = Philox4x32-10 blocks."""
    ms, ops = C.c_float(), C.c_double()
    abi.check(abi.lib().pbn_issue_peak(kind, iters, C.byref(ms), C.byref(ops)))
    return ops.value / (ms.value * 1e-3), ms.value
