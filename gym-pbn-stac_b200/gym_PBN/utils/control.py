"""Attractor-level control of the target envs.

One env.step of `PBNTargetEnv` flips one gene and then updates until the state lies in some attractor, and the reward
depends only on which attractor that is.  The env's dynamics therefore come down to one table: for source attractor `a`
and action `i`, the probability of ending the step in attractor `b`.  CABEAN, the tool the reference hands attractor
detection to (utils/get_attractors_from_cabean.py), solves source-target control on the same abstraction.

  attractor_transitions      estimates that table on the GPU (env.step kernels + pbn_env_attractor_index)
  attractor_policy           value iteration on the estimated attractor-level MDP (host, NumPy)
  evaluate_attractor_policy  runs a policy table on the real PBNVectorEnv: the Monte-Carlo truth for its prediction
"""
import numpy as np
import torch

from gym_PBN.b200 import abi, engine


def _target_env(env, multi_ok):
    from gym_PBN.envs.pbn_target import PBNTargetEnv
    from gym_PBN.envs.pbn_target_multi import PBNTargetMultiEnv

    env = getattr(env, "unwrapped", env)
    if not isinstance(env, PBNTargetEnv) or (not multi_ok and isinstance(env, PBNTargetMultiEnv)):
        raise TypeError(f"expected {'a PBNTargetEnv or PBNTargetMultiEnv' if multi_ok else 'a PBNTargetEnv'}, "
                        f"got {type(env).__name__}")
    if len(env.all_attractors) < 2:
        raise ValueError("the env needs at least two attractors (env.all_attractors)")
    return env


def attractor_transitions(env, samples, seed=0, num_envs=None, force=False):
    """Counts of where one env.step takes each attractor under each single-gene intervention.

    env: a PBNTargetEnv or PBNTargetMultiEnv (gymnasium wrappers are unwrapped) with at least two attractors.  The step is
    the target env's: flip gene i-1 (action 0 = no flip), one asynchronous update, then updates until the state matches a
    cube of env.all_attractors or env.max_inner_steps updates were made.  A one-slot action of the multi env runs the same
    step.  force=True (exactly one update per step) ends steps outside every attractor and is rejected.

    Start states are drawn as PBNTargetEnv.reset draws them: a uniform attractor, a uniform cube of it, uniform bits for
    its wildcards.  Each start is classified (pbn_env_attractor_index) to give `a`, and actions are dealt out per source
    attractor in turn, so that every (a, i) cell gets about the same number of steps; rounds of `num_envs` envs repeat until
    every cell has at least `samples`.  Round r uses Philox epochs 2r (reset) and 2r + 1 (step) of `seed`: results are
    deterministic for a given seed and num_envs.

    Returns int64 counts [A][N+1][A+1]: [a][i][b] = steps started in attractor a with action i that ended in attractor b
    (the first attractor with a matching cube); column A = steps that hit max_inner_steps outside every attractor."""
    if force:
        raise ValueError("force=True makes an env.step exactly one update, which in general ends outside every attractor")
    env = _target_env(env, multi_ok=True)
    samples = int(samples)
    if samples < 1:
        raise ValueError("samples must be >= 1")
    net = env.network
    A, n_act = len(env.all_attractors), net.n + 1
    image = engine.EnvImage(net, abi.ENV_TARGET, attractors=env.all_attractors, horizon=env.horizon,
                            max_inner=env.max_inner_steps)
    B = int(num_envs) if num_envs else min(A * n_act * samples, 1 << 20)
    if B < 1:
        raise ValueError("num_envs must be >= 1")
    dev = net.device
    sim = engine.Simulator(net, B, seed=seed)
    counts = torch.zeros(A * n_act * (A + 1), dtype=torch.int64, device=dev)
    offset = torch.zeros(A, dtype=torch.int64, device=dev)  # next action to deal to each source attractor
    ids = torch.arange(B, dtype=torch.int64, device=dev)
    rank = torch.empty(B, dtype=torch.int64, device=dev)
    with engine.on_device(dev):
        while True:
            sim.env_reset(image)
            a = engine.attractor_index(sim, image).long()  # >= 0: the reset state lies in a cube of its attractor
            per = torch.bincount(a, minlength=A)
            order = torch.argsort(a, stable=True)
            rank[order] = ids - (torch.cumsum(per, 0) - per)[a[order]]  # position of env e among the envs starting in a
            act = (offset[a] + rank) % n_act
            offset = (offset + per) % n_act
            sim.env_step(image, act.to(torch.int32))
            b = engine.attractor_index(sim, image).long()
            b = torch.where(b < 0, A, b)
            counts += torch.bincount((a * n_act + act) * (A + 1) + b, minlength=counts.numel())
            if int(counts.view(A, n_act, A + 1).sum(2).min()) >= samples:
                break
    return counts.view(A, n_act, A + 1).cpu().numpy()


def attractor_policy(counts, target, horizon):
    """Best attractor-level policy for reaching attractor `target` within `horizon` env.steps (value iteration, host).

    The MDP is the one `counts` estimates (attractor_transitions): P(b | a, i) = counts[a][i][b] / sum_b' counts[a][i][b'].
    Ending a step in the cap column (outside every attractor) counts as failure; an (a, i) cell without any count never
    succeeds.  Ties (within 1e-12) go to the lowest action index.

    Assumption: an attractor-level policy sees only which attractor the env is in, not its state.  This is exact when every
    attractor is a single state; otherwise the landing law of a step also depends on the state inside the source attractor,
    and the result is a baseline (the best a policy that observes only attractors can do if the env's occupancy of each
    attractor follows the start distribution of attractor_transitions).

    Returns (action, success), both [horizon + 1][A]: with k steps left in attractor a, action[k][a] is the action to take
    and success[k][a] the largest probability of being in `target` after at most k more steps.  success[k][target] = 1
    and action[k][target] = 0 (already there); row 0 has no steps left."""
    c = np.asarray(counts)
    if c.ndim != 3 or c.shape[2] != c.shape[0] + 1 or c.shape[1] < 1 or (c < 0).any():
        raise ValueError("counts must be non-negative [A][N+1][A+1]")
    A = c.shape[0]
    target, horizon = int(target), int(horizon)
    if not 0 <= target < A:
        raise ValueError(f"target must be an attractor index in [0, {A})")
    if horizon < 0:
        raise ValueError("horizon must be >= 0")
    c = c.astype(np.float64)
    tot = c.sum(2, keepdims=True)
    P = np.divide(c[:, :, :A], tot, out=np.zeros_like(c[:, :, :A]), where=tot > 0)  # the cap column carries no value
    success = np.zeros((horizon + 1, A))
    action = np.zeros((horizon + 1, A), np.int64)
    success[0, target] = 1.0
    for k in range(1, horizon + 1):
        q = P @ success[k - 1]  # [A][N+1]
        best = q.max(1)
        action[k] = np.argmax(q >= best[:, None] - 1e-12, axis=1)
        success[k] = best
        success[k, target], action[k, target] = 1.0, 0
    return action, success


def evaluate_attractor_policy(env, action_table, target, episodes, seed=0):
    """Monte-Carlo run of an attractor-level policy on the real env (PBNVectorEnv, `episodes` envs, no autoreset).

    env: a PBNTargetEnv with at least two attractors (not the multi env, whose reset always starts in its first attractor).
    Episodes start from the env's reset, a uniform attractor; horizon H = len(action_table) - 1.
    Before each step every env's state is classified (pbn_env_attractor_index) and the env takes
    action_table[steps_left][its attractor].  An episode succeeds when a step ends in attractor `target` (or it starts there)
    and fails when a step hits max_inner_steps outside every attractor (the policy has no action for such a state, and
    attractor_policy counts it as failure) or H steps pass.

    Returns (success rate, mean env.steps per episode until success or the end of the episode)."""
    from gym_PBN.b200.vector_env import PBNVectorEnv

    env = _target_env(env, multi_ok=False)
    A = len(env.all_attractors)
    table = np.asarray(action_table)
    if table.ndim != 2 or table.shape[1] != A or table.shape[0] < 1:
        raise ValueError(f"action_table must be [H + 1][{A}]")
    if not ((0 <= table) & (table <= env.network.n)).all():
        raise ValueError(f"actions must lie in [0, {env.network.n}]")
    target, episodes = int(target), int(episodes)
    if not 0 <= target < A:
        raise ValueError(f"target must be an attractor index in [0, {A})")
    H = table.shape[0] - 1
    vec = PBNVectorEnv(env, num_envs=episodes, seed=seed, autoreset=False, obs="packed")
    table = torch.as_tensor(table, dtype=torch.int32, device=vec.device)
    with engine.on_device(vec.device):
        vec.reset()
        cls = engine.attractor_index(vec.sim, vec.image)
        reached = cls == target
        failed = torch.zeros_like(reached)
        steps = torch.zeros(episodes, dtype=torch.int64, device=vec.device)
        for t in range(H):
            live = ~(reached | failed)
            act = torch.where(live, table[H - t][cls.clamp(min=0).long()], 0)
            vec.step(act.view(-1, 1))
            steps += live
            engine.attractor_index(vec.sim, vec.image, out=cls)
            reached |= live & (cls == target)
            failed |= live & (cls < 0)
        return float(reached.double().mean()), float(steps.double().mean())
