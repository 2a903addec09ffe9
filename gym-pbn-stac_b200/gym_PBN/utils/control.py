"""Attractor-level control of the target envs.

One env.step of `PBNTargetEnv` flips one gene and then updates until the state lies in some attractor, and the reward
depends only on which attractor that is.  The env's dynamics therefore come down to one table: for source attractor `a`
and action `i`, the probability of ending the step in attractor `b`.  CABEAN, the tool the reference hands attractor
detection to (utils/get_attractors_from_cabean.py), solves source-target control on the same abstraction.

  attractor_transitions      estimates that table on the GPU (env.step kernels + pbn_env_attractor_index)
  attractor_policy           value iteration on the estimated attractor-level MDP (host, NumPy)
  evaluate_attractor_policy  runs a policy table on the real PBNVectorEnv: the Monte-Carlo truth for its prediction

Permanent control holds genes at fixed values instead (structural interventions: knockout = 0, overexpression = 1), or
blocks or forces single regulatory interactions (edge pins: the target gene's function reads a constant for one input):

  pinned_ssd                 steady-state histograms of the network under many pin sets at once (pbn_ssd_pinned_edges)
  rank_pins                  every single-gene knockout and overexpression, ranked by the SSD mass it moves onto
                             env.target_node_values (the measure of utils.eval.eval_increase)
  regulatory_edges           the (src, dst) pairs of the network: src is read by some function of dst
  rank_edge_pins             every single-edge pin (src -> dst read as 0, as 1), ranked the same way
  first_passage              how many iterations each chain needs to reach a set of target-gene patterns under each pin
                             set (pbn_first_passage); rank_pins / rank_edge_pins(measure="passage") rank pins by it
"""
import numpy as np
import torch

from gym_PBN.b200 import abi, engine
from gym_PBN.b200 import dist as pdist


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


def _node_index(env, net, node):
    """A node index, or a gene id of the env's graph (resolved as target_node_indices does)."""
    ids = env.graph.getIDs() if env is not None and hasattr(getattr(env, "graph", None), "getIDs") else None
    if ids is not None and node in ids:
        return ids.index(node)
    if isinstance(node, (int, np.integer)) and 0 <= int(node) < net.n:
        return int(node)
    raise ValueError(f"{node!r} is neither a gene id of the env nor a node index in [0, {net.n})")


def _env_and_net(env_or_network):
    """(env or None, engine.Network) of pinned_ssd's and first_passage's first argument."""
    env = None if isinstance(env_or_network, engine.Network) else getattr(env_or_network, "unwrapped", env_or_network)
    return env, (env_or_network if env is None else env.network)


def _pin_masks(env, net, pins):
    """The launch arguments of a list of pin sets (pinned_ssd's `pins`): care, value uint32 [K][W32] and edges uint32 [K][E]
    (None when no set pins an edge)."""
    pins = list(pins)
    K = len(pins)
    if not 1 <= K <= 65535:
        raise ValueError("1 <= len(pins) <= 65535 pin sets")
    care = np.zeros((K, net.w32), np.uint32)
    value = np.zeros((K, net.w32), np.uint32)
    rows, known = [], None
    for k, pin in enumerate(pins):
        row = []
        for node, v in dict(pin).items():
            if v not in (0, 1):
                raise ValueError(f"pinned values are 0 or 1, got {v!r}")
            if isinstance(node, tuple) and len(node) == 2:
                src, dst = (_node_index(env, net, x) for x in node)
                if known is None:
                    known = set(_edge_nodes(net.spec))
                if (src, dst) not in known:
                    raise ValueError(f"{node!r} is not a regulatory edge (src, dst) of the network: no function of "
                                     f"{node[1]!r} reads {node[0]!r}")
                row.append(dst | src << 12 | int(v) << 24)
                continue
            i = _node_index(env, net, node)
            care[k, i >> 5] |= np.uint32(1 << (i & 31))
            value[k, i >> 5] |= np.uint32(int(v) << (i & 31))
        rows.append(row)
    E = max(len(r) for r in rows)
    if E > 64:
        raise ValueError(f"at most 64 edge pins per pin set, got {E}")
    edges = None
    if E:
        edges = np.full((K, E), 0xFFFFFFFF, np.uint32)
        for k, row in enumerate(rows):
            edges[k, :len(row)] = row
    return care, value, edges


def pinned_ssd(env_or_network, pins, iters, chains, bit_flip_prob=0.01, target_nodes=None, seed=0, distributed=False):
    """Visit histograms of the target-gene patterns under each pin set of `pins`, from one launch per iteration chunk.

    env_or_network: an env (its network; target_nodes default to env.target_node_indices) or an engine.Network.
    pins: list of {node: 0 or 1} dicts, node = node index or gene id (Bittner envs); {} = the network unpinned.
    A variant holds its pinned nodes at their values: they are set before the first iteration, an update that picks one
    leaves it as it is, and perturbations skip it.  A key (src, dst), both ends resolved as node keys are, pins that edge
    of regulatory_edges: whenever dst is updated its function reads the pinned value in place of src (src itself, and every
    other node that reads it, are unchanged); a pair that is not an edge raises ValueError.  Up to 64 edge pins per
    variant; truth-table networks with more than 16 KB of threshold table take none.  Otherwise every iteration is the one
    of utils.eval.ssd_histogram without an env: count the pattern, flip each gene w.p. bit_flip_prob, one asynchronous
    update (include/pbn_b200.h: pbn_ssd_pinned_edges).  Every variant starts from the same uniform random states (Graph.genRandState) and runs on the same
    random numbers, so differences between rows are not drowned in independent sampling noise, and the row of {} is
    utils.eval.ssd_histogram's estimate for those start states.  With distributed=True chains are sharded over ranks by
    global chain id (multiples of 32) and the histograms are summed.

    Returns int64 [K][2^g] (NumPy), bucket = target-node bits, first target most significant; each row sums to
    iters * chains."""
    from gym_PBN.utils.eval import MAX_ITERS_PER_LAUNCH

    env, net = _env_and_net(env_or_network)
    if target_nodes is None:
        if env is None:
            raise ValueError("target_nodes are needed with a bare network")
        target_nodes = env.target_node_indices
    tgt = np.asarray([_node_index(env, net, t) for t in target_nodes], np.int32)
    care, value, edges = _pin_masks(env, net, pins)
    K = care.shape[0]
    start, stop = pdist.shard_range(chains, align=32) if distributed else (0, int(chains))
    local = stop - start
    hist = torch.zeros((K, 1 << len(tgt)), dtype=torch.int64, device=net.device)
    if local > 0:
        sim = engine.Simulator(net, local, seed=seed, env0=start)
        with engine.on_device(net.device):
            sim.rand_state()
            state = sim.state.repeat(1, K)  # column k * local + c: chain c of variant k, one start per chain
            left = int(iters)
            while left > 0:
                chunk = min(left, MAX_ITERS_PER_LAUNCH)
                engine.ssd_pinned(sim, state, chunk, bit_flip_prob, tgt, care, value, hist, edges=edges)
                left -= chunk
    if distributed:
        pdist.allreduce_sum_(hist)
    return hist.cpu().numpy()


def goal_words(patterns, g):
    """The goal mask of pbn_first_passage for a list of target-gene patterns (g values 0/1 each, first target most
    significant, as env.target_node_values holds them): uint32 [max(1, 2^g / 32)], bit b set for every pattern's bucket b."""
    words = np.zeros(max(1, (1 << g) // 32), np.uint32)
    for b in _bucket_ids(patterns, g, "goal patterns"):
        words[b >> 5] |= np.uint32(1 << (b & 31))
    return words


def first_passage(env_or_network, pins, iters, chains, goal=None, start=None, bit_flip_prob=0.01, target_nodes=None, seed=0,
                  distributed=False):
    """First-passage times into the goal patterns of the target genes, for each pin set of `pins` (pinned_ssd's keys: node,
    gene id or (src, dst) edge) on common random numbers.

    An iteration is pinned_ssd's (look at the pattern, flip each gene w.p. bit_flip_prob, one asynchronous update) with the
    count replaced by a test: a chain whose pattern lies in `goal` at iteration t has first-passage time t and stops.  So 0
    means the start state, with its pins applied, is already there; -1 means the goal was not reached within `iters`.
    goal: list of patterns of the target genes (default env.target_node_values), at most 12 target genes.
    start: None = the env's reset states (a uniform attractor, a uniform cube of it) when it has at least two attractors,
    otherwise uniform random states (Graph.genRandState), as utils.eval.ssd_histogram chooses; or a uint8 [chains][N] array.
    Every variant starts chain c from the same state.  Launches run MAX_ITERS_PER_LAUNCH iterations at most and stop once
    every chain has arrived.  With distributed=True chains are sharded over ranks by global chain id (multiples of 32) and
    every rank gets the whole table.

    Returns {"time": int64 [K][chains] (NumPy, -1 = not reached), "source": int64 [chains], the attractor index of each
    reset start (pbn_env_attractor_index, -1 = none), or None for other starts}."""
    from gym_PBN.utils.eval import MAX_ITERS_PER_LAUNCH

    env, net = _env_and_net(env_or_network)
    if target_nodes is None:
        if env is None:
            raise ValueError("target_nodes are needed with a bare network")
        target_nodes = env.target_node_indices
    tgt = np.asarray([_node_index(env, net, t) for t in target_nodes], np.int32)
    if goal is None:
        if env is None:
            raise ValueError("a goal is needed with a bare network")
        goal = env.target_node_values
    words = goal_words(goal, len(tgt))
    care, value, edges = _pin_masks(env, net, pins)
    K, chains, iters = care.shape[0], int(chains), int(iters)
    image = getattr(env, "env_image", None) if start is None else None
    reset = image is not None and image.n_att >= 2
    if start is not None:
        start = np.asarray(start, np.uint8)
        if start.shape != (chains, net.n):
            raise ValueError(f"start must be uint8 [{chains}][{net.n}], got shape {start.shape}")
    lo, hi = pdist.shard_range(chains, align=32) if distributed else (0, chains)
    local = hi - lo
    time = torch.zeros((K, chains), dtype=torch.int64, device=net.device)  # t + 1 on this rank's chains, 0 elsewhere
    source = torch.zeros(chains, dtype=torch.int64, device=net.device)     # attractor index + 1 likewise
    if local > 0:
        sim = engine.Simulator(net, local, seed=seed, env0=lo)
        with engine.on_device(net.device):
            if start is not None:
                sim.set_state(start[lo:hi])
            elif reset:
                sim.env_reset(image)
                source[lo:hi] = engine.attractor_index(sim, image).long() + 1
            else:
                sim.rand_state()
            state = sim.state.repeat(1, K)  # column k * local + c: chain c of variant k
            t_hit = torch.full((K, local), -1, dtype=torch.int64, device=net.device)
            t0 = 0
            while t0 < iters and bool((t_hit < 0).any()):
                chunk = min(iters - t0, MAX_ITERS_PER_LAUNCH)
                engine.first_passage(sim, state, chunk, t0, bit_flip_prob, tgt, words, care, value, t_hit, edges=edges)
                t0 += chunk
            time[:, lo:hi] = t_hit + 1
    if distributed:
        pdist.allreduce_sum_(time)
        pdist.allreduce_sum_(source)
    return {"time": (time - 1).cpu().numpy(), "source": (source - 1).cpu().numpy() if reset else None}


def _bucket_ids(patterns, g, what):
    """Histogram buckets of target-gene patterns (first target most significant)."""
    out = []
    for p in patterns or ():
        if len(p) != g or any(b not in (0, 1) for b in p):
            raise ValueError(f"{what} must hold patterns of {g} target-gene values 0/1, got {p!r}")
        out.append(int("".join(str(int(b)) for b in p), 2))
    return out


def _rank(env, pins, rows, iters, chains, bit_flip_prob, seed, measure="ssd"):
    """The ranking of rank_pins and rank_edge_pins: pins[0] = {} and pins[k] the variant of rows[k - 1] (the identifying
    fields of its ranking entry), all estimated on common random numbers by one pinned_ssd (measure "ssd") or
    first_passage (measure "passage") run.  The passage fields: "reached" = the fraction of chains that arrived,
    "mean_time" = the restricted mean mean(min(T, iters)) (a chain that did not arrive counts as iters), "change" =
    mean_time minus the unpinned one; fastest first."""
    if measure == "passage":
        t = first_passage(env, pins, iters, chains, bit_flip_prob=bit_flip_prob, seed=seed)["time"]
        reached = (t >= 0).mean(1)
        mean_time = np.where(t >= 0, np.minimum(t, iters), iters).mean(1)
        ranking = [dict(row, reached=float(reached[k]), mean_time=float(mean_time[k]),
                        change=float(mean_time[k] - mean_time[0])) for k, row in enumerate(rows, start=1)]
        ranking.sort(key=lambda r: r["change"])
        return {"unpinned": {"reached": float(reached[0]), "mean_time": float(mean_time[0])}, "ranking": ranking}
    if measure != "ssd":
        raise ValueError(f'measure is "ssd" or "passage", got {measure!r}')
    hist = pinned_ssd(env, pins, iters, chains, bit_flip_prob=bit_flip_prob, seed=seed).astype(np.float64)
    mass = hist / hist.sum(1, keepdims=True)
    g = len(env.target_node_indices)
    good = _bucket_ids(env.target_node_values, g, "env.target_node_values")
    bad = _bucket_ids(env.undesired_node_values, g, "env.undesired_node_values")
    tm, um = mass[:, good].sum(1), mass[:, bad].sum(1)
    ranking = [dict(row, target_mass=float(tm[k]), undesired_mass=float(um[k]), increase=float(tm[k] - tm[0]))
               for k, row in enumerate(rows, start=1)]
    ranking.sort(key=lambda r: -r["increase"])
    return {"unpinned": {"target_mass": float(tm[0]), "undesired_mass": float(um[0])}, "ranking": ranking}


def rank_pins(env, genes=None, iters=4000, chains=300, bit_flip_prob=0.01, seed=0, measure="ssd"):
    """Every single-gene pin (gene -> 0, gene -> 1) of `genes` (gene ids or node indices; default every node), ranked by the
    change of steady-state mass on env.target_node_values against the unpinned network: eval_increase's measure, with the
    pin in place of a controller.  One pinned_ssd launch estimates all 1 + 2 * len(genes) variants on common random numbers;
    the default budget is the reference's (1.2e6 iterations per SSD: 300 chains x 4000).

    Returns {"unpinned": {"target_mass", "undesired_mass"}, "ranking": [...]}: one dict per pin with "gene" (id or index as
    given), "node" (index), "value", "target_mass", "undesired_mass" (mass on env.undesired_node_values) and "increase"
    (target_mass minus the unpinned one), best first.

    measure="passage" ranks by how fast the pin gets there instead: first_passage (from the env's reset states) into
    env.target_node_values, `iters` iterations at most, all variants in one run.  Each dict then has "reached" (fraction of
    chains that got there), "mean_time" (mean of min(T, iters), a chain that did not get there counting as iters) and
    "change" (mean_time minus the unpinned one) in place of the mass fields, fastest first; "unpinned" has "reached" and
    "mean_time"."""
    env = getattr(env, "unwrapped", env)
    net = env.network
    if genes is None:
        genes = list(env.graph.getIDs()) if hasattr(getattr(env, "graph", None), "getIDs") else list(range(net.n))
    genes = list(genes)
    pins = [{}] + [{g: v} for g in genes for v in (0, 1)]
    rows = [{"gene": g, "node": _node_index(env, net, g), "value": v} for g in genes for v in (0, 1)]
    return _rank(env, pins, rows, iters, chains, bit_flip_prob, seed, measure)


def _edge_nodes(spec):
    """The distinct (src, dst) node-index pairs of a compiled network, in (dst, input slot) order: src is an input of some
    predictor of dst (its three regulators and dst itself), or of dst's truth table."""
    a, out, seen = spec.arrays, [], set()
    for dst in range(spec.n):
        if "pr_in" in a:
            srcs = a["pr_in"][4 * a["pr_off"][dst]:4 * a["pr_off"][dst + 1]]
        else:
            srcs = a["tt_in"][a["tt_in_off"][dst]:a["tt_in_off"][dst + 1]]
        for src in srcs:
            e = (int(src), dst)
            if e not in seen:
                seen.add(e)
                out.append(e)
    return out


def regulatory_edges(env_or_network):
    """The regulatory edges of a network: every distinct pair (src, dst) such that some function of node dst reads node src
    (for predictor networks each predictor reads three regulators and dst itself, so every node has its self-input), in
    (dst, input slot) order.  env_or_network: an env (pairs of gene ids when its graph has them, node indices otherwise), an
    engine.Network or a compiler.NetworkSpec (node indices)."""
    if isinstance(env_or_network, engine.Network):
        env, spec = None, env_or_network.spec
    elif hasattr(env_or_network, "arrays") and hasattr(env_or_network, "n"):
        env, spec = None, env_or_network
    else:
        env = getattr(env_or_network, "unwrapped", env_or_network)
        spec = env.network.spec
    edges = _edge_nodes(spec)
    ids = env.graph.getIDs() if env is not None and hasattr(getattr(env, "graph", None), "getIDs") else None
    return [(ids[s], ids[d]) for s, d in edges] if ids is not None else edges


def rank_edge_pins(env, edges=None, iters=4000, chains=300, bit_flip_prob=0.01, seed=0, measure="ssd"):
    """Every single-edge pin ((src, dst) -> 0, -> 1) of `edges` ((src, dst) pairs of gene ids or node indices; default
    regulatory_edges(env), self-inputs included), ranked as rank_pins ranks gene pins: by the change of steady-state mass
    on env.target_node_values against the unpinned network.  Pinning (src, dst) at c makes dst's function read c in place
    of src, and leaves src and every other reader of src as they are: it blocks (or forces) one interaction where a gene
    pin removes all of the gene's.  One pinned_ssd launch estimates all 1 + 2 * len(edges) variants on common random
    numbers (at most 65 535 variants).

    Returns {"unpinned": {"target_mass", "undesired_mass"}, "ranking": [...]}: one dict per edge pin with "src", "dst" (as
    given), "src_node", "dst_node" (indices), "value", "target_mass", "undesired_mass" and "increase", best first.
    measure="passage" ranks them by first-passage time, with rank_pins' passage fields."""
    env = getattr(env, "unwrapped", env)
    net = env.network
    edges = regulatory_edges(env) if edges is None else [tuple(e) for e in edges]
    pins = [{}] + [{e: v} for e in edges for v in (0, 1)]
    rows = [{"src": s, "dst": d, "src_node": _node_index(env, net, s), "dst_node": _node_index(env, net, d), "value": v}
            for s, d in edges for v in (0, 1)]
    return _rank(env, pins, rows, iters, chains, bit_flip_prob, seed, measure)
