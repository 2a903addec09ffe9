"""First-passage times on Bittner-100: the cost of the goal test against the count, and a real pin screen.

1. Worst case: all 201 variants of rank_pins (unpinned + every gene pinned at 0 and at 1) x `--chains` chains x `--iters`
   iterations, the seven melanoma target genes, p = 0.01, with an EMPTY goal, so that no chain stops and no warp leaves its
   loop early.  pbn_first_passage then does the work of pbn_ssd_pinned_edges on the same chains with a goal test in place
   of the histogram count, and the ratio of the two rates prices that test.  The two launches alternate in one run, timed
   with CUDA events, and a 256 MB buffer is zeroed before every timed launch so that neither finds its state columns in
   the 126 MB L2; median of `--reps`.
2. Real screen: control.rank_pins(env, measure="passage") on the Bittner-100 env, from its reset states, into
   env.target_node_values, capped at `--cap` iterations: the wall time of the call (ending in a device synchronise), the
   time of its k_passage kernels (torch.profiler, in a second call of its own), and the warp-iterations the kernels
   executed, computed from the returned times: per warp of 32 chains, the largest time of its lanes + 1, or the cap when a
   lane did not arrive (a warp leaves when all its lanes have arrived, checked once per two iterations on the static
   path, so this is a lower bound by less than one iteration per warp).

The card's name, power limit and clock are read in the same run.  Also reports the static SASS of the hot loop of
k_ssd_pinned and k_passage (cuobjdump of the built library).

    python tools/passage_bench.py [--chains 5216] [--iters 9600] [--reps 5] [--cap 100000] [--screen-chains 300] [--out FILE]
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gym-pbn-stac_b200"))
sys.path.insert(0, str(ROOT / "tools"))

from pinned_ssd_bench import card, static_loop_counts  # noqa: E402

NET, P = "100_5_kmeans", 0.01
HOT = {"k_ssd_pinned": "_Z12k_ssd_pinnedILi1ELi1EEv7NetView8DrawView9SsdParamsPjxxiPyPKjS6_jS6_i",
       "k_passage": "_Z9k_passageILi1ELi1EEv7NetView8DrawView9SsdParamsPjxxixPxPKjS6_jS6_i8GoalMask"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=5216)  # x 201 variants = 1 048 416 chains, about bench.py's 2^20
    ap.add_argument("--iters", type=int, default=9600)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cap", type=int, default=100000)
    ap.add_argument("--screen-chains", type=int, default=300)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    import gym_PBN
    from gym_PBN.b200 import abi, compiler, engine
    from gym_PBN.utils import control

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    net = engine.Network(compiler.load_bittner(NET))
    tgt = np.arange(7, dtype=np.int32)  # compile order puts the seven target genes first
    pins = [{}] + [{i: v} for i in range(net.n) for v in (0, 1)]
    K = len(pins)
    care, value, _ = control._pin_masks(None, net, pins)
    empty = np.zeros(4, np.uint32)

    sp = engine.Simulator(net, a.chains, seed=1)
    sp.rand_state()
    s_pinned = sp.state.repeat(1, K)
    sg = engine.Simulator(net, a.chains, seed=1)
    sg.rand_state()
    s_goal = sg.state.repeat(1, K)
    hist = torch.zeros((K, 128), dtype=torch.int64, device="cuda")
    t_hit = torch.full((K, a.chains), -1, dtype=torch.int64, device="cuda")
    flush = torch.empty(64 << 20, dtype=torch.int32, device="cuda")

    def run(which):
        if which == "pinned":
            engine.ssd_pinned(sp, s_pinned, a.iters, P, tgt, care, value, hist)
        else:
            engine.first_passage(sg, s_goal, a.iters, 0, P, tgt, empty, care, value, t_hit)

    for w in ("pinned", "passage"):  # warm-up: module load, gap-shortcut verification
        run(w)
    times = {"pinned": [], "passage": []}
    for _ in range(a.reps):
        for w in ("pinned", "passage"):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(w)
            e1.record()
            e1.synchronize()
            times[w].append(e0.elapsed_time(e1) * 1e-3)
    total = K * a.chains * a.iters
    rate = {w: total / float(np.median(t)) for w, t in times.items()}
    same = bool(torch.equal(s_pinned, s_goal)) and bool((t_hit == -1).all().item())

    # 2. the real screen
    env = gym_PBN.make("gym-PBN/Bittner-100-v0").unwrapped
    res = control.first_passage(env, [{}], 10, 64, seed=9)  # warm-up of the env's image and kernels
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ranked = control.rank_pins(env, iters=a.cap, chains=a.screen_chains, seed=9, measure="passage")
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = control.first_passage(env, [{}] + [{g: v} for g in env.graph.getIDs() for v in (0, 1)], a.cap,
                                    a.screen_chains, seed=9)
        torch.cuda.synchronize()
    kern = [e for e in prof.key_averages() if "k_passage" in e.key]
    kernel_s = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0)) for e in kern) * 1e-6
    T = res["time"]
    C = T.shape[1]
    warp_iters = 0
    for w0 in range(0, C, 32):
        tw = T[:, w0:w0 + 32]
        warp_iters += int(np.where((tw < 0).any(1), a.cap, tw.max(1) + 1).sum())
    out = {
        "card": card(),
        "worst_case": {
            "workload": f"Bittner-100, 7 targets, p = {P}, empty goal, K = {K} variants x {a.chains} chains x {a.iters} "
                        f"iterations, L2 flushed before each timed launch, median of {a.reps}",
            "iters_per_s": {"pbn_first_passage": rate["passage"], "pbn_ssd_pinned_edges": rate["pinned"]},
            "ratio": rate["passage"] / rate["pinned"],
            "seconds": times,
            "final_states_equal": same,
        },
        "screen": {
            "workload": f"rank_pins(measure='passage') on Bittner-100, {K} variants x {a.screen_chains} chains from reset "
                        f"states, goal = target_node_values, cap {a.cap}, p = {P}",
            "wall_s": wall,
            "k_passage_s": kernel_s,
            "k_passage_launches": int(sum(e.count for e in kern)),
            "warp_iterations": warp_iters,
            "warp_iterations_cap": K * ((C + 31) // 32) * a.cap,
            "unpinned": ranked["unpinned"],
            "fastest": ranked["ranking"][:5],
            "same_as_ranked": bool(abs(ranked["unpinned"]["mean_time"] - np.where(T[0] >= 0, np.minimum(T[0], a.cap), a.cap).mean()) < 1e-9),
        },
        "static_sass_per_iter": {k: static_loop_counts(abi.LIB_PATH, fn)[0] for k, fn in HOT.items()},
        "static_sass_round_loops": {k: static_loop_counts(abi.LIB_PATH, fn)[1] for k, fn in HOT.items()},
    }
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
