"""Rate of pbn_ssd_pinned_edges against pbn_ssd on the single-gene or the single-edge screen of Bittner-100.

Workload: Bittner-100 (100_5_kmeans), the seven melanoma target genes, p = 0.01, and `--chains` chains per variant of
  --screen genes  all 201 variants of rank_pins (unpinned + every gene pinned at 0 and at 1), or
  --screen edges  all 1 921 variants of rank_edge_pins (unpinned + each of the 960 regulatory edges pinned at 0 and at 1).
The reference is pbn_ssd on the same total chain count (K * chains) and the same iterations: the pinned launch does the same
work, so the ratio of the two rates is the cost of pinning.  The two launches alternate in one run, timed with CUDA events,
and a 256 MB buffer is zeroed before every timed launch so that neither finds its state columns in the 126 MB L2.  The
card's name and power limit are read in the same run.

Also reports the static SASS of the hot loop of both kernels (cuobjdump of the built library): the instructions of the
static predictor loop body per iteration, and of the body that draws a perturbation round.

    python tools/pinned_ssd_bench.py [--screen genes|edges] [--chains N] [--iters 9600] [--reps 5] [--out FILE]
"""
import argparse
import json
import re
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "gym-pbn-stac_b200"))

NET, P = "100_5_kmeans", 0.01
HOT = {"k_ssd": "_Z5k_ssdILi1ELi0ELi1ELb0EEv7NetView7EnvView8DrawView9SsdParamsPjxxiPy",
       "k_ssd_pinned": "_Z12k_ssd_pinnedILi1ELi1EEv7NetView8DrawView9SsdParamsPjxxiPyPKjS6_jS6_i"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def static_loop_counts(lib, fn):
    """(instructions per iteration of the static loop, instructions of its round-drawing loop) of kernel `fn`: the static
    predictor loop is the backward-branch loop with two bucket counts (BREV) and the most shared-memory atomics; it runs two
    iterations per trip, and the perturbation rounds are the loops nested in it."""
    txt = subprocess.run(["cuobjdump", "-sass", "-fun", fn, str(lib)], capture_output=True, text=True).stdout
    ins = []
    for line in txt.splitlines():
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(2)))
    loops = []
    for a, t in ins:
        m = re.search(r"\bBRA\b.*0x([0-9a-f]+)", t)
        if m and int(m.group(1), 16) < a:
            lo = int(m.group(1), 16)
            body = [x for b, x in ins if lo <= b <= a]
            loops.append((lo, a, len(body), sum("BREV" in x for x in body), sum("ATOMS" in x for x in body)))
    outer = max((l for l in loops if l[3] == 2), key=lambda l: l[4])
    inner = [l for l in loops if outer[0] <= l[0] and l[1] < outer[1]]
    return (outer[2] - sum(l[2] for l in inner)) / 2, [l[2] for l in inner]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--screen", choices=("genes", "edges"), default="genes")
    # default: 5216 x 201 variants = 1 048 416 chains, about the 2^20 of bench.py; 512 x 1921 = 983 552 (a variant's last
    # block holds chains % 256 of them: 546 chains, the nearest count to 2^20, leaves a third of the blocks a ninth full)
    ap.add_argument("--chains", type=int, default=None)
    ap.add_argument("--iters", type=int, default=9600)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch

    from gym_PBN.b200 import abi, compiler, engine
    from gym_PBN.utils import control

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    net = engine.Network(compiler.load_bittner(NET))
    tgt = np.arange(7, dtype=np.int32)  # compile order puts the seven target genes first
    edges = None
    if a.screen == "genes":
        pins = [{}] + [{i: v} for i in range(net.n) for v in (0, 1)]
    else:
        pins = [{}] * (1 + 2 * len(control.regulatory_edges(net)))
        edges = np.full((len(pins), 1), 0xFFFFFFFF, np.uint32)
        edges[1:, 0] = [d | s << 12 | v << 24 for s, d in control.regulatory_edges(net) for v in (0, 1)]
    K = len(pins)
    if a.chains is None:
        a.chains = 5216 if a.screen == "genes" else 512
    care, value = np.zeros((K, net.w32), np.uint32), np.zeros((K, net.w32), np.uint32)
    for k, pin in enumerate(pins):
        for i, v in pin.items():
            care[k, i >> 5] |= np.uint32(1 << (i & 31))
            value[k, i >> 5] |= np.uint32(v << (i & 31))

    pinned = engine.Simulator(net, a.chains, seed=1)
    pinned.rand_state()
    state = pinned.state.repeat(1, K)
    plain = engine.Simulator(net, K * a.chains, seed=1)
    plain.rand_state()
    hp = torch.zeros((K, 128), dtype=torch.int64, device="cuda")
    hu = torch.zeros(128, dtype=torch.int64, device="cuda")
    flush = torch.empty(64 << 20, dtype=torch.int32, device="cuda")

    def run(which):
        if which == "pinned":
            engine.ssd_pinned(pinned, state, a.iters, P, tgt, care, value, hp, edges=edges)
        else:
            plain.ssd(a.iters, P, tgt, hist=hu)

    for w in ("pinned", "plain"):  # warm-up: module load, gap-shortcut verification
        run(w)
    times = {"pinned": [], "plain": []}
    for _ in range(a.reps):
        for w in ("plain", "pinned"):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(w)
            e1.record()
            e1.synchronize()
            times[w].append(e0.elapsed_time(e1) * 1e-3)
    total = K * a.chains * a.iters
    rate = {w: total / float(np.median(t)) for w, t in times.items()}
    lib = abi.LIB_PATH
    sass = {k: static_loop_counts(lib, fn) for k, fn in HOT.items()}
    out = {
        "card": card(),
        "workload": f"Bittner-100, 7 targets, p = {P}, {a.screen} screen, K = {K} variants x {a.chains} chains x {a.iters} iterations "
                    f"(pbn_ssd: {K * a.chains} chains), L2 flushed before each timed launch, median of {a.reps}",
        "iters_per_s": {"pbn_ssd_pinned_edges": rate["pinned"], "pbn_ssd": rate["plain"]},
        "ratio": rate["pinned"] / rate["plain"],
        "seconds": times,
        "static_sass_per_iter": {k: v[0] for k, v in sass.items()},
        "static_sass_round_loops": {k: v[1] for k, v in sass.items()},
        "rows_sum_ok": bool((hp.sum(1) == (1 + a.reps) * a.chains * a.iters).all().item()),
    }
    line = json.dumps(out)
    print(line)
    if a.out:
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
