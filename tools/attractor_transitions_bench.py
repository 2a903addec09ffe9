"""Timings of the attractor-control path, printed as one JSON line together with the card they were measured on.

  * wall time of gym_PBN.utils.control.attractor_transitions at `--samples` steps per (attractor, action) cell for
    Bittner-28 (its two exact attractors, 29 actions) and Bittner-100 (its verified attractors, 101 actions);
  * CUDA-event time of pbn_env_attractor_index (engine.attractor_index) on 2^20 Bittner-100 envs, and its share of one
    env.step of the same envs.

    python tools/attractor_transitions_bench.py [--samples 10000] [--out FILE]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "gym-pbn-stac_b200"))

import torch  # noqa: E402

import gym_PBN  # noqa: E402
from gym_PBN.b200 import abi, engine  # noqa: E402
from gym_PBN.utils.control import attractor_transitions  # noqa: E402


def card():
    """Name and power limit of the GPU this process runs on."""
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                        f"--id={torch.cuda.current_device()}"], capture_output=True, text=True)
    name, _, limit = q.stdout.strip().partition(",")
    return {"gpu": name.strip() or torch.cuda.get_device_name(), "power_limit": limit.strip() or "unknown"}


def wall(env, samples):
    attractor_transitions(env, 10, num_envs=4096)  # loads the kernels, sizes the allocator
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    counts = attractor_transitions(env, samples)  # ends in a device-to-host copy of the counts
    return time.perf_counter() - t0, counts


def event_ms(fn, reps):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=10_000)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    res = card()
    atts28 = [[tuple(c) for c in a] for a in json.loads((ROOT / "tests" / "golden" / "b28_exact_attractors.json").read_text())]
    b28 = gym_PBN.make("gym-PBN/Bittner-28-v0", all_attractors=atts28).unwrapped
    b100 = gym_PBN.make("gym-PBN/Bittner-100-v0", seed=1).unwrapped  # the verified route (pbn_target.py: default_attractors)
    for name, env in (("bittner28", b28), ("bittner100", b100)):
        s, counts = wall(env, args.samples)
        res[name] = {"attractors": counts.shape[0], "actions": counts.shape[1], "samples_per_cell": args.samples,
                     "env_steps": int(counts.sum()), "cap_hits": int(counts[..., -1].sum()), "wall_s": round(s, 3),
                     "env_steps_per_s": round(counts.sum() / s)}
    B = 1 << 20
    image = engine.EnvImage(b100.network, abi.ENV_TARGET, attractors=b100.all_attractors, max_inner=b100.max_inner_steps)
    sim = engine.Simulator(b100.network, B, seed=3)
    sim.env_reset(image)
    out = torch.empty(B, dtype=torch.int32, device=sim.device)
    acts = torch.randint(0, b100.network.n + 1, (B,), dtype=torch.int32, device=sim.device)
    index_ms = event_ms(lambda: engine.attractor_index(sim, image, out=out), 200)
    step_ms = event_ms(lambda: sim.env_step(image, acts), 20)  # states drift between steps; the step stays on attractors
    res["attractor_index_2^20"] = {"network": "Bittner-100", "attractors": image.n_att,
                                   "cubes": sum(len(a) for a in b100.all_attractors), "index_ms": round(index_ms, 4),
                                   "env_step_ms": round(step_ms, 4), "share_of_step": round(index_ms / step_ms, 4)}
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
