#!/usr/bin/env python
"""bench.py — the BASELINE.json workloads on N B200s, one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W]              # headline: configs[2], Bittner-100 SSD estimation
    python bench.py --config {2,4,5} ...                             # the env.step configurations (parity cases with numbers)
    python bench.py --impl reference [--config C] ...                # CPU arm: the oracle port on all host cores (+ the
                                                                     #   Python reference per core when baseline/_ref is staged)
    torchrun --nproc-per-node N ... bench.py --gpus N ...            # N > 1: one rank per GPU, NCCL
    python bench.py ... --dump-outputs DIR                           # + what the last timed step computed, DIR/<name>.npy

--config 3 (default; BASELINE.json configs[2], SURVEY.md §8d): gym-PBN/Bittner-100 steady-state-distribution estimate —
2^20 chains per GPU, each step advances every chain by 9600 SSD iterations (histogram the 7 target genes, flip each gene
w.p. 0.01, one asynchronous node update = one env.step(0) under the all-attracting fixture); one step = the 1.0e10-iteration
estimate of configs[2].  value = SSD iterations (= env-steps) per second over all ranks, WEAK scaling (2^20 chains per GPU, the
128-bucket histogram all-reduced over NCCL every step).  The same line carries the STRONG-scaling number (`strong`: the one
1.0e10-iteration estimate sharded over the N ranks by global chain id) and a cross-N result check (`cross_n_check`: a fixed
small estimate computed sharded + all-reduced and, on rank 0, unsharded — the two histograms must be equal, and the checksum
must be the same at every N).

--config 2 / 4 / 5: one step = one vector env.step (+ auto-reset) of every env: Bittner-28 PBN-target-v0 with its exact
attractors (65 536 envs per GPU), Bittner-200 PBN-target_multi-v0 on its sampled + verified (closed) attractors (131 072 envs
per GPU, K = 3 actions), synthetic PBCN N = 1024 sampled-data with intervals ~ U{1..64} (262 144 envs per GPU).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "gym-pbn-stac_b200"))

NET_NAME = "100_5_kmeans"
TARGET_NODES = list(range(7))  # genes 234237..130057 are nodes 0..6 of the shipped set (pbn_target.py:447)
CHAINS_PER_GPU = 1 << 20
ITERS_PER_STEP = 9600  # 2^20 chains x 9600 = 1.0066e10 iterations: one step = one full SSD estimate per GPU
FLIP_P = 0.01
SEED = 0
METRIC = "bittner100_env_steps_per_s"
UNIT = "env-steps/s"
SURVEY_INSTR_PER_UPDATE = 150.0  # SURVEY.md §8d: algorithmic thread-instructions per asynchronous micro-step
DUMP_SAMPLE = 8192  # chains / envs whose state --dump-outputs writes (a fixed seeded sample: config 5 alone has 2^28 state bits)
DUMP_LIMIT = 64 << 20


def workload_config(n_gpus):
    return {
        "workload": f"gym-PBN/Bittner-100 SSD estimation ({NET_NAME}): {CHAINS_PER_GPU} chains/GPU x {ITERS_PER_STEP} "
                    f"iterations/step, bit_flip_prob={FLIP_P}, 7 target genes (128 buckets), async update, all-attracting",
        "chains_per_gpu": CHAINS_PER_GPU, "iters_per_step": ITERS_PER_STEP, "update": "async",
        "rng": "philox4x32-10", "parallelism": f"env-sharded x{n_gpus}", "l2": "flushed between timed steps (256 MiB write)",
    }


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 7 for k in range(4) if r[3 + k].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def dump_outputs(out_dir, sim, planes, arrays):
    """--dump-outputs: writes out_dir/<name>.npy for every device tensor in `arrays` (whole) and, for every packed state in
    `planes`, the 0/1 node values of the same DUMP_SAMPLE chains (seeded, sorted ids) as float32 [sample][n].  Integer
    results are stored as float64, which holds every count the workloads reach exactly."""
    import torch

    pick = np.sort(np.random.default_rng(0).choice(sim.B, min(sim.B, DUMP_SAMPLE), replace=False))
    idx = torch.from_numpy(pick).to(sim.device)
    arrays = dict(arrays, **{name: sim.unpack(p).index_select(0, idx) for name, p in planes.items()})
    host = {}
    for name, t in arrays.items():
        a = t.cpu().numpy()
        host[name] = a.astype(np.float32 if a.dtype.itemsize < 4 or a.dtype == np.float32 else np.float64)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte limit")
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in host.items():
        np.save(out / f"{name}.npy", a)


# ------------------------------------------------------------------------------------------------ env.step workloads
class EnvWorkload:
    """configs 2 / 4 / 5: B envs per GPU, one step = one fused vector env.step (+ auto-reset where the env has one)."""

    def __init__(self, config):
        self.config = config

    def describe(self, n_gpus):
        c = self.config
        if c == 2:
            d = {"workload": "gym-PBN/Bittner-28-v0 PBN-target-v0 (28_15_median) with its exact attractors (120 + 49152 states), "
                             "65536 lockstep envs per GPU, random flip actions, horizon 100, inner cap 4096, step + auto-reset",
                 "envs_per_gpu": 65536}
        elif c == 4:
            d = {"workload": "gym-PBN/Bittner-200 (199 nodes, 200_5_kmeans) PBN-target_multi-v0, sampled + verified (closed) "
                             "attractor cubes, 131072 envs per GPU, K=3 node flips per action, inner cap 4096, step + auto-reset",
                 "envs_per_gpu": 131072}
        else:
            d = {"workload": "synthetic PBCN N=1024 (3 inputs, 2 functions per node, 8 control nodes) PBCN-sampled-data-v0, "
                             "262144 envs per GPU, interval ~ U{1..64}, control='write'", "envs_per_gpu": 262144}
        d.update({"update": "async", "rng": "philox4x32-10", "parallelism": f"env-sharded x{n_gpus}",
                  "l2": "flushed between timed steps (256 MiB write)"})
        return d

    @property
    def metric(self):
        return {2: "bittner28_target_env_steps_per_s", 4: "bittner200_multi_env_steps_per_s", 5: "pbcn1024_sampled_env_steps_per_s"}[self.config]

    def envs(self):
        return {2: 65536, 4: 131072, 5: 262144}[self.config]

    # ---- product side
    def build(self, dev, rank):
        import torch

        from gym_PBN.b200 import abi, attractors, compiler, engine
        from gym_PBN.b200.synthetic import synthetic_pbcn

        B = self.envs()
        g = torch.Generator().manual_seed(100 + rank)
        self.fixture = {}
        if self.config == 2:
            net = engine.Network(compiler.load_bittner("28_15_median"), device=dev)
            atts = attractors.exact_attractor_cubes(net)
            env = engine.EnvImage(net, abi.ENV_TARGET, attractors=atts, horizon=100, max_inner=4096)
            acts = [torch.randint(0, 29, (B, 1), generator=g, dtype=torch.int32) for _ in range(8)]
            self.fixture = {"attractors": "exact (device search over 2^28 states)", "attractor_states": [120, 49152]}
        elif self.config == 4:
            net = engine.Network(compiler.load_bittner("200_5_kmeans"), device=dev)
            atts, info = attractors.verified_attractors(net, resets=512, seed=0)
            if len(atts) < 1:
                raise SystemExit("config 4 needs an attractor; the sampled + verified route found none")
            env = engine.EnvImage(net, abi.ENV_MULTI, attractors=atts, horizon=100, max_inner=4096, dedup=True)
            acts = [torch.randint(0, net.n + 1, (B, 3), generator=g, dtype=torch.int32) for _ in range(8)]
            self.fixture = {"attractors": "sampled + verified trap spaces (closed under every update)",
                            "attractor_free_nodes": [i["free"] for i in info]}
        else:
            net = engine.Network(compiler.compile_pbn_data(synthetic_pbcn()), device=dev)
            rng = np.random.default_rng(0)
            targets = [tuple(int(v) for v in rng.integers(0, 2, 1024)) for _ in range(4)]
            env = engine.EnvImage(net, abi.ENV_PBCN_SD, attractors=[[t] for t in targets], targets=targets[:1], n_control=8,
                                  control_write=True)
            acts = [torch.cat([torch.randint(1, 65, (B, 1), generator=g), torch.randint(0, 2, (B, 8), generator=g)], 1).to(torch.int32)
                    for _ in range(8)]
        self.net, self.env, self.B = net, env, B
        self.sim = engine.Simulator(net, B, seed=SEED, env0=rank * B)
        self.acts_host = [a.pin_memory() for a in acts]
        self.acts_dev = [a.to(dev) for a in acts]
        self.ep_return = torch.zeros(B, dtype=torch.int64, device=dev)
        self.ep_len = torch.zeros(B, dtype=torch.int32, device=dev)
        self.stats = torch.zeros(8, dtype=torch.int64, device=dev)
        self.final_obs = torch.zeros_like(self.sim.state)
        self.inner_sum = torch.zeros((), dtype=torch.int64, device=dev)
        if self.config == 5:
            self.sim.rand_state()
        else:
            self.sim.env_reset(env)
        self.out_host = torch.empty(B, dtype=torch.int32).pin_memory()
        self.flag_host = torch.empty(B, dtype=torch.bool).pin_memory()

    def step(self, k, count_inner=True):
        sim = self.sim
        if self.config == 5:  # no episode end to reset on: the sampled-data env has no attractor loop
            sim.env_step(self.env, self.acts_dev[k % 8])
        else:
            sim.vec_step(self.env, self.acts_dev[k % 8], self.ep_return, self.ep_len, self.stats, final_obs=self.final_obs)
        if count_inner:
            self.inner_sum += sim.inner.sum()

    def step_e2e(self, k):
        """Host actions up (pinned), the step, rewards + terminated flags back to the host."""
        a = self.acts_host[k % 8].to(self.sim.device, non_blocking=True)
        sim = self.sim
        if self.config == 5:
            sim.env_step(self.env, a)
        else:
            sim.vec_step(self.env, a, self.ep_return, self.ep_len, self.stats, final_obs=self.final_obs)
        self.out_host.copy_(sim.reward, non_blocking=True)
        self.flag_host.copy_(sim.terminated, non_blocking=True)

    def e2e_bytes(self):
        return int(self.acts_host[0].numel() * 4), int(self.B * 5)

    # ---- CPU arm: the oracle port (test infrastructure; bench.py may time it, nothing else may use it)
    def cpu_sample(self, target_seconds):
        sys.path.insert(0, str(ROOT / "oracle"))
        os.environ["OMP_NUM_THREADS"] = os.environ.get("PBN_BENCH_THREADS", str(os.cpu_count() or 1))
        import oracle as orc

        from gym_PBN.b200.synthetic import synthetic_pbcn

        rng = np.random.default_rng(1)
        cores = orc.num_threads()
        if self.config == 2:
            sets, ids = orc.load_bittner("28_15_median")
            onet = orc.net_from_predictor_sets(sets, ids)
            atts = json.loads((ROOT / "tests" / "golden" / "b28_exact_attractors.json").read_text())
            atts = [[tuple(v if v != "*" else "*" for v in c) for c in a] for a in atts]
            oenv = orc.Env(orc.ENV_TARGET, 28, attractors=atts, horizon=100, max_inner=4096)
            n, width, hi = 28, 1, 29
        elif self.config == 4:
            sets, ids = orc.load_bittner("200_5_kmeans")
            onet = orc.net_from_predictor_sets(sets, ids)
            atts = json.loads((ROOT / "tests" / "golden" / "b200_verified_attractors.json").read_text())
            atts = [[tuple(v if v != "*" else "*" for v in c) for c in a] for a in atts]
            n = len(atts[0][0])
            oenv = orc.Env(orc.ENV_MULTI, n, attractors=atts, horizon=100, max_inner=4096, dedup=1)
            width, hi = 3, n + 1
        else:
            onet = orc.net_from_pbn_data(synthetic_pbcn())
            n = 1024
            targets = [tuple(int(v) for v in np.random.default_rng(0).integers(0, 2, n)) for _ in range(4)]
            oenv = orc.Env(orc.ENV_PBCN_SD, n, attractors=[[t] for t in targets], targets=targets[:1], n_control=8, control_write=1)
            width, hi = 9, None
        Bs = 2048 * cores

        def one(Bc, epoch):
            st, ns, ta = np.zeros((Bc, n), np.uint8), np.zeros(Bc, np.int32), np.zeros(Bc, np.int32)
            if self.config == 5:
                st[:] = rng.integers(0, 2, size=(Bc, n))
                st[:, 0] = 0
                act = np.concatenate([rng.integers(1, 65, (Bc, 1)), rng.integers(0, 2, (Bc, 8))], 1).astype(np.int32)
            else:
                orc.env_reset(onet, oenv, st, ns, ta, orc.Draws(seed=SEED, epoch=epoch))
                act = rng.integers(0, hi, size=(Bc, width)).astype(np.int32)
            t0 = time.perf_counter()
            orc.env_step(onet, oenv, st, ns, ta, act, orc.Draws(seed=SEED, epoch=epoch + 1))
            return time.perf_counter() - t0

        dt = one(Bs, 0)
        Bc = int(max(cores, min(self.envs(), Bs * target_seconds / max(dt, 1e-6))))
        dt = one(Bc, 2)
        return {"value": Bc / dt, "unit": UNIT, "cores": cores, "kind": "port", "algorithm": "C restatement of the reference's env.step loop, Philox draws, OpenMP over envs",
                "sample": f"one env.step of {Bc} envs of the same workload through oracle/pbn_oracle.c, {dt:.1f} s"}


# ------------------------------------------------------------------------------------------------ CPU arm (config 3)
def cpu_sample(target_seconds=12.0):
    """Times the oracle port (oracle/pbn_oracle.c, OpenMP over chains) on a bounded sample of the same workload."""
    sys.path.insert(0, str(ROOT / "oracle"))
    # all host threads (torchrun pins OMP_NUM_THREADS=1 for its workers; the CPU arm is meant to use every core)
    os.environ["OMP_NUM_THREADS"] = os.environ.get("PBN_BENCH_THREADS", str(os.cpu_count() or 1))
    import oracle as orc

    sets, ids = orc.load_bittner(NET_NAME)
    net = orc.net_from_predictor_sets(sets, ids)
    cores = orc.num_threads()
    tgt = np.array(TARGET_NODES, np.int32)
    # calibrate, then size the sample (chains) for ~target_seconds at the workload's own chain length
    chains = 256 * cores
    st = orc.rand_state(net, chains, orc.Draws(seed=SEED, epoch=0))
    t0 = time.perf_counter()
    orc.ssd(net, None, st, 200, FLIP_P, tgt, orc.Draws(seed=SEED, epoch=1))
    rate = chains * 200 / (time.perf_counter() - t0)
    iters = ITERS_PER_STEP
    chains = int(max(cores, min(CHAINS_PER_GPU, rate * target_seconds / iters)))
    st = orc.rand_state(net, chains, orc.Draws(seed=SEED, epoch=0))
    t0 = time.perf_counter()
    orc.ssd(net, None, st, iters, FLIP_P, tgt, orc.Draws(seed=SEED, epoch=2))
    dt = time.perf_counter() - t0
    return {"value": chains * iters / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "algorithm": "geometric-skip port: the builder's own SSD algorithm (one geometric gap draw instead of N Bernoulli "
                         "draws per iteration), ~1500x faster per core than the Python reference it restates",
            "sample": f"{chains} chains x {iters} iterations of the same Bittner-100 SSD workload, oracle/pbn_oracle.c "
                      f"(C restatement of the pure-Python reference, Philox draws, OpenMP), {dt:.1f} s"}


def reference_python_sample(seconds=10.0):
    """The UNMODIFIED Python reference (staged under baseline/_ref by __graft_entry__.build) timed per host core on this
    box: Graph.step (bittner/base.py:306-312) and the shimmed _ssd_run loop (utils/eval.py:76-103) on the Bittner-100 set,
    one process per core.  Reported beside the port; not the ratio's denominator.  None when the staging is absent."""
    script = ROOT / "baseline" / "time_reference.py"
    if not (ROOT / "baseline" / "_ref" / "gym_PBN").is_dir() or not script.exists():
        return None
    try:
        out = subprocess.run([sys.executable, str(script), "--seconds", str(seconds)], capture_output=True, text=True,
                             timeout=seconds * 4 + 120)
        for line in reversed(out.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        return {"error": (out.stderr or out.stdout)[-300:]}
    except Exception as e:  # the reference arm must never take the bench line down
        return {"error": repr(e)[:300]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    per_step = max(2.0, min(12.0, 60.0 / (steps + args.warmup)))
    wl = EnvWorkload(args.config) if args.config != 3 else None
    sample = (lambda s: wl.cpu_sample(s)) if wl else cpu_sample
    for _ in range(args.warmup):
        sample(per_step)
    vals, t0 = [], time.perf_counter()
    last = None
    for _ in range(steps):
        last = sample(per_step)
        vals.append(last["value"])
    value = float(np.mean(vals))
    last["value"] = value
    if args.config == 3:
        last["reference_python"] = reference_python_sample(10.0)
    line = {"impl": "reference", "metric": METRIC if not wl else wl.metric, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": (time.perf_counter() - t0) * 1e3 / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": workload_config(args.gpus) if not wl else wl.describe(args.gpus), "cpu_baseline": last,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def load_inst_per_iter():
    """Executed thread-level instructions per SSD iteration, measured once with ncu (profiles/); used for the
    issue-rate roofline.  Falls back to a static estimate if the profile summary is absent."""
    p = ROOT / "profiles" / "ssd_inst_per_iter.json"
    if p.exists():
        return json.loads(p.read_text())
    return {"thread_inst_per_iter": None, "source": "absent"}


class Dist:
    def __init__(self):
        import torch

        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        # NCCL may print its version banner on the C-level stdout at its first collective; the contract is ONE JSON line on
        # stdout, so file descriptor 1 points at stderr until the warm-up (which runs the first all-reduce) is over
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        if self.world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=self.dev)

    def restore_stdout(self):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)

    def barrier(self):
        import torch

        if self.world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    def all_reduce(self, t, op=None):
        if self.world > 1:
            import torch.distributed as dist

            dist.all_reduce(t, op=op or dist.ReduceOp.SUM)
        return t

    def max_seconds(self, seconds):
        import torch
        import torch.distributed as dist

        t = torch.tensor([seconds], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            import torch.distributed as dist

            dist.barrier()
            dist.destroy_process_group()


def timed_ssd(D, net, chains_local, env0, steps, tgt, flush, warm=0):
    """K steps of the SSD kernel on this rank's chains: per-step CUDA events around [kernel + all-reduce] (every step writes
    its own histogram row, so no zeroing sits between the kernel and the collective) and around the kernel alone."""
    import torch

    from gym_PBN.b200 import engine

    sim = engine.Simulator(net, max(chains_local, 1), seed=SEED, env0=env0)
    sim.rand_state()
    rows = torch.zeros((steps + warm, 128), dtype=torch.int64, device=D.dev)
    for k in range(warm):
        if chains_local > 0:
            sim.ssd(ITERS_PER_STEP, FLIP_P, tgt, hist=rows[k])
        D.all_reduce(rows[k])
    D.barrier()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    launches0 = sim.launches
    for k in range(steps):
        flush.zero_()
        ev[k][0].record()
        if chains_local > 0:
            sim.ssd(ITERS_PER_STEP, FLIP_P, tgt, hist=rows[warm + k])
        ev[k][1].record()
        D.all_reduce(rows[warm + k])
        ev[k][2].record()
    D.barrier()
    t_steps = sum(e[0].elapsed_time(e[2]) for e in ev) * 1e-3
    t_kernel = sum(e[0].elapsed_time(e[1]) for e in ev) * 1e-3 / steps
    tail_us = sum(e[1].elapsed_time(e[2]) for e in ev) * 1e3 / steps
    return D.max_seconds(t_steps), t_kernel, tail_us, rows, sim.launches - launches0, sim


def cross_n_check(D, net, tgt):
    """A fixed small estimate (2^16 chains x 256 iterations, seed 12345) computed sharded over the ranks + all-reduced and,
    on rank 0, unsharded: the histograms must be equal.  Its checksum must also be the same whatever N is (SCALE file)."""
    import torch

    from gym_PBN.b200 import dist as pdist
    from gym_PBN.b200 import engine

    chains, iters, seed = 1 << 16, 256, 12345

    def run(start, stop):
        h = torch.zeros(128, dtype=torch.int64, device=D.dev)
        if stop > start:
            sim = engine.Simulator(net, stop - start, seed=seed, env0=start)
            sim.rand_state()
            sim.ssd(iters, FLIP_P, tgt, hist=h)
        return h

    start, stop = pdist.shard_range(chains, D.rank, D.world, align=32)
    h = D.all_reduce(run(start, stop))
    out = None
    if D.rank == 0:
        full = run(0, chains)
        out = {"chains": chains, "iters": iters, "seed": seed, "equal_to_one_rank": bool(torch.equal(h, full)),
               "checksum": hashlib.sha256(h.cpu().numpy().tobytes()).hexdigest()[:16]}
        assert out["equal_to_one_rank"], "the N-rank all-reduced histogram differs from the 1-rank histogram"
    return out


def run_gpu_ssd(args):
    import torch

    from gym_PBN.b200 import compiler, engine
    from gym_PBN.b200 import dist as pdist
    from gym_PBN.utils.eval import pack_states, ssd_histogram_host

    D = Dist()
    world, rank, dev = D.world, D.rank, D.dev
    net = engine.Network(compiler.load_bittner(NET_NAME), device=dev)
    tgt = np.array(TARGET_NODES, np.int32)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    warm = max(3, args.warmup)

    # ---- weak scaling (value): 2^20 chains per GPU
    sampler = ClockSampler(D.local)
    t_w, t_kernel, tail_w, rows, launches = None, None, None, None, 0
    # warm-up happens inside timed_ssd before its timed region; stdout is restored after the first collective has run
    sampler.start()
    time.sleep(0.2)
    t_w, t_kernel, tail_w, rows, launches, sim = timed_ssd(D, net, CHAINS_PER_GPU, rank * CHAINS_PER_GPU, args.steps, tgt, flush,
                                                           warm)
    clocks = sampler.stop()
    D.restore_stdout()
    units = float(CHAINS_PER_GPU) * ITERS_PER_STEP * args.steps * world
    value = units / t_w
    assert int(rows.sum().item()) == (warm + args.steps) * CHAINS_PER_GPU * ITERS_PER_STEP * world  # every iteration was histogrammed
    if args.dump_outputs and rank == 0:  # the all-reduced histogram of the last step and the chains' states after it
        dump_outputs(args.dump_outputs, sim, {"state": sim.state}, {"hist": rows[-1]})
    del sim

    # ---- strong scaling: the ONE 1.0e10-iteration estimate (2^20 chains in all) sharded over the ranks by global chain id
    s0, s1 = pdist.shard_range(CHAINS_PER_GPU, rank, world, align=32)
    t_s, t_kernel_s, tail_s, rows_s, _, _ = timed_ssd(D, net, s1 - s0, s0, args.steps, tgt, flush, 1)
    assert int(rows_s.sum().item()) == (1 + args.steps) * CHAINS_PER_GPU * ITERS_PER_STEP
    strong = {"value": float(CHAINS_PER_GPU) * ITERS_PER_STEP * args.steps / t_s, "unit": UNIT, "scaling": "strong",
              "chains_total": CHAINS_PER_GPU, "ms_per_step": t_s * 1e3 / args.steps, "kernel_ms": t_kernel_s * 1e3,
              "allreduce_tail_us": tail_s,
              "note": "one 1.0066e10-iteration estimate per step, chains sharded by dist.shard_range(align=32); the tail is the "
                      "stream-ordered NCCL all-reduce of the int64[128] histogram row the kernel just wrote"}
    check = cross_n_check(D, net, tgt)

    # ---- end-to-end through the public API with HOST buffers (bit-packed start states up, histogram back), every step
    n = net.n
    host_bits = np.random.default_rng(7).integers(0, 2, (CHAINS_PER_GPU, n)).astype(np.uint8)
    host_states = torch.from_numpy(pack_states(host_bits)).pin_memory()  # int32 [4][2^20]: 16 B per chain
    ssd_histogram_host(net, host_states, ITERS_PER_STEP, FLIP_P, tgt, seed=SEED, env0=rank * CHAINS_PER_GPU)  # warm
    D.barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        h = ssd_histogram_host(net, host_states, ITERS_PER_STEP, FLIP_P, tgt, seed=SEED + k, env0=rank * CHAINS_PER_GPU,
                               distributed=(world > 1))
    D.barrier()
    e2e_value = units / D.max_seconds(time.perf_counter() - t0)
    assert int(h.sum()) == CHAINS_PER_GPU * ITERS_PER_STEP * world

    if rank == 0:
        # ---- roofline of the dominant kernel (k_ssd): instruction issue, not HBM (near-zero DRAM traffic by design)
        alu_peak, _ = engine.issue_peak(0, 4000)      # thread-level INT ops/s, measured on this GPU now
        philox_peak, _ = engine.issue_peak(1, 4000)   # Philox4x32-10 blocks/s, measured on this GPU now
        per_launch_iters = float(CHAINS_PER_GPU) * ITERS_PER_STEP
        ipi = load_inst_per_iter()
        tipi = ipi.get("thread_inst_per_iter")
        executed = per_launch_iters * tipi / t_kernel if tipi else None
        algorithmic = SURVEY_INSTR_PER_UPDATE * per_launch_iters / t_kernel
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        state_bytes = per_launch_iters * (8 * 2 + 8)  # SURVEY §8d: 8W read + 8 written per micro-step, W = 2 (uint64 words)
        hbm_alg = (2 * net.w32 * 4 * CHAINS_PER_GPU + 128 * 8)  # bytes that must cross HBM per launch: state in + out, histogram
        roofline = {
            # PRIMARY: ALGORITHMIC work (SURVEY §8d: 150 thread-instructions per asynchronous micro-step) per second against
            # the INT issue peak measured in this run — rises when the kernel gets leaner
            "bound": "issue", "kernel": "k_ssd<PRED,PHILOX>",
            "achieved": algorithmic / 1e9, "peak": alu_peak / 1e9, "unit": "G thread-instr/s", "frac": algorithmic / alu_peak,
            "algorithmic_thread_inst_per_iter": SURVEY_INSTR_PER_UPDATE,
            "peak_source": "pbn_issue_peak(0): dependency-free LOP3+IADD3 chains, measured in this run",
            # issue utilisation of the instructions actually EXECUTED (ncu count in profiles/ssd_inst_per_iter.json): falls when
            # instructions are removed, so it is secondary
            "executed_thread_inst_per_iter": tipi, "inst_source": ipi.get("source"),
            "frac_executed": (executed / alu_peak) if executed else None,
            "kernel_ms": t_kernel * 1e3,
            "iters_per_s_kernel": per_launch_iters / t_kernel,
            "philox_blocks_per_s": 0.75 * per_launch_iters / t_kernel,  # 2 update draws + ~1 gap draw per iteration
            "philox_blocks_per_s_peak": philox_peak, "philox_frac": 0.75 * per_launch_iters / t_kernel / philox_peak,
            "state_bytes_per_s": state_bytes / t_kernel,
            "traffic": ipi.get("dram_bytes_per_launch"),
            "hbm": {"algorithmic_bytes_per_launch": hbm_alg, "achieved_gbs": hbm_alg / t_kernel / 1e9, "peak_gbs": hbm_peak,
                    "frac": hbm_alg / t_kernel / 1e9 / hbm_peak,
                    "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
        }
        cpu = cpu_sample(12.0) if world == 1 else None  # reported on rank 0 at N=1 only
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": t_w * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32", "data": "synthetic", "config": workload_config(world), "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(host_states.numel() * 4),
                        "d2h_bytes_per_step": 128 * 8,
                        "api": "gym_PBN.utils.eval.ssd_histogram_host (pinned bit-packed int32[4][chains] start states up, "
                               "uint64 histogram back)"},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "allreduce_tail_us": tail_w, "strong": strong, "cross_n_check": check,
                "node_updates_per_s": value, "ssd_1e10_seconds": 1.0e10 / value}
        print(json.dumps(line), flush=True)
    D.close()


def run_gpu_env(args):
    import torch

    from gym_PBN.b200 import engine

    D = Dist()
    world, rank, dev = D.world, D.rank, D.dev
    wl = EnvWorkload(args.config)
    wl.build(dev, rank)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    warm = max(3, args.warmup)
    for k in range(warm):
        wl.step(k)
    D.all_reduce(wl.stats.clone())
    D.barrier()
    D.restore_stdout()
    sampler = ClockSampler(D.local)
    sampler.start()
    time.sleep(0.2)
    wl.inner_sum.zero_()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = wl.sim.launches
    D.barrier()
    for k in range(args.steps):
        flush.zero_()
        ev[k][0].record()
        wl.step(warm + k, count_inner=False)
        ev[k][1].record()
        wl.inner_sum += wl.sim.inner.sum()  # (outside the timed region: bookkeeping of this script)
    stats = D.all_reduce(wl.stats.clone())  # episode statistics: the one collective of these workloads
    D.barrier()
    launches = wl.sim.launches - launches0
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:  # what the last step handed back, before the end-to-end loop steps the envs again
        sim = wl.sim
        arrays = {"reward": sim.reward, "terminated": sim.terminated, "truncated": sim.truncated, "inner": sim.inner}
        planes = {"obs": sim.obs_state}
        if args.config != 5:  # vec_step: episode bookkeeping and the observation each finished episode ended in
            arrays.update(ep_return=wl.ep_return, ep_len=wl.ep_len, stats=wl.stats)
            planes["final_obs"] = wl.final_obs
        dump_outputs(args.dump_outputs, sim, planes, arrays)
    t = D.max_seconds(sum(a.elapsed_time(b) for a, b in ev) * 1e-3)
    units = float(wl.B) * args.steps * world
    value = units / t
    inner = D.all_reduce(wl.inner_sum.clone())
    updates_per_s = float(inner.item()) / t
    # ---- end to end: host actions up, rewards/flags back, every step
    for k in range(2):
        wl.step_e2e(k)
    D.barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        wl.step_e2e(k)
        torch.cuda.synchronize()  # the caller consumes the step's result before it acts again
    D.barrier()
    e2e_value = units / D.max_seconds(time.perf_counter() - t0)
    if rank == 0:
        alu_peak, _ = engine.issue_peak(0, 4000)
        h2d, d2h = wl.e2e_bytes()
        algorithmic = SURVEY_INSTR_PER_UPDATE * updates_per_s / world
        roofline = {"bound": "issue", "kernel": "k_env_step_first + k_env_step_att" if args.config != 5 else "k_env_step",
                    "achieved": algorithmic / 1e9, "peak": alu_peak / 1e9, "unit": "G thread-instr/s", "frac": algorithmic / alu_peak,
                    "algorithmic_thread_inst_per_update": SURVEY_INSTR_PER_UPDATE,
                    "peak_source": "pbn_issue_peak(0): dependency-free LOP3+IADD3 chains, measured in this run",
                    "node_updates_per_s_per_gpu": updates_per_s / world, "traffic": None,
                    "note": "step-until-attractor launches are bounded by the serial chain of their slowest env (inner cap x "
                            "per-update latency), not by issue: see DESIGN.md §4a" if args.config != 5 else
                            "latency-bound: two blocks per SM (46 KB network image + 32-word state columns)"}
        cpu = wl.cpu_sample(12.0) if world == 1 else None
        line = {"metric": wl.metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": t * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32", "data": "synthetic", "config": dict(wl.describe(world), **wl.fixture), "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "api": "Simulator.vec_step / env_step with pinned host actions up, int32 rewards + bool flags back"},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "node_updates_per_s": updates_per_s, "mean_inner_updates": float(inner.item()) / units,
                "episode_stats": dict(zip(("episodes", "return_sum", "length_sum", "successes", "cap_hits", "env_steps"),
                                          [int(v) for v in stats.tolist()[:6]]))}
        print(json.dumps(line), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[2, 3, 4, 5],
                    help="BASELINE.json configuration, 1-based as SURVEY.md §8d numbers them (3 = the headline SSD workload)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32/float64; state "
                         f"arrays for a fixed seeded sample of {DUMP_SAMPLE} chains or envs); same arguments, same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; the reference arm times samples and keeps none")
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 3:
        run_gpu_ssd(args)
    else:
        run_gpu_env(args)


if __name__ == "__main__":
    main()
