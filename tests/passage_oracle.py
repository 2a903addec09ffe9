"""TEST INFRASTRUCTURE — ctypes front end of tests/passage_oracle.c, the oracle's first-passage loop (orc_first_passage).

The library is oracle/pbn_oracle.c plus orc_first_passage in one translation unit, built with the oracle's own flags into
the oracle's build directory; networks and draws are the oracle's (oracle.Net, oracle.Draws)."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

import oracle as orc

SRC = Path(__file__).resolve().parent / "passage_oracle.c"
LIB = orc.BUILD / "libpbn_oracle_passage.so"

_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = (SRC, orc.HERE / "pbn_oracle.c")
        if not LIB.exists() or any(LIB.stat().st_mtime < d.stat().st_mtime for d in deps):
            orc.BUILD.mkdir(exist_ok=True)
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-ffp-contract=off", f"-I{orc.HERE}",
                                   "-o", str(LIB), str(SRC), "-lm"])
        _lib = C.CDLL(str(LIB))
    return _lib


def first_passage(net, state, iters, p, pins, tgt_nodes, goal, draws, env0=0, edges=None, t0=0, t_hit=None):
    """orc_first_passage for each pin set of `pins` (dicts {node index: 0 or 1}) with edge pins `edges` (None, or uint32
    [K][E] rows as in edge_pin_oracle.ssd_pinned) and goal buckets `goal` (list of ints), every variant on the same draws.
    state: uint8 [chains][N] (the same start for every variant) or [K][chains][N]; t_hit: None (every chain runs) or int64
    [K][chains], in/out.  Returns (t_hit int64 [K][chains], final states uint8 [K][chains][N])."""
    K = len(pins)
    tgt = np.ascontiguousarray(tgt_nodes, np.int32)
    st = np.ascontiguousarray(state, np.uint8)
    out = np.ascontiguousarray(np.repeat(st[None], K, axis=0) if st.ndim == 2 else st.copy())
    chains = out.shape[1]
    hit = np.full((K, chains), -1, np.int64) if t_hit is None else np.ascontiguousarray(t_hit, np.int64).copy()
    edges = np.zeros((K, 0), np.uint32) if edges is None else np.ascontiguousarray(edges, np.uint32)
    gl = np.ascontiguousarray(list(goal) or [-1], np.int64)
    for k, pin in enumerate(pins):
        vec = np.full(net.n, -1, np.int8)
        for i, v in pin.items():
            vec[int(i)] = int(v)
        row = np.ascontiguousarray(edges[k])
        rc = lib().orc_first_passage(C.byref(net.c), orc._p(out[k]), C.c_int64(chains), C.c_int64(env0), C.c_int64(iters),
                                     C.c_int64(t0), C.c_double(p), orc._p(vec), orc._p(row), C.c_int(row.shape[0]),
                                     orc._p(tgt), C.c_int(len(tgt)), orc._p(gl), C.c_int(len(goal)), orc._p(hit[k]),
                                     C.byref(draws.c))
        if rc:
            raise ValueError("orc_first_passage: Philox draws only, env0 a multiple of 32 when p > 0")
    return hit, out
