"""TEST INFRASTRUCTURE — ctypes front end of tests/edge_pin_oracle.c, the oracle's SSD with genes and regulatory edges pinned
(orc_ssd_pinned_edges).

The library is oracle/pbn_oracle.c plus orc_ssd_pinned_edges in one translation unit, built with the oracle's own flags into
the oracle's build directory; networks and draws are the oracle's (oracle.Net, oracle.Draws)."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

import oracle as orc

SRC = Path(__file__).resolve().parent / "edge_pin_oracle.c"
LIB = orc.BUILD / "libpbn_oracle_edge_pins.so"

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


def ssd_pinned(net, state, iters, p, pins, tgt_nodes, draws, env0=0, edges=None):
    """orc_ssd_pinned_edges for each pin set of `pins` (dicts {node index: 0 or 1}) with edge pins `edges` (None, or uint32
    [K][E]: row k = the entries dst | src << 12 | c << 24 of variant k, 0xFFFFFFFF = empty), every variant from its own copy
    of the start states `state` uint8 [chains][N] on the same draws.  Returns (hist uint64 [K][2^g], final states uint8
    [K][chains][N])."""
    tgt = np.ascontiguousarray(tgt_nodes, np.int32)
    hist = np.zeros((len(pins), 1 << len(tgt)), np.uint64)
    out = np.repeat(np.ascontiguousarray(state, np.uint8)[None], len(pins), axis=0)
    edges = np.zeros((len(pins), 0), np.uint32) if edges is None else np.ascontiguousarray(edges, np.uint32)
    assert edges.shape[0] == len(pins)
    for k, pin in enumerate(pins):
        vec = np.full(net.n, -1, np.int8)
        for i, v in pin.items():
            vec[int(i)] = int(v)
        row = np.ascontiguousarray(edges[k])
        rc = lib().orc_ssd_pinned_edges(C.byref(net.c), orc._p(out[k]), C.c_int64(out.shape[1]), C.c_int64(env0),
                                        C.c_int64(iters), C.c_double(p), orc._p(vec), orc._p(row), C.c_int(row.shape[0]),
                                        orc._p(tgt), C.c_int(len(tgt)), orc._p(hist[k]), C.byref(draws.c))
        if rc:
            raise ValueError("orc_ssd_pinned_edges: Philox draws only, env0 a multiple of 32 when p > 0")
    return hist, out
