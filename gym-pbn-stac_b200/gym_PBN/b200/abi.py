"""ctypes binding of the C-ABI declared in include/pbn_b200.h.

The CUDA library is the only compute path: if libpbn_b200.so is missing or fails to load this module
raises — there is no CPU fallback anywhere in the product.
"""
import ctypes as C
import os
from pathlib import Path

PKG_ROOT = Path(__file__).resolve().parents[2]  # gym-pbn-stac_b200/
LIB_PATH = Path(os.environ.get("PBN_B200_LIB", PKG_ROOT / "lib" / "libpbn_b200.so"))  # override = kernel experiments only

NET_TT, NET_PRED = 0, 1
ENV_PBN, ENV_PBCN, ENV_TARGET, ENV_MULTI, ENV_PBN_SD, ENV_PBCN_SD, ENV_PBN_ST, ENV_PBCN_ST = range(8)
DRAW_PHILOX, DRAW_REPLAY = 0, 1


class PbnNetDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_nodes", C.c_int32), ("first_updatable", C.c_int32),
                ("tt_in_off", C.c_void_p), ("tt_in", C.c_void_p), ("tt_tab_off", C.c_void_p), ("tt_prob", C.c_void_p),
                ("pr_off", C.c_void_p), ("pr_in", C.c_void_p), ("pr_lut", C.c_void_p),
                ("pr_cum", C.c_void_p), ("pr_codsum", C.c_void_p)]


class PbnEnvDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("horizon", C.c_int32), ("max_inner", C.c_int32), ("force", C.c_int32),
                ("dedup", C.c_int32), ("control_write", C.c_int32), ("n_control", C.c_int32),
                ("successful_reward", C.c_int32), ("wrong_attractor_cost", C.c_int32),
                ("n_att", C.c_int32), ("att_off", C.c_void_p), ("cube", C.c_void_p),
                ("tgt_first", C.c_int32), ("n_tgt", C.c_int32),
                ("gamma_pow", C.c_void_p), ("n_gamma", C.c_int32), ("max_interval", C.c_int32)]


class PbnDraws(C.Structure):
    _fields_ = [("mode", C.c_int32), ("epoch", C.c_uint32), ("seed", C.c_uint64),
                ("ints", C.c_void_p), ("dbls", C.c_void_p), ("int_stride", C.c_int64), ("dbl_stride", C.c_int64),
                ("used", C.c_void_p), ("epoch_dev", C.c_void_p)]


class PbnFitDesc(C.Structure):
    _fields_ = [("n_genes", C.c_int32), ("n_samples", C.c_int32), ("row_off", C.c_void_p), ("rows", C.c_void_p),
                ("cod_rank", C.c_void_p)]


class PbnVecState(C.Structure):
    _fields_ = [("ep_return", C.c_void_p), ("ep_len", C.c_void_p), ("stats", C.c_void_p), ("final_obs", C.c_void_p),
                ("target_state", C.c_void_p), ("autoreset", C.c_int32), ("reset_draws", PbnDraws),
                ("probabilities", C.c_void_p), ("pair_ids", C.c_void_p), ("sample_pair", C.c_int32),
                ("reward_f64", C.c_void_p), ("ep_return_f64", C.c_void_p), ("return_sum_f64", C.c_void_p)]


class PbnStepPlan(C.Structure):
    _fields_ = [("running", C.c_void_p), ("work", C.c_void_p), ("budget", C.c_int32), ("resume", C.c_int32), ("phase", C.c_int32)]


EXPORTS = {
    # name: (restype, argtypes)
    "pbn_net_create": (C.c_int, [C.POINTER(PbnNetDesc), C.POINTER(C.c_void_p)]),
    "pbn_net_destroy": (C.c_int, [C.c_void_p]),
    "pbn_net_words": (C.c_int, [C.c_void_p]),
    "pbn_env_create": (C.c_int, [C.c_void_p, C.POINTER(PbnEnvDesc), C.POINTER(C.c_void_p)]),
    "pbn_env_destroy": (C.c_int, [C.c_void_p]),
    "pbn_rollout": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int32,
                              C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_env_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                               C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_env_step_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                   C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_vec_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(PbnVecState), C.c_int64, C.c_int64,
                               C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_env_step_plan": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(PbnVecState), C.POINTER(PbnStepPlan),
                                    C.c_int64, C.c_int64, C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_env_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                C.c_int64, C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_env_reset_cur": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_int64, C.c_int64, C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_env_attractor_index": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "pbn_rand_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_ssd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_double,
                          C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(PbnDraws), C.c_void_p]),
    "pbn_bucket_hist": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "pbn_ssd_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_void_p,
                               C.c_int32, C.c_uint64, C.c_uint32, C.c_void_p]),
    "pbn_unpack_state": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "pbn_pack_state": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "pbn_stg_change_masks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "pbn_stg_expand": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "pbn_stg_walk": (C.c_int, [C.c_void_p, C.c_int32, C.c_uint32, C.c_int64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "pbn_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "pbn_fetch_host": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.c_int32, C.c_void_p, C.c_void_p]),
    "pbn_fetch_step_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                      C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pbn_fit_scan_host": (C.c_int, [C.POINTER(PbnFitDesc), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_float)]),
    "pbn_fit_eval_host": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]),
    "pbn_issue_peak": (C.c_int, [C.c_int32, C.c_int64, C.POINTER(C.c_float), C.POINTER(C.c_double)]),
    "pbn_geom_shortcut_check": (C.c_int, [C.c_double, C.POINTER(C.c_float), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "pbn_last_error": (C.c_char_p, []),
    "pbn_version": (C.c_char_p, []),
}

_lib = None


class PbnError(RuntimeError):
    pass


def lib():
    """Load libpbn_b200.so (built in-tree by gym-pbn-stac_b200/build.py).  No fallback."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise PbnError(
                f"CUDA library not found at {LIB_PATH}. Build it with `python gym-pbn-stac_b200/build.py` "
                "(nvcc, sm_100a). gym_PBN on B200 has no CPU fallback."
            )
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in EXPORTS.items():
            fn = getattr(l, name)  # AttributeError if the library does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = l
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().pbn_last_error().decode()
        if rc == 1:
            raise ValueError(msg)
        raise PbnError(f"pbn_b200 error {rc}: {msg}")
