"""ctypes binding of librae.so (C ABI declared in include/rae.h).

There is no CPU fallback: if the shared library is missing the import of the engine fails loudly, and every entry
point that computes refuses to run without a CUDA device (RAE_ENODEVICE).
"""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RAE_LIB") or os.path.join(HERE, "librae.so")    # RAE_LIB: A/B measurement of two builds
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "rae.h")

RAE_ABI_VERSION = 4
RAE_MODEL_A, RAE_MODEL_C, RAE_MODEL_AC = 0, 1, 2
RAE_OPT_ADAGRAD, RAE_OPT_SGD = 0, 1
RAE_P_W, RAE_P_WB, RAE_P_A, RAE_P_AB, RAE_P_C, RAE_P_C1, RAE_P_C2 = range(7)
PARAM_IDS = {"W": RAE_P_W, "Wb": RAE_P_WB, "A": RAE_P_A, "Ab": RAE_P_AB, "C": RAE_P_C, "C1": RAE_P_C1, "C2": RAE_P_C2}
RAE_SPLIT = {"train": 0, "valid": 1, "test": 2}          # settings.py:26
RAE_FLAG_FIX_SP_QUIRK = 1
RAE_FLAG_DENSE_GRADS = 2
RAE_FLAG_FORCE_SIMT = 4
RAE_FLAG_FORCE_TENSOR = 8
RAE_FLAG_NO_FEATURE_CACHE = 16
RAE_FLAG_EMIT_ONLY = 32
RAE_FLAG_CLUSTER_MULTICAST = 64
RAE_FLAG_NO_PDL = 128
RAE_ENODEVICE = -5
RAE_NUM_PHASES = 15
RAE_FLAG_WORDS = 64
RAE_MAX_TOPK = 16


class RaeConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("model", C.c_int32), ("K", C.c_int32), ("d", C.c_int32), ("S", C.c_int32),
        ("B", C.c_int32), ("F", C.c_int64), ("N", C.c_int64), ("optimizer", C.c_int32), ("ext_reg", C.c_int32),
        ("flags", C.c_uint32), ("device", C.c_int32), ("lr", C.c_double), ("l1", C.c_double), ("l2", C.c_double),
        ("alpha", C.c_double), ("adj", C.c_double), ("z_total", C.c_int64),
    ]


class RaeDistStep(C.Structure):
    _fields_ = ([("world", C.c_int32), ("reserved", C.c_int32)]
                + [(n, C.c_void_p) for n in ("w_shards", "a_shards", "ab_shards", "gw_bufs", "ga_bufs", "gab_bufs", "Wc", "Ac", "Abc")]
                + [("f_ids", C.c_void_p), ("n_f", C.c_int64), ("e_ids", C.c_void_p), ("n_e", C.c_int64), ("batch_index", C.c_int64)]
                + [(n, C.c_void_p) for n in ("a1c", "a2c", "n1c", "n2c")] + [("neg_ld", C.c_int64)]
                + [(n, C.c_void_p) for n in ("W", "accW", "A", "accA", "Ab", "accAb")]
                + [("fr_rows", C.c_void_p), ("fr_off", C.c_void_p), ("n_fr", C.c_int64), ("f_src", C.c_void_p), ("f_slot", C.c_void_p)]
                + [("er_rows", C.c_void_p), ("er_off", C.c_void_p), ("n_er", C.c_int64), ("e_src", C.c_void_p), ("e_slot", C.c_void_p)]
                + [("cost_dev", C.c_void_p), ("flag_bufs", C.c_void_p), ("dense_bufs", C.c_void_p), ("rank", C.c_int32),
                   ("global_cost", C.c_int32), ("w_rows", C.c_int64)])


class RaeStepStats(C.Structure):
    _fields_ = [
        ("nnz", C.c_int64), ("unique_w_rows", C.c_int64), ("unique_e_rows", C.c_int64), ("entity_occ", C.c_int64),
        ("kernel_launches", C.c_int32), ("tensor_path", C.c_int32), ("algorithmic_bytes", C.c_double),
    ]


_P = C.c_void_p
_SIGNATURES = {
    "rae_abi_version": (C.c_int, []),
    "rae_create": (C.c_int, [C.POINTER(RaeConfig), C.POINTER(_P)]),
    "rae_destroy": (None, [_P]),
    "rae_last_error": (C.c_char_p, [_P]),
    "rae_bind_params": (C.c_int, [_P] + [_P] * 7),
    "rae_bind_accumulators": (C.c_int, [_P] + [_P] * 7),
    "rae_bind_split": (C.c_int, [_P, C.c_int32, _P, _P, C.c_int64, _P, _P, _P]),
    "rae_bind_epoch_negatives": (C.c_int, [_P, _P, _P, C.c_int64]),
    "rae_train_step": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_double), _P]),
    "rae_train_step_host": (C.c_int, [_P, C.c_int64, _P, _P, C.POINTER(C.c_double), _P]),
    "rae_train_step_host_ld": (C.c_int, [_P, C.c_int64, _P, C.c_int64, _P, C.c_int64, C.POINTER(C.c_double), _P]),
    "rae_train_step_explicit": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_int64, C.POINTER(C.c_double), _P]),
    "rae_label": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, _P]),
    "rae_label_host": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, _P]),
    "rae_get_probs": (C.c_int, [_P, _P, _P]),
    "rae_get_dense_grad": (C.c_int, [_P, C.c_int32, _P, _P]),
    "rae_get_entity_segments": (C.c_int, [_P, _P, _P, _P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P]),
    "rae_get_step_stats": (C.c_int, [_P, C.POINTER(RaeStepStats)]),
    "rae_bind_grad_buffers": (C.c_int, [_P, _P, _P, _P, _P]),
    "rae_dense_grad_size": (C.c_int64, [_P]),
    "rae_train_step_end": (C.c_int, [_P, _P]),
    "rae_read_cost": (C.c_int, [_P, C.POINTER(C.c_double), _P]),
    "rae_peer_alloc": (C.c_int, [C.c_int64, C.POINTER(_P), _P]),
    "rae_peer_free": (C.c_int, [_P]),
    "rae_peer_open": (C.c_int, [_P, C.POINTER(_P)]),
    "rae_peer_close": (C.c_int, [_P]),
    "rae_fetch_rows": (C.c_int, [_P, _P, C.c_int32, C.c_int64, _P, C.c_int64, _P, _P]),
    "rae_pull_apply": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, _P, C.c_int64, _P, C.c_int32, _P]),
    "rae_shard_apply": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, _P, C.c_int64, _P, C.c_int32, C.c_int64, _P]),
    "rae_train_step_begin": (C.c_int, [_P, C.c_int64, _P, _P, _P, _P, C.c_int64, _P]),
    "rae_dist_step_begin": (C.c_int, [_P, C.POINTER(RaeDistStep), _P]),
    "rae_dist_step_end": (C.c_int, [_P, C.POINTER(RaeDistStep), _P]),
    "rae_dist_step_begin_host": (C.c_int, [_P, C.POINTER(RaeDistStep), _P, C.c_int64, _P, C.c_int64, _P]),
    "rae_bind_push_targets": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int64, C.c_int64]),
    "rae_dist_set_dense_wait": (C.c_int, [_P, _P]),
    "rae_dist_read_cost": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "rae_peer_barrier": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P]),
    "rae_peer_status": (C.c_int, [_P, _P]),
    "rae_copy_cost": (C.c_int, [_P, _P, _P]),
    "rae_label_shards": (C.c_int, [_P, _P, C.c_int32, _P, _P, C.c_int64, _P, _P, _P]),
    "rae_label_topk": (C.c_int, [_P, _P, C.c_int32, _P, _P, C.c_int64, C.c_int32, _P, _P, _P]),
    "rae_rank_arguments": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, _P, _P, _P]),
    "rae_predict_arguments": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_int32, _P, _P, _P, _P, _P]),
    "rae_sample_negatives": (C.c_int, [_P, _P, _P, C.c_int64, C.c_double, _P, C.c_int64, _P, _P]),
    "rae_set_profiling": (C.c_int, [_P, C.c_int32]),
    "rae_get_phase_times": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "rae_get_timeline": (C.c_int, [_P, C.c_char_p, C.c_int64]),
    "rae_phase_name": (C.c_char_p, [C.c_int32]),
}

_lib = None


def header_symbols(path: str = HEADER_PATH):
    """Names of every function declared in include/rae.h (used by the CPU test that checks the exports)."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rae_[a-z_0-9]+)\s*\(", src)))


def load():
    """Load librae.so; raises if it has not been built (``python -m relation_autoencoder_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "librae.so is missing (%s): build it with `python -m relation_autoencoder_b200.build`; "
            "there is no CPU fallback for the training hot path" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.rae_abi_version() != RAE_ABI_VERSION:
        raise RuntimeError("librae.so ABI version %d != %d" % (lib.rae_abi_version(), RAE_ABI_VERSION))
    _lib = lib
    return lib
