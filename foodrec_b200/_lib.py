"""ctypes binding of include/foodrec_b200.h.  There is no fallback: if the shared
library is missing or a symbol is absent this module raises at import/use time."""
from __future__ import annotations

import ctypes as C
import os

from . import _build

FR_OK = 0
FR_ERR_ARG, FR_ERR_CUDA, FR_ERR_STATE, FR_ERR_UNSUPPORTED = -1, -2, -3, -4
FR_SGD, FR_ADAGRAD, FR_RMSPROP, FR_ADAM = 0, 1, 2, 3
FR_ADAM_DENSE, FR_ADAM_LAZY_EXACT, FR_ADAM_LAZY_SERIES = 0, 1, 2
FR_POINTWISE, FR_BPR = 0, 1
FR_TABLE_F32, FR_TABLE_BF16 = 0, 1
(FR_OUT_LOSS, FR_OUT_NORM, FR_OUT_SCALE, FR_OUT_GENERAL, FR_OUT_PERSONAL, FR_OUT_LR,
 FR_OUT_UNIQ_USERS, FR_OUT_UNIQ_ITEMS, FR_OUT_LABEL_ENTRIES, FR_OUT_OVERFLOW) = range(10)
FR_OUT_COUNT = 12
FR_T_NAMES = ("sort", "fwd", "finalize", "user_chunk", "user_combine", "label", "item_chunk",
              "item_combine", "sweep", "misc")
FR_T_COUNT = len(FR_T_NAMES)

LEARNERS = {"sgd": FR_SGD, "adagrad": FR_ADAGRAD, "rmsprop": FR_RMSPROP, "adam": FR_ADAM}


def learner_code(name: str) -> int:
    """Model_Recommender.py:228-235: case-insensitive match, anything else is SGD."""
    return LEARNERS.get(str(name).lower(), FR_SGD)


class fr_config(C.Structure):
    _fields_ = [("embed_size", C.c_int32), ("num_users", C.c_int32), ("num_items", C.c_int32),
                ("num_labels", C.c_int32), ("learner", C.c_int32), ("adam_mode", C.c_int32),
                ("max_rows", C.c_int32), ("max_label_entries", C.c_int32),
                ("lr", C.c_float), ("high_level_score_coefficient", C.c_float),
                ("beta_1", C.c_float), ("beta_2", C.c_float), ("alpha", C.c_float),
                ("clip_norm", C.c_float),
                ("adam_beta1", C.c_float), ("adam_beta2", C.c_float), ("adam_eps", C.c_float),
                ("rms_decay", C.c_float), ("rms_eps", C.c_float)]


class fr_tables(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("P", "R", "Cat", "G", "s1_P", "s2_P", "s1_R", "s2_R", "s1_Cat", "s2_Cat",
                 "last_P", "last_R", "item_cats", "user_label_off", "user_label_idx")]


class fr_batch(C.Structure):
    _fields_ = [("mode", C.c_int32), ("n_groups", C.c_int32),
                ("users", C.c_void_p), ("items", C.c_void_p), ("cats", C.c_void_p),
                ("labels", C.c_void_p), ("write_sign", C.c_void_p), ("user_labels", C.c_void_p)]


class fr_catalog_opts(C.Structure):
    _fields_ = [("cta_group", C.c_int32), ("max_pass_rows", C.c_int32), ("splits", C.c_int32), ("epi_sets", C.c_int32), ("tile_n", C.c_int32), ("a_split", C.c_int32)]


class fr_shard(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("cap", C.c_int32),
                ("items_per_rank", C.c_int32), ("global_batch", C.c_int32)]


_PROTOS = {
    "fr_abi_version": (C.c_int, []),
    "fr_create": (C.c_int, [C.POINTER(fr_config), C.POINTER(C.c_void_p)]),
    "fr_destroy": (C.c_int, [C.c_void_p]),
    "fr_last_error": (C.c_char_p, [C.c_void_p]),
    "fr_set_tables": (C.c_int, [C.c_void_p, C.POINTER(fr_tables)]),
    "fr_set_table_format": (C.c_int, [C.c_void_p, C.c_int32]),
    "fr_set_shadow": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_get_step": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "fr_set_step": (C.c_int, [C.c_void_p, C.c_int64]),
    "fr_set_health_blend": (C.c_int, [C.c_void_p, C.c_int32]),
    "fr_fwd_score": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "fr_train_step": (C.c_int, [C.c_void_p, C.POINTER(fr_batch), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_train_step_host": (C.c_int, [C.c_void_p, C.POINTER(fr_batch), C.c_int32, C.c_void_p, C.c_void_p]),
    "fr_feed_prefetch": (C.c_int, [C.c_void_p, C.POINTER(fr_batch)]),
    "fr_adam_flush": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fr_launch_count": (C.c_int64, []),
    "fr_timing_enable": (C.c_int, [C.c_void_p, C.c_int32]),
    "fr_timing_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]),
    "fr_eval_sampled_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_sort_pairs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_catalog_prepare": (C.c_int, [C.c_void_p, C.POINTER(fr_catalog_opts), C.c_void_p, C.c_void_p]),
    "fr_catalog_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_catalog_topk_excluding": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                            C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_gather_user_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "fr_catalog_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_catalog_timing_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_int32]),
    "fr_catalog_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "fr_catalog_cycle_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p]),
    "fr_catalog_fallback_rows": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.c_void_p]),
    "fr_sample_negatives": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "fr_sample_bpr_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_uint64, C.c_int64,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_philox4x32_10": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "fr_shard_packed_len": (C.c_int64, [C.c_void_p]),
    "fr_shard_route_block": (C.c_int64, [C.POINTER(fr_batch), C.c_int32]),
    "fr_shard_route": (C.c_int, [C.c_void_p, C.POINTER(fr_batch), C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_shard_unroute": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_shard_set_peers": (C.c_int, [C.c_void_p, C.POINTER(fr_shard), C.c_void_p, C.c_void_p]),
    "fr_shard_plan": (C.c_int, [C.c_void_p, C.POINTER(fr_batch), C.POINTER(fr_shard), C.c_void_p, C.c_void_p]),
    "fr_shard_serve": (C.c_int, [C.c_void_p, C.POINTER(fr_shard), C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_shard_serve_prepare": (C.c_int, [C.c_void_p, C.POINTER(fr_shard), C.c_void_p, C.c_void_p]),
    "fr_shard_forward": (C.c_int, [C.c_void_p, C.POINTER(fr_batch), C.POINTER(fr_shard), C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_shard_update": (C.c_int, [C.c_void_p, C.POINTER(fr_batch), C.POINTER(fr_shard), C.c_int32, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "fr_shard_apply": (C.c_int, [C.c_void_p, C.POINTER(fr_shard), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None


def header_symbols():
    """Every function the public header declares (parsed, so the CPU test can check
    that the library exports all of them)."""
    import re
    hdr = os.path.join(os.path.dirname(_build.HERE), "include", "foodrec_b200.h")
    txt = open(hdr).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(fr_[a-z0-9_]+)\s*\(", txt)))


def lib():
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("FOODREC_B200_LIB", _build.LIB)     # override: A/B builds of the same sources
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: build it with `python -m foodrec_b200._build` "
            "(foodrec_b200 has no CPU or eager fallback)")
    L = C.CDLL(path)
    for name, (res, args) in _PROTOS.items():
        if not hasattr(L, name):
            raise RuntimeError(f"libfoodrec_b200.so does not export {name}")
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    if L.fr_abi_version() != 1:
        raise RuntimeError("libfoodrec_b200.so ABI mismatch")
    _lib = L
    return L


class FoodRecError(RuntimeError):
    pass


def check(handle, rc: int):
    if rc != FR_OK:
        msg = lib().fr_last_error(handle)
        raise FoodRecError(f"foodrec_b200 error {rc}: {msg.decode() if msg else '?'}")
