"""ctypes binding of libnais_b200.so (include/nais_b200.h).  No CPU fallback: a missing library is a hard error."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libnais_b200.so")

DIST_NONE, DIST_LATLON, DIST_KM = 0, 1, 2
PREC_FP32, PREC_TC_SPLIT, PREC_TC_FAST, PREC_TC_MIX, PREC_TC_AUTO = 0, 1, 2, 3, 4
PREC_FLAG_GENERIC = 0x100  # run-time-shape tensor kernel even where a compile-time-shape instantiation exists
PRECISIONS = {"fp32": PREC_FP32, "tc_split": PREC_TC_SPLIT, "tc_fast": PREC_TC_FAST, "tc_mix": PREC_TC_MIX,
              "tc_auto": PREC_TC_AUTO}
PREC_FLAG_ONE_CTA = 0x200  # keep one CTA per SM where the CTA-pair (cta_group::2) kernel would run (D = hid = 64)
PRECISIONS.update({k + "_generic": v | PREC_FLAG_GENERIC for k, v in list(PRECISIONS.items()) if k != "fp32"})
PRECISIONS.update({k + "_onecta": v | PREC_FLAG_ONE_CTA for k, v in list(PRECISIONS.items()) if k in ("tc_auto", "tc_split", "tc_mix")})
PAIRS_PRECISIONS = {"auto": 0, "fp32": 1, "tc": 2}  # NAIS_PAIRS_*
ERR_INDEX = -7

ABI_VERSION = 2  # NAIS_ABI_VERSION of include/nais_b200.h
c_float_p = C.c_void_p  # device pointers travel as integers


class NaisBranch(C.Structure):
    _fields_ = [("hist_poi", C.c_void_p), ("tgt_poi", C.c_void_p), ("hist_reg", C.c_void_p), ("tgt_reg", C.c_void_p),
                ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("w_poi", C.c_int32), ("w_reg", C.c_int32)]


class NaisParams(C.Structure):
    _fields_ = [("branch", NaisBranch * 2), ("n_branch", C.c_int32), ("hid", C.c_int32), ("item_num", C.c_int32),
                ("region_num", C.c_int32), ("dist_mode", C.c_int32), ("dist_scale", C.c_float), ("dist_w", C.c_void_p),
                ("dist_b", C.c_void_p), ("dist_embed", C.c_void_p), ("dist_buckets", C.c_int32),
                ("dist_bucket_km", C.c_float), ("beta", C.c_float), ("dropout_p", C.c_float),
                ("dropout_seed", C.c_uint64), ("pairs_precision", C.c_int32), ("reserved0", C.c_int32)]


class NaisPairs(C.Structure):
    _fields_ = [("hist", C.c_void_p), ("tgt", C.c_void_p), ("hreg", C.c_void_p), ("treg", C.c_void_p),
                ("aux", C.c_void_p), ("B", C.c_int64), ("H", C.c_int32), ("n_seg", C.c_int32), ("seg_offsets", C.c_void_p),
                ("row_offsets", C.c_void_p), ("seg_cell_offsets", C.c_void_p), ("tile_seg", C.c_void_p), ("tile_row0", C.c_void_p),
                ("n_tiles", C.c_int64), ("n_cells", C.c_int64), ("hist_coords", C.c_void_p), ("tgt_coords", C.c_void_p),
                ("center_lat", C.c_float), ("center_lon", C.c_float)]


class NaisGrads(C.Structure):
    _fields_ = [("hist_poi", C.c_void_p * 2), ("tgt_poi", C.c_void_p * 2), ("reg", C.c_void_p * 2),
                ("w1", C.c_void_p * 2), ("b1", C.c_void_p * 2), ("w2", C.c_void_p * 2), ("dist_w", C.c_void_p),
                ("dist_b", C.c_void_p), ("dist_embed", C.c_void_p), ("remap_hist_poi", C.c_void_p * 2),
                ("remap_tgt_poi", C.c_void_p * 2), ("remap_reg", C.c_void_p * 2)]


class NaisAdagrad(C.Structure):
    _fields_ = [("lr", C.c_float), ("eps", C.c_float), ("sum_hist_poi", C.c_void_p * 2), ("sum_tgt_poi", C.c_void_p * 2),
                ("sum_reg", C.c_void_p * 2)]


class NaisDenseAdagrad(C.Structure):
    _fields_ = [("lr", C.c_float), ("eps", C.c_float), ("sum_w1", C.c_void_p), ("sum_b1", C.c_void_p), ("sum_w2", C.c_void_p),
                ("sum_dist_w", C.c_void_p), ("sum_dist_b", C.c_void_p), ("sum_region_w1", C.c_void_p), ("sum_region_b1", C.c_void_p),
                ("sum_region_w2", C.c_void_p), ("sum_dist_embed", C.c_void_p)]


class NaisBprLoss(C.Structure):
    _fields_ = [("num_neg", C.c_int32), ("reserved0", C.c_int32), ("group_weight", C.c_void_p)]


class NaisCatalog(C.Structure):
    _fields_ = [("region", C.c_void_p), ("coords", C.c_void_p), ("row_base", C.c_int64), ("n_rows", C.c_int64),
                ("center_lat", C.c_float), ("center_lon", C.c_float)]


class NaisUsers(C.Structure):
    _fields_ = [("offsets", C.c_void_p), ("items", C.c_void_p), ("region", C.c_void_p), ("coords", C.c_void_p),
                ("n_users", C.c_int32)]


class NaisGeoMix(C.Structure):
    _fields_ = [("a", C.c_float), ("b", C.c_float), ("alpha", C.c_float), ("user_logmax", C.c_void_p)]


# every symbol include/nais_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "nais_abi_version": (C.c_int, []),
    "nais_strerror": (C.c_char_p, [C.c_int]),
    "nais_launch_count": (C.c_uint64, []),
    "nais_pairs_dispatch": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "nais_pairs_forward": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "nais_pairs_explain_workspace_bytes": (C.c_size_t, [C.POINTER(NaisParams), C.POINTER(NaisPairs)]),
    "nais_pairs_explain": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_pairs_backward_workspace_bytes": (C.c_size_t, [C.POINTER(NaisParams), C.POINTER(NaisPairs)]),
    "nais_pairs_train_step_workspace_bytes": (C.c_size_t, [C.POINTER(NaisParams), C.POINTER(NaisPairs)]),
    "nais_pairs_train_step": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.c_void_p, C.c_void_p, C.POINTER(NaisAdagrad),
                                        C.POINTER(NaisDenseAdagrad), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_pairs_train_step_bpr": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.POINTER(NaisBprLoss), C.POINTER(NaisAdagrad),
                                            C.POINTER(NaisDenseAdagrad), C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_train_users_workspace_bytes": (C.c_size_t, [C.POINTER(NaisParams), C.c_int32, C.c_int32]),
    "nais_train_users": (C.c_int, [C.POINTER(NaisParams), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_int32, C.c_int32, C.c_uint64, C.POINTER(NaisAdagrad), C.POINTER(NaisDenseAdagrad),
                                   C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_train_users_centred": (C.c_int, [C.POINTER(NaisParams), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_uint64, C.POINTER(NaisAdagrad),
                                           C.POINTER(NaisDenseAdagrad), C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float,
                                           C.c_void_p]),
    "nais_train_users_dropout": (C.c_int, [C.POINTER(NaisParams), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_uint64, C.POINTER(NaisAdagrad),
                                           C.POINTER(NaisDenseAdagrad), C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float,
                                           C.c_void_p, C.c_void_p]),
    "nais_train_users_bpr": (C.c_int, [C.POINTER(NaisParams), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_uint64, C.POINTER(NaisAdagrad),
                                       C.POINTER(NaisDenseAdagrad), C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float,
                                       C.c_void_p, C.c_void_p]),
    "nais_rows_adagrad_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "nais_rows_adagrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_float, C.c_float, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_sample_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "nais_pairs_backward": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.POINTER(NaisGrads), C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_pairs_forward_presort": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.POINTER(NaisGrads), C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_pairs_backward_presorted": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.POINTER(NaisGrads), C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_pairs_backward_adagrad": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisPairs), C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.POINTER(NaisGrads), C.POINTER(NaisAdagrad), C.c_void_p, C.c_size_t,
                                              C.c_void_p]),
    "nais_powerlaw_logscore": (C.c_int, [C.POINTER(NaisCatalog), C.POINTER(NaisUsers), C.c_int64, C.c_int64, C.c_float, C.c_float,
                                         C.c_void_p, C.c_void_p]),
    "nais_fullrank_workspace_bytes": (C.c_size_t, [C.POINTER(NaisParams), C.c_int32, C.c_int64, C.c_int64, C.c_int64,
                                                   C.c_int32, C.c_int32]),
    "nais_fullrank_topk": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisCatalog), C.POINTER(NaisUsers), C.c_int64,
                                     C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_size_t, C.c_void_p]),
    "nais_fullrank_scores": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisCatalog), C.POINTER(NaisUsers), C.c_int64,
                                       C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_hits_at_k": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                 C.c_void_p]),
    "nais_topk_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "nais_fullrank_plan_bytes": (C.c_size_t, [C.POINTER(NaisParams), C.c_int64, C.c_int64, C.c_int32]),
    "nais_fullrank_prepare": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisCatalog), C.c_int64, C.c_int64, C.c_int32,
                                        C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_fullrank_planned_workspace_bytes": (C.c_size_t, [C.POINTER(NaisParams), C.c_int32, C.c_int64, C.c_int64, C.c_int64,
                                                           C.c_int32, C.c_int32]),
    "nais_fullrank_topk_planned": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisCatalog), C.POINTER(NaisUsers), C.c_int64,
                                             C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "nais_powerlaw_logmax": (C.c_int, [C.POINTER(NaisCatalog), C.POINTER(NaisUsers), C.c_int64, C.c_int64, C.c_float, C.c_float,
                                       C.c_int32, C.c_void_p, C.c_void_p]),
    "nais_fullrank_topk_geo_planned": (C.c_int, [C.POINTER(NaisParams), C.POINTER(NaisCatalog), C.POINTER(NaisUsers), C.c_int64,
                                                 C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t,
                                                 C.POINTER(NaisGeoMix), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                                 C.c_void_p]),
    "nais_topk_merge_keys": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "nais_poll_bad_index": (C.c_int, [C.c_void_p, C.c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Load the in-tree library.  Raises if it has not been built (`python -m poi_recommendation_models_b200.build_ext`
    or `__graft_entry__.build()`): there is deliberately no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python poi_recommendation_models_b200/build_ext.py` "
                           "(nvcc, sm_100a).  There is no CPU / PyTorch fallback for the NAIS ops.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.nais_abi_version() != ABI_VERSION:
        raise RuntimeError("libnais_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().nais_strerror(rc).decode()
        raise RuntimeError(f"{what} failed ({rc}): {msg}")
