"""ctypes binding of include/recsys_b200.h (the C-ABI boundary of the hot path).

There is NO CPU fallback: if librecsys_b200.so is missing and cannot be built, importing the ops raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librecsys_b200.so")
RS_MAX_FIELDS = 64
RS_CHUNK = 64
RS_UPD_GRAD, RS_UPD_SGD, RS_UPD_ADAM = 0, 1, 2

f32p = C.c_void_p   # device pointers travel as integers
i64p = C.c_void_p
i32p = C.c_void_p


class rs_tables(C.Structure):
    _fields_ = [("num_fields", C.c_int32), ("width", C.c_int32),
                ("base", C.c_void_p * RS_MAX_FIELDS), ("rows", C.c_int64 * RS_MAX_FIELDS)]


RS_MAX_RANKS = 64


class rs_routes(C.Structure):
    _fields_ = [("n", C.c_int32), ("start", C.c_int64 * (RS_MAX_RANKS + 1)), ("base", C.c_void_p * RS_MAX_RANKS),
                ("row0", C.c_int64 * RS_MAX_RANKS), ("dyn_start", C.c_void_p), ("dyn_row0", C.c_void_p), ("cap_rows", C.c_int64), ("self", C.c_int32)]


class rs_dedup_opts(C.Structure):
    _fields_ = [("n_valid", C.c_void_p), ("shard_world", C.c_int32), ("shard_rows", C.c_int64)]


RS_SHARD_CTL_WORDS = 384
RS_CTL_CNT_IN, RS_CTL_BLK0_IN, RS_CTL_G0_IN, RS_CTL_SEND_START, RS_CTL_RECV_START, RS_CTL_M_TOTAL = 0, 64, 128, 192, 257, 322


RS_MAX_DIRECT = 8


class rs_shard(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("rows_per_rank", C.c_int64), ("cap_req", C.c_int64),
                ("cap_recv", C.c_int64), ("req", C.c_void_p * RS_MAX_RANKS), ("ctl", C.c_void_p * RS_MAX_RANKS),
                ("n_direct", C.c_int32), ("direct_lo", C.c_int64 * RS_MAX_DIRECT), ("direct_hi", C.c_int64 * RS_MAX_DIRECT)]


class rs_peer_tables(C.Structure):
    _fields_ = [("world", C.c_int32), ("direct_mask", C.c_uint64), ("shard", C.c_void_p * RS_MAX_RANKS), ("total_rows", C.c_int64),
                ("split_mask", C.c_uint64), ("stash_split", C.c_void_p)]


class rs_fields_io(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("ids", "dense_in", "cross", "bi", "pairs", "concat", "stash", "dot2", "had2")]


class rs_fields_grad(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("ids", "dense_in", "g_cross", "g_bi", "g_pairs", "g_concat", "g_dot2", "g_had2", "dE")]


class rs_segments(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("sorted_key", "sorted_pos", "uniq", "inverse", "counts", "seg_start", "seg_first_chunk",
                 "chunk_start", "chunk_seg", "multi_seg", "lookup_desc", "work_counter", "unit_start", "scale_sorted", "n_uniq", "n_chunks", "n_multi", "partial")] + [("partial_floats", C.c_int64)]


class rs_update(C.Structure):
    _fields_ = [("mode", C.c_int32), ("width", C.c_int32), ("F", C.c_int32), ("scale_width", C.c_int32),
                ("stash", C.c_void_p), ("scale", C.c_void_p), ("dense", C.c_void_p),
                ("table", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("dense_grad", C.c_void_p),
                ("lr", C.c_float), ("wd", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("step", C.c_int32), ("grad_routes", C.POINTER(rs_routes)), ("half_sm", C.c_int32)]


class rs_xslots(C.Structure):
    _fields_ = [("num_slots", C.c_int32), ("width", C.c_int32), ("xcols", C.c_int32),
                ("col", C.c_int32 * RS_MAX_FIELDS), ("ncols", C.c_int32 * RS_MAX_FIELDS),
                ("kind", C.c_int32 * RS_MAX_FIELDS), ("table", C.c_void_p * RS_MAX_FIELDS),
                ("rows", C.c_int64 * RS_MAX_FIELDS)]


class rs_gemm_nt(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("A", "B", "bias", "rowbias", "mask", "C")] + \
               [(n, C.c_int64) for n in ("M", "lda", "a_group", "a_group_stride", "ldb", "rb_group", "ldm", "ldc")] + \
               [(n, C.c_int32) for n in ("K", "N", "relu")]


class rs_din_weights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("W0", "b0", "W1", "b1", "W2", "b2")] + [("H1", C.c_int32), ("H2", C.c_int32)]


_I, _L, _P, _F, _Z = C.c_int32, C.c_int64, C.c_void_p, C.c_float, C.c_size_t
_PP = C.POINTER

# symbol -> argtypes; every function returns int except rs_last_error
SIGNATURES = {
    "rs_version": [],
    "rs_gather_rows": [_PP(rs_tables), _P, _L, _P, _P, _P],
    "rs_gather_rows_peer": [_P, _L, _I, _P, _L, _PP(rs_routes), _P, _P],
    "rs_fields_fwd": [_PP(rs_tables), _PP(rs_fields_io), _L, _P, _P],
    "rs_fields_bwd": [_PP(rs_tables), _PP(rs_fields_grad), _L, _P],
    "rs_ffm_fwd": [_PP(rs_tables), _P, _L, _I, _P, _P, _P, _P],
    "rs_ffm_dense_fwd": [_P, _L, _I, _I, _I, _PP(_I), _P, _P],
    "rs_ffm_dense_bwd": [_P, _P, _L, _I, _I, _I, _PP(_I), _P, _P],
    "rs_dedup_workspace_bytes": [_L, _I, _PP(_Z)],
    "rs_dedup_sort": [_P, _L, _I, _PP(_L), _L, _P, _Z, _PP(rs_segments), _P, _P],
    "rs_dedup_sort_ex": [_P, _L, _I, _PP(_L), _L, _PP(rs_dedup_opts), _P, _Z, _PP(rs_segments), _P, _P],
    "rs_segments_relabel": [_PP(rs_segments), _L, _P],
    "rs_shard_post": [_PP(rs_shard), _PP(rs_segments), _L, _P, _P],
    "rs_shard_collect": [_PP(rs_shard), _P, _P, _P, _P, _P],
    "rs_shard_serve": [_PP(rs_shard), _P, _L, _I, _P, _P, _PP(_P), _L, _P, _P],
    "rs_ffm_fwd_peer": [_PP(rs_tables), _P, _L, _I, _PP(rs_peer_tables), _P, _P, _P, _P],
    "rs_segment_update": [_PP(rs_segments), _L, _PP(rs_update), _P],
    "rs_ffm_bwd_ws_bytes": [_L, _L, _I, _PP(_Z)],
    "rs_ffm_fwd_train": [_PP(rs_tables), _P, _L, _I, C.c_uint64, _P, _P, _P, _P],
    "rs_ffm_bwd_update": [_PP(rs_tables), _P, _L, _I, C.c_uint64, _P, _PP(rs_segments), _PP(rs_update), _P, _Z, _P, _P],
    "rs_replica_sgd": [_PP(_P), _PP(_P), _L, _I, _I, _F, _F, _P],
    "rs_mark_rows": [_PP(rs_segments), _L, _P, _L, _P, _P],
    "rs_replica_update": [_PP(_P), _PP(_P), _PP(_P), _L, _I, _I, _PP(rs_update), _P],
    "rs_adam_dense": [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _I, _P],
    "rs_xembed_fwd": [_PP(rs_xslots), _P, _L, _P, _P, _P],
    "rs_xembed_bag_bwd": [_PP(rs_xslots), _P, _P, _L, _PP(_P), _P, _Z, _P],
    "rs_xembed_bag_ws_bytes": [_PP(rs_xslots), _L, _PP(_Z)],
    "rs_xcol_to_ids": [_P, _L, _I, _I, _P, _P],
    "rs_sigmoid_bce": [_P, _P, _L, _P, _P, _P, _P, _P],
    "rs_sigmoid_bce_bias": [_P, _P, _P, _L, _P, _P, _P, _P, _P, _P],
    "rs_sample_negatives": [_P, _L, _L, _L, _I, C.c_uint64, C.c_uint32, _P, _P, _P, _P],
    "rs_assemble_features": [_P, _P, _P, _L, _I, _P, _L, _I, _L, _P, _P, _P],
    "rs_rank_segments": [_P, _P, _L, _L, _I, _P, _P, _P, _P],
    "rs_mf_rank_ws_bytes": [_L, _L, _I, _I, _PP(_Z)],
    "rs_mf_rank": [_P, _P, _L, _L, _I, _I, _P, _P, _P, _P, _Z, _P],
    "rs_afm_num_parts": [_L, _I, _I, _I, _PP(_I)],
    "rs_afm_fwd": [_P, _L, _I, _I, _I, _P, _P, _P, _P, _P, _P],
    "rs_afm_bwd": [_P, _L, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P],
    "rs_afm_bwd_tc_plan": [_L, _I, _I, _I, _PP(_I), _PP(_Z)],
    "rs_afm_bwd_tc": [_P, _L, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P, _Z, _P],
    "rs_din_num_parts": [_L, _PP(_I)],
    "rs_din_fwd": [_P, _L, _I, _I, _PP(rs_din_weights), _I, _P, _P, _P],
    "rs_din_fwd_tc_ws_bytes": [_L, _I, _I, _I, _I, _PP(_Z)],
    "rs_din_fwd_tc": [_P, _L, _I, _I, _PP(rs_din_weights), _I, _P, _P, _P, _P, _P, _Z, _P],
    "rs_din_bwd_tc": [_P, _L, _I, _I, _PP(rs_din_weights), _I, _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "rs_din_bwd": [_P, _L, _I, _I, _PP(rs_din_weights), _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P],
    "rs_gemm_tn_ws_bytes": [_L, _I, _I, _PP(_Z)],
    "rs_gemm_tn_3xtf32": [_P, _P, _L, _I, _I, _P, _P, _Z, _P],
    "rs_gemm_nt_3xtf32": [_PP(rs_gemm_nt), _P],
    "rs_pnn_outer_ws_bytes": [_L, _I, _I, _PP(_Z), _PP(_Z)],
    "rs_pnn_outer_fwd": [_P, _L, _I, _I, _I, _P, _P, _P, _P, _P, _Z, _P],
    "rs_pnn_outer_bwd": [_P, _P, _L, _I, _I, _P, _P, _P, _P, _P, _Z, _P],
    "rs_gru_fwd": [_P, _L, _I, _I, _P, _P, _P, _P, _P],
    "rs_gru_bwd": [_P, _P, _P, _P, _P, _L, _I, _I, _P, _P, _P],
    "rs_augru_fwd": [_P, _P, _L, _I, _I, _P, _P, _P, _P, _P],
    "rs_augru_bwd": [_P, _P, _P, _P, _P, _P, _L, _I, _I, _P, _P, _P, _P],
    "rs_dien_negatives": [_P, _L, _I, _L, C.c_uint64, _P, _P, _P, _P],
    "rs_dien_aux_fwd": [_P, _L, _P, _L, _P, _L, _L, _I, _I, _P, _P, _P, _P],
    "rs_dien_aux_bwd": [_P, _L, _P, _L, _P, _L, _L, _I, _I, _P, _P, _P, _P, _P, _P],
}

_lib = None


def header_symbols():
    """Names of every function declared in include/recsys_b200.h (parsed, so the test cannot drift)."""
    import re
    path = os.path.join(HERE, "..", "include", "recsys_b200.h")
    with open(path) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(rs_[a-z0-9_]+)\s*\(", text)))


def load():
    """Load (building first if the sources are newer and nvcc exists).  Raises if unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if os.environ.get("RS_NO_BUILD") != "1" and os.path.exists("/usr/local/cuda/bin/nvcc"):
        try:
            from . import build as _b
            _b.build()
        except Exception as e:  # a stale-but-present library is still usable; a missing one is fatal below
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(f"librecsys_b200.so is missing and the nvcc build failed: {e}") from e
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} not found: the CUDA extension is required (no CPU fallback). "
                           "Run `python -c 'import __graft_entry__ as g; g.build()'`.")
    lib = C.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.rs_last_error.argtypes = []
    lib.rs_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().rs_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")
