"""ctypes binding of libccr_b200.so (C ABI: include/ccr_b200.h).

The product path has NO CPU fallback: if the shared library is missing, or a CUDA device is
not present when a kernel is requested, this raises instead of computing something else.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CCR_B200_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libccr_b200.so")

MASK_NONE, MASK_SET, MASK_ADD = 0, 1, 2
ALGO_AUTO, ALGO_SIMT, ALGO_TCGEN05 = 0, 1, 2
FLAG_ALLOW_SHORT = 0x10
FLAG_PACKED_KEYS = 0x20
FLAG_F16 = 0x40  # q and items hold fp16 instead of bf16
MAX_K = 2048
ABI_VERSION = 6

OK, EINVAL, EUNSUPPORTED, EWORKSPACE, ECUDA, EK_RANGE = 0, -1, -2, -3, -4, -5

# every symbol include/ccr_b200.h declares (tests check they are all exported)
EXPORTS = [
    "ccr_abi_version",
    "ccr_last_error_string",
    "ccr_score_topk_bf16",
    "ccr_score_topk_workspace_bytes",
    "ccr_merge_topk",
    "ccr_merge_topk_keys",
    "ccr_unpack_topk_keys",
    "ccr_mask_column_shard",
    "ccr_ingest_rows_f32",
    "ccr_normalize_rows_bf16",
    "ccr_ingest_rows_f32_f16",
    "ccr_normalize_rows_f16",
    "ccr_score_dense_f32",
    "ccr_score_dense_f16",
    "ccr_choose_algo",
    "ccr_plan_info",
    "ccr_set_profile_events",
    "ccr_set_status_record",
    "ccr_debug_reload_env",
    "ccr_argsort_workspace_bytes",
    "ccr_argsort_scores_f32",
    "ccr_first_hit_rank",
    "ccr_topk_dense_workspace_bytes",
    "ccr_topk_dense_f32",
    "ccr_bm25_build_impacts",
    "ccr_bm25_head_row_pitch",
    "ccr_bm25_build_head_rows",
    "ccr_bm25_topk_workspace_bytes",
    "ccr_bm25_topk",
    "ccr_bm25_scores_f64",
    "ccr_exact_k_candidates",
    "ccr_exact_error_bound",
    "ccr_score_topk_exact_workspace_bytes",
    "ccr_score_topk_exact",
    "ccr_ingest_rows_f32_f32",
    "ccr_rerank_exact_workspace_bytes",
    "ccr_rerank_exact",
    "ccr_threshold_compact",
    "ccr_score_dense_exact",
]

_lib = None


class CcrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libccr_b200 error {code}: {msg}")
        self.code = code


def lib():
    """Load (once) and return the ctypes handle; raise if the CUDA extension is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA extension is required (no CPU fallback). "
            "Build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`make -C crowd-coachable-recommendations_b200/csrc`."
        )
    L = ctypes.CDLL(LIB_PATH)
    c = ctypes
    vp, i64, i32, sz = c.c_void_p, c.c_int64, c.c_int, c.c_size_t
    L.ccr_abi_version.restype = i32
    L.ccr_last_error_string.restype = c.c_char_p
    L.ccr_score_topk_bf16.restype = i32
    L.ccr_score_topk_bf16.argtypes = [vp, i64, i64, vp, i64, i64, i32, i32, vp, vp, vp, i64, i64, i32, i64,
                                      vp, vp, vp, vp, sz, i32, vp]
    L.ccr_score_topk_workspace_bytes.restype = sz
    L.ccr_score_topk_workspace_bytes.argtypes = [i64, i64, i32, i32, i64, i64, i32]
    L.ccr_merge_topk.restype = i32
    L.ccr_merge_topk.argtypes = [vp, vp, i32, i64, i32, i32, vp, vp, vp, vp]
    L.ccr_merge_topk_keys.restype = i32
    L.ccr_merge_topk_keys.argtypes = [vp, i32, i64, i32, i32, vp, vp, vp, vp]
    L.ccr_unpack_topk_keys.restype = i32
    L.ccr_unpack_topk_keys.argtypes = [vp, i64, vp, vp, vp]
    L.ccr_mask_column_shard.restype = i32
    L.ccr_mask_column_shard.argtypes = [vp, vp, vp, i64, i64, i64, vp, vp, vp, vp]
    L.ccr_ingest_rows_f32.restype = i32
    L.ccr_ingest_rows_f32.argtypes = [vp, i64, i32, i64, vp, i64, i32, vp]
    L.ccr_normalize_rows_bf16.restype = i32
    L.ccr_normalize_rows_bf16.argtypes = [vp, i64, i32, i64, vp, i64, vp]
    L.ccr_score_dense_f32.restype = i32
    L.ccr_score_dense_f32.argtypes = [vp, i64, i64, vp, i64, i64, i32, vp, i64, vp]
    L.ccr_ingest_rows_f32_f16.restype = i32
    L.ccr_ingest_rows_f32_f16.argtypes = [vp, i64, i32, i64, vp, i64, i32, vp, vp]
    L.ccr_normalize_rows_f16.restype = i32
    L.ccr_normalize_rows_f16.argtypes = [vp, i64, i32, i64, vp, i64, vp]
    L.ccr_score_dense_f16.restype = i32
    L.ccr_score_dense_f16.argtypes = [vp, i64, i64, vp, i64, i64, i32, vp, i64, vp]
    L.ccr_choose_algo.restype = i32
    L.ccr_choose_algo.argtypes = [i64, i64, i32, i32]
    L.ccr_set_profile_events.restype = None
    L.ccr_set_profile_events.argtypes = [vp, vp]
    L.ccr_plan_info.restype = i32
    L.ccr_plan_info.argtypes = [i64, i64, i32, i32, i64, i64, i32, c.POINTER(c.c_int32)]
    L.ccr_set_status_record.restype = None
    L.ccr_set_status_record.argtypes = [vp]
    L.ccr_debug_reload_env.restype = None
    L.ccr_debug_reload_env.argtypes = []
    L.ccr_argsort_workspace_bytes.restype = sz
    L.ccr_argsort_workspace_bytes.argtypes = [i64]
    L.ccr_argsort_scores_f32.restype = i32
    L.ccr_argsort_scores_f32.argtypes = [vp, i64, i64, i64, vp, vp, vp, i64, i32, vp, vp, vp, sz, vp]
    L.ccr_first_hit_rank.restype = i32
    L.ccr_first_hit_rank.argtypes = [vp, i64, i32, vp, vp, vp, vp]
    f64 = c.c_double
    L.ccr_topk_dense_workspace_bytes.restype = sz
    L.ccr_topk_dense_workspace_bytes.argtypes = [i64, i64, i32, i64, i64]
    L.ccr_topk_dense_f32.restype = i32
    L.ccr_topk_dense_f32.argtypes = [vp, i64, i64, i64, i32, vp, vp, vp, i64, i64, i32, vp, vp, vp, vp, sz, vp]
    L.ccr_bm25_build_impacts.restype = i32
    L.ccr_bm25_build_impacts.argtypes = [vp, vp, vp, vp, vp, f64, i64, i64, vp, vp]
    L.ccr_bm25_topk_workspace_bytes.restype = sz
    L.ccr_bm25_topk_workspace_bytes.argtypes = [i64, i64, i32]
    L.ccr_bm25_topk.restype = i32
    L.ccr_bm25_topk.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, i32, vp, vp, vp, sz, vp]
    L.ccr_bm25_scores_f64.restype = i32
    L.ccr_bm25_scores_f64.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, vp, i64, vp]
    L.ccr_bm25_head_row_pitch.restype = i64
    L.ccr_bm25_head_row_pitch.argtypes = [i64]
    L.ccr_bm25_build_head_rows.restype = i32
    L.ccr_bm25_build_head_rows.argtypes = [vp, vp, vp, vp, i32, i64, i64, vp, vp, vp]
    L.ccr_exact_k_candidates.restype = i32
    L.ccr_exact_k_candidates.argtypes = [i64, i64, i32, i32, i32]
    L.ccr_exact_error_bound.restype = f64
    L.ccr_exact_error_bound.argtypes = [f64, f64, i32, i32]
    L.ccr_score_topk_exact_workspace_bytes.restype = sz
    L.ccr_score_topk_exact_workspace_bytes.argtypes = [i64, i64, i32, i32, i64, i64, i32]
    L.ccr_score_topk_exact.restype = i32
    L.ccr_score_topk_exact.argtypes = [vp, vp, i64, i64, vp, vp, i64, i64, i32, i32, vp, vp, vp, vp, i64, i64, i32,
                                       i64, vp, vp, vp, vp, vp, vp, vp, sz, i32, vp]
    L.ccr_ingest_rows_f32_f32.restype = i32
    L.ccr_ingest_rows_f32_f32.argtypes = [vp, i64, i32, i64, vp, i64, i32, vp, vp]
    L.ccr_rerank_exact_workspace_bytes.restype = sz
    L.ccr_rerank_exact_workspace_bytes.argtypes = [i64, i64, i64]
    L.ccr_rerank_exact.restype = i32
    L.ccr_rerank_exact.argtypes = [vp, i64, i64, vp, i64, i64, i32, i32, vp, vp, i64, vp, vp, vp, i64, i32, i64,
                                   vp, vp, vp, vp, sz, i32, vp]
    L.ccr_threshold_compact.restype = i32
    L.ccr_threshold_compact.argtypes = [vp, i64, i64, i64, vp, vp, vp, vp]
    L.ccr_score_dense_exact.restype = i32
    L.ccr_score_dense_exact.argtypes = [vp, i64, i64, vp, i64, i64, i32, vp, i64, vp]
    if L.ccr_abi_version() != ABI_VERSION:
        raise RuntimeError("libccr_b200 ABI version mismatch")
    _lib = L
    return L


def check(rc):
    if rc != OK:
        msg = lib().ccr_last_error_string().decode("utf-8", "replace")
        if rc == EK_RANGE:
            raise RuntimeError(msg)  # torch.topk raises RuntimeError("selected index k out of range")
        if rc in (EINVAL, EUNSUPPORTED):
            raise ValueError(f"libccr_b200: {msg}")
        raise CcrError(rc, msg)


def plan_info(B, n_items, D, k, flags=0, mask_nnz=0, mask_max_row_nnz=-1):
    arr = (ctypes.c_int32 * 8)()
    check(lib().ccr_plan_info(B, n_items, D, k, mask_nnz, mask_max_row_nnz, flags, arr))
    return {"n_q_tiles": arr[0], "n_splits": arr[1], "cand_capacity": arr[2], "algo": arr[3], "two_cta": arr[4],
            "seed_items": arr[5], "n_kernel_launches": arr[6], "lead_tiles": arr[7]}


def exact_k_candidates(B, n_items, D, k, flags=0):
    """k': candidates per row the scan stage of an exact search returns (the plan's rule, no GPU needed)."""
    kc = lib().ccr_exact_k_candidates(B, n_items, D, k, flags)
    if kc < 0:
        check(kc)
    return kc


def reload_env():
    """Diagnostics: make libccr_b200 re-read the CCR_* knobs after os.environ was changed."""
    lib().ccr_debug_reload_env()
