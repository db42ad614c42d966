"""ctypes binding of the C ABI declared in include/tcar_b200.h.

There is deliberately NO fallback: if libtcar_b200.so is missing or a call fails, we raise.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtcar_b200.so")

H, HP, TH, XW, PW, NBINS, KEXT, QROWS, MAXT, TOPK, CHUNK, NCAND_CHUNKS = 250, 256, 64, 500, 320, 139, 640, 512, 40, 20, 8, 32
NORM_SPLIT = 8
EXP_LIMIT2 = 80.0        # TCAR_EXP_LIMIT2
EVAL_OFF_SCORES, EVAL_OFF_IDS, EVAL_OFF_NGT = 0, QROWS * TOPK, 2 * QROWS * TOPK      # TCAR_EVAL_OFF_*
EVAL_OFF_SUMEXP, EVAL_OFF_ROWMAX, EVAL_BLOCK_WORDS = EVAL_OFF_NGT + QROWS, EVAL_OFF_NGT + 2 * QROWS, EVAL_OFF_NGT + 3 * QROWS
EVAL_NSEL = 33           # TCAR_EVAL_NSEL
# candidate-list block of one (item range, query owner) pair in the two-stage sharded evaluation:
# [vals 512x33 f32 | chunk ids 512x33 i32 | sumexp 512 f32 | rowmax 512 f32]
SEL_OFF_IDS, SEL_OFF_SUMEXP = QROWS * EVAL_NSEL, 2 * QROWS * EVAL_NSEL
SEL_OFF_ROWMAX, SEL_BLOCK_WORDS = SEL_OFF_SUMEXP + QROWS, SEL_OFF_SUMEXP + 2 * QROWS
MAX_PEERS, PEER_HANDLE_BYTES = 16, 64      # TCAR_MAX_PEERS, TCAR_PEER_HANDLE_BYTES
BIN_OFF = (0, 13, 45, 53, 78, 139)
CLUSTER_PAIR = -2      # TCAR_CLUSTER_PAIR: tcar_score_fwd with tcgen05.mma.cta_group::2 CTA pairs
RERANK_MAXL = 2048     # TCAR_RERANK_MAXL: longest candidate list of tcar_rerank
RECOMMEND_MAXK = 256   # TCAR_RECOMMEND_MAXK: largest K of tcar_recommend
RECOMMEND_MAXX = 1024  # TCAR_RECOMMEND_MAXX: exclusion entries per session of tcar_recommend, clicks included
RECOMMEND_MAXG = 1024  # TCAR_RECOMMEND_MAXG: most categories of tcar_recommend_category
DECAY_MAX_AGE = 2 ** 23 - 1  # TCAR_DECAY_MAX_AGE: ages of the freshness decay saturate here (clock units)

_P, _I, _F, _LL = C.c_void_p, C.c_int, C.c_float, C.c_longlong

# name -> argtypes (all return int)
SIGNATURES = {
    "tcar_gather_fwd": [_P] * 15 + [_I, _I, _P],
    "tcar_assemble_batch": [_P] * 4 + [_I] * 4 + [_P, _I, C.c_ulonglong, C.c_ulonglong, _P, _P],
    "tcar_impression_negatives": [_P, _P, _P, _I, _I, _I, C.c_ulonglong, C.c_ulonglong, _P, _P],
    "tcar_pool_fwd": [_P] * 10 + [_I, _I, _P],
    "tcar_pool_bwd": [_P] * 16 + [_I, _I, _P],
    "tcar_build_iext": [_P] * 4 + [_I, _I, _P],
    "tcar_clip_time_tables": [_P] * 7 + [_P],
    "tcar_build_query": [_P] * 10 + [_I, _P],
    "tcar_score_fwd": [_P] * 7 + [_I] * 5 + [_P],
    "tcar_score_fwd_guarded": [_P] * 9 + [_I] * 5 + [_P],
    "tcar_score_fwd_tiles": [_I],
    "tcar_score_fwd_window": [_P] * 9 + [_I] * 3 + [_P],
    "tcar_score_fwd_decay": [_P] * 9 + [_I] * 3 + [_P],
    "tcar_ce_finish": [_P] * 3 + [_I, _I, _P],
    "tcar_ce_finish_guarded": [_P] * 5 + [_I, _I, _I, _P],
    "tcar_neg_loss": [_P] * 9 + [_I, _I, _P],
    "tcar_loss_combine": [_P, _P, _P, _I, _P],
    "tcar_ce_from_sums": [_P, _I, _P, _P, _P, _I, _P],
    "tcar_score_bwd_q_splits": [_I, _I],
    "tcar_score_bwd_q": [_P] * 4 + [_I, _I, _P],
    "tcar_score_bwd_finish": [_P] * 13 + [_I, _P],
    "tcar_score_bwd_i": [_P] * 4 + [_I, _I, _I, _P],
    "tcar_score_bwd_i_acc": [_P] * 4 + [_I, _I, _I, _I, _P],
    "tcar_score_bwd_i_multi": [_P, _LL, _P, _LL, _P, _P, _P, _I, _I, _I, _P],
    "tcar_score_bwd_i_ctas": [_I],
    "tcar_sqnorm_combine": [_P, _I, _P, _I, _P, _P],
    "tcar_small_table_grads": [_P] * 23 + [_I, _I, _P],
    "tcar_act_bwd_colsum": [_P] * 4 + [_I, _I, _I, _I, _P],
    "tcar_col_jobs": [_P, _I, _P],
    "tcar_gemm_tf32": [_P, _I, _I, _I, _P, _I, _P, _I, _I, _I, _I, _P, _P],
    "tcar_gemm_tf32_group": [_P, _I, _P],
    "tcar_gemm_tf32_splits": [_I, _I, _I, _I],
    "tcar_gemm_tf32_part_elems": [_I, _I, _I],
    "tcar_debug_gemm_trace": [_P],
    "tcar_prep_weights": [_P, _P, _I, _P, _P, _P],
    "tcar_scatter_add_rows": [_P] * 13 + [_I] * 4 + [_P],
    "tcar_scatter_add_rows_range": [_P] * 13 + [_I] * 6 + [_P],
    "tcar_peer_export": [_P, _P, _P],
    "tcar_peer_open": [_P, _LL, _P],
    "tcar_peer_close": [_P, _LL],
    "tcar_peer_fetch_rows": [_P, _P, _P, _I, _I, _I, _P, _P, _I, _I, _P, _P],
    "tcar_rowsum_finish": [_P, _P, _I, _I, _I, _P],
    "tcar_score_fwd_groups": [_P, _LL, _P, _LL, _P, _P, _LL, _P, _LL, _P, _I, _I, _I, _I, _P],
    "tcar_score_fwd_groups_guarded": [_P, _LL, _P, _LL, _P, _P, _LL, _P, _LL, _P, _P, _P, _I, _I, _I, _I, _P],
    "tcar_score_fwd_multi": [_P, _LL, _P, _LL, _P, _P, _LL, _P, _LL, _P, _P, _P, _I, _I, _I, _P],
    "tcar_score_fwd_multi_eval": [_P, _LL, _P, _LL, _P, _P, _LL, _P, _LL, _P, _LL, _P, _P, _LL, _P, _I, _I, _I, _P],
    "tcar_rowmax_groups": [_P, _LL, _P, _I, _P, _I, _P],
    "tcar_ce_finish_groups": [_P, _P, _LL, _P, _P, _LL, _I, _P, _I, _I, _P],
    "tcar_score_bwd_q_multi_part_elems": [_I],
    "tcar_score_bwd_q_multi": [_P, _LL, _P, _P, _P, _P, _I, _I, _P],
    "tcar_score_bwd_q_groups": [_P, _LL, _P, _P, _P, _LL, _P, _LL, _I, _P, _I, _I, _P],
    "tcar_score_bwd_i_groups": [_P, _LL, _P, _LL, _P, _P, _P, _I, _I, _I, _P],
    "tcar_scatter_add_rows_groups": [_P, _LL, _P, _LL, _P, _P, _P, _P, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _P],
    "tcar_scatter_add_rows_multi": [_P, _LL, _P, _LL, _P, _P, _P, _P, _P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _P],
    "tcar_sqnorm_segments": [_P] * 3 + [_I, _P],
    "tcar_sqnorm_big": [_P] * 3 + [_LL, _P],
    "tcar_update_norms": [_P, _P, _P, _I, _P, _I, _P, _I, _P, _P, _P, _P, _P],
    "tcar_adam_small": [_P] * 6 + [_I, _P, _F, _F, _P],
    "tcar_adam_item": [_P] * 6 + [_F, _F, _P, _I, _I, _P, _I, _P],
    "tcar_adam_item_rows": [_P] * 6 + [_F, _F, _P, _P, _I, _P, _I, _P, _I, _P],
    "tcar_adam_item_rows_groups": [_P] * 6 + [_F, _F, _P, _P, _LL, _P, _I, _I, _I, _P, _I, _I, _P],
    "tcar_refresh_iext_items": [_P, _P, _I, _P],
    "tcar_eval_topk_certified": [_P] * 11 + [_I] * 4 + [_P] * 3 + [_P],
    "tcar_eval_select": [_P] * 4 + [_I] * 4 + [_P],
    "tcar_eval_rescore": [_P, _P, _I, _LL] + [_P] * 9 + [_I, _I] + [_P] * 3 + [_P],
    "tcar_eval_topk_widen": [_P] * 13 + [_I] * 4 + [_P, _P],
    "tcar_eval_topk_widen_ws_bytes": [_I],
    "tcar_eval_select_groups": [_P, _LL, _P, _LL, _P, _P, _LL, _P, _I, _I, _I, _I, _P],
    "tcar_eval_topk_widen_groups": [_P, _LL, _P, _LL, _P, _P, _P, _LL, _P, _P, _P, _P, _P, _LL, _P, _P, _P, _LL, _P,
                                    _I, _I, _I, _I, _P, _P],
    "tcar_catalog_stats": [_P, _P, _I, _I, _P, _P],
    "tcar_topk_merge": [_P] * 4 + [_I, _I, _P],
    "tcar_eval_merge": [_P, _LL, _P, _P, _P, _P, _I, _I, _P],
    "tcar_eval_ce_combine": [_P, _P, _LL, _P, _I, _I, _P],
    "tcar_eval_merge_flagged": [_P, _LL, _P, _P, _P, _P, _I, _I, _P],
    "tcar_rerank": [_P] * 8 + [_I] * 3 + [_P] * 4 + [_P],
    "tcar_recommend_ws_bytes": [_I],
    "tcar_recommend": [_P] * 11 + [_I] * 5 + [_P] * 4 + [_P],
    "tcar_recommend_window": [_P] * 11 + [_I] * 5 + [_P] * 7 + [_P],
    "tcar_recommend_decay": [_P] * 11 + [_I] * 5 + [_P] * 9 + [_P],
    "tcar_recommend_category_ws_bytes": [_I],
    "tcar_recommend_category": [_P] * 10 + [_I] * 4 + [_P] * 3 + [_I] + [_P] * 2 + [_I] + [_P] * 4 + [_P],
}

_lib = None


class TcarNativeError(RuntimeError):
    pass


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TcarNativeError(
                f"{LIB_PATH} not found: build it with __graft_entry__.build() -- there is no CPU/PyTorch fallback")
        l = C.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(l, name)
            fn.argtypes = argtypes
            fn.restype = C.c_longlong if name.endswith(("_part_elems", "_ws_bytes")) else C.c_int
        _lib = l
    return _lib


def ptr(t):
    """Device pointer of a torch tensor (or None) as a plain int: the c_void_p argtypes convert it, and building a
    ctypes object per argument was a measurable share of the ~0.5 ms a step's ~35 calls cost the host."""
    return None if t is None else t.data_ptr()


_raw_stream = None
_dev_index = None


def stream_ptr():
    """cudaStream_t of torch's current stream on the current device (torch._C._cuda_getCurrentRawStream: one C call
    instead of building a torch.cuda.Stream object per launch)."""
    global _raw_stream, _dev_index
    if _raw_stream is None:
        import torch
        _raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
        if _raw_stream is None:
            _raw_stream = lambda idx: torch.cuda.current_stream().cuda_stream
        _dev_index = torch.cuda.current_device()
    return _raw_stream(_dev_index)


def call(name, *args):
    """Invoke a C-ABI entry point on the current torch stream; raise on a non-zero return code."""
    rc = getattr(lib(), name)(*args, stream_ptr())
    if rc != 0:
        raise TcarNativeError(f"{name} failed with code {rc}")
    return rc


class GemmSeg(C.Structure):
    """tcar_gemm_seg of include/tcar_b200.h."""
    _fields_ = [("a", C.c_void_p), ("b", C.c_void_p), ("b_lo", C.c_void_p), ("lda", C.c_int), ("ldb", C.c_int),
                ("k", C.c_int), ("a_mn_major", C.c_int), ("b_mn_major", C.c_int), ("a_koff", C.c_int)]


class GemmProblem(C.Structure):
    """tcar_gemm_problem of include/tcar_b200.h."""
    _fields_ = [("segs", GemmSeg * 3), ("nseg", C.c_int), ("M", C.c_int), ("N", C.c_int), ("bias", C.c_void_p),
                ("act", C.c_int), ("C", C.c_void_p), ("ldc", C.c_int), ("accumulate", C.c_int), ("precise", C.c_int),
                ("splits", C.c_int), ("part", C.c_void_p), ("C2", C.c_void_p), ("c2_row0", C.c_int)]


def _seg(sg):
    a, lda, a_mn, b, b_lo, ldb, b_mn, k = sg[:8]
    return GemmSeg(a.data_ptr(), b.data_ptr(), b_lo.data_ptr() if b_lo is not None else None, lda, ldb, k,
                   int(a_mn), int(b_mn), sg[8] if len(sg) > 8 else 0)


def problem(segs, M, N, out, ldc, bias=None, act=0, accumulate=False, precise=False, splits=1, part=None, out2=None,
            out2_row0=0):
    """One tcar_gemm_problem; segs as in gemm().  out2: rows >= out2_row0 are also written to out2 (pitch ldc)."""
    q = GemmProblem()
    for i, sg in enumerate(segs):
        q.segs[i] = _seg(sg)
    q.nseg, q.M, q.N = len(segs), M, N
    q.bias = bias.data_ptr() if bias is not None else None
    q.act, q.C, q.ldc = act, out.data_ptr(), ldc
    q.accumulate, q.precise, q.splits = int(accumulate), int(precise), splits
    q.part = part.data_ptr() if part is not None else None
    q.C2 = out2.data_ptr() if out2 is not None else None
    q.c2_row0 = out2_row0
    return q


def gemm_group(problems):
    """Launch several independent problems (built with problem()) as one kernel (+ one split-reduction kernel)."""
    arr = (GemmProblem * len(problems))(*problems)
    LAUNCHES["count"] += 1 + (1 if any(q.splits > 1 for q in problems) else 0)
    return call("tcar_gemm_tf32_group", C.cast(arr, C.c_void_p), len(problems))


def gemm(segs, M, N, out, ldc, bias=None, act=0, accumulate=False, precise=False, splits=1, part=None):
    """C[M,N] = act(sum_s A_s . B_s + bias) on the tensor cores.  segs: list of
    (a, lda, a_mn, b, b_lo, ldb, b_mn, k[, a_koff]) with a / b / b_lo torch tensors (data_ptr = operand origin)."""
    arr = (GemmSeg * len(segs))()
    for i, sg in enumerate(segs):
        a, lda, a_mn, b, b_lo, ldb, b_mn, k = sg[:8]
        arr[i] = GemmSeg(a.data_ptr(), b.data_ptr(), b_lo.data_ptr() if b_lo is not None else None, lda, ldb, k,
                         int(a_mn), int(b_mn), sg[8] if len(sg) > 8 else 0)
    LAUNCHES["count"] += 1 + (1 if splits > 1 else 0)
    return call("tcar_gemm_tf32", C.cast(arr, C.c_void_p), len(segs), M, N, ptr(bias), act, ptr(out), ldc,
                int(accumulate), int(precise), splits, ptr(part))


class ColJob(C.Structure):
    """tcar_col_job of include/tcar_b200.h."""
    _fields_ = [("a", C.c_void_p), ("y", C.c_void_p), ("dz", C.c_void_p), ("out", C.c_void_p),
                ("scratch", C.c_void_p), ("rows", C.c_int), ("cols", C.c_int), ("ld", C.c_int), ("mode", C.c_int)]


def col_jobs(jobs):
    """jobs: list of (a, y, dz | None, out, rows, cols, ld, mode[, scratch]) -- one launch (tcar_col_jobs)."""
    arr = (ColJob * len(jobs))()
    for i, job in enumerate(jobs):
        a, y, dz, out, rows, cols, ld, mode = job[:8]
        scratch = job[8] if len(job) > 8 else None
        arr[i] = ColJob(a.data_ptr(), y.data_ptr(), dz.data_ptr() if dz is not None else None, out.data_ptr(),
                        scratch.data_ptr() if scratch is not None else None, rows, cols, ld, mode)
    LAUNCHES["count"] += 1
    return call("tcar_col_jobs", C.cast(arr, C.c_void_p), len(jobs))


LAUNCHES = {"count": 0}


def counted_call(name, nlaunch, *args):
    LAUNCHES["count"] += nlaunch
    return call(name, *args)
