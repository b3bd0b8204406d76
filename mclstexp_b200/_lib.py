"""ctypes binding of libmclst_b200.so (see include/mclst_b200.h).

There is deliberately NO CPU fallback: if the shared object is missing or a call
fails, the product path raises.  ``load()`` is cheap and needs no GPU (the CPU
test-suite uses it to check that every symbol the header declares is exported).
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import List

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, os.environ.get("MCLST_LIB_NAME", "libmclst_b200.so"))
HEADER = os.path.join(os.path.dirname(HERE), "include", "mclst_b200.h")

# weight modes / flags (mirrors of the header enums)
W_INV_SQ_L1, W_INV_SQ_L2, W_SIMILARITY, W_UNIFORM, W_BLEEP_EXP = range(5)
WEIGHT_MODES = {"inv_sq_l1": 0, "inv_sq_l2": 1, "similarity": 2, "uniform": 3, "bleep_exp": 4}
FM_DEFAULT, FM_EXACT_ONLY, FM_BANK_PACKED, FM_NO_SPECULATION = 0, 1, 2, 4
T_EYE, T_SOFT_DIV, T_SOFT_MUL = 0, 1, 2
LOSS_STAT_ROWS = 9        # MCLST_LOSS_STAT_ROWS: rl, cl, za, wbar, cs, diag, rl_lo, cl_lo, za_lo

_lib = None


class MclstError(RuntimeError):
    pass


def header_symbols() -> List[str]:
    """Every function the public header declares."""
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mclst_[a-z0-9_]+)\s*\(", src)))


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MclstError(
            f"{LIB_PATH} is missing: build it with `python -m mclstexp_b200.build` "
            "(there is no CPU fallback for the mclSTExp hot path)")
    lib = C.CDLL(LIB_PATH)
    p, i64, i32, sz = C.c_void_p, C.c_int64, C.c_int, C.c_size_t
    lib.mclst_version.restype = i32
    lib.mclst_last_error.restype = C.c_char_p
    lib.mclst_launch_count.restype = i64
    lib.mclst_device_info.argtypes = [C.POINTER(i32)] * 3
    lib.mclst_profile_enable.argtypes = [i32]
    lib.mclst_profile_collect.argtypes = [C.c_char_p, C.POINTER(C.c_float), i32, C.POINTER(i32)]
    lib.mclst_read_counters.argtypes = [p, C.POINTER(i64), p]
    lib.mclst_find_matches_workspace_bytes.argtypes = [i64, i64, i32, i32, i32, C.POINTER(sz)]
    lib.mclst_find_matches_tc_eligible.argtypes = [i64, i32, i32, i32]
    lib.mclst_find_matches.argtypes = [p, i64, i64, p, i64, i64, i32, i32, i64, p, p, p, sz, i32, p]
    lib.mclst_find_matches_pack_bank.argtypes = [p, i64, i64, i32, i32, p, sz, p]
    lib.mclst_find_matches_seed.argtypes = [p, i64, i64, p, i64, i64, i32, i32, i32, p, p, p, sz, i32, p]
    lib.mclst_find_matches_main.argtypes = [p, i64, i64, p, i64, i64, i32, i32, i64, p, p, p, i32, p, p, sz,
                                            i32, p]
    lib.mclst_find_matches_candidates.argtypes = [p, i64, i64, p, i64, i64, i32, i32, i32, p, p, p, p, sz, i32, p]
    lib.mclst_find_matches_finish.argtypes = lib.mclst_find_matches_main.argtypes
    lib.mclst_debug_similarity.argtypes = [p, i64, i64, p, i64, i64, i32, p, i64, p, sz, p]
    lib.mclst_gene_metrics_scratch_doubles.argtypes = [i32, C.POINTER(sz)]
    lib.mclst_gene_metrics.argtypes = [p, i64, i32, p, i64, i32, i64, i32, p, p, p, p, p, p]
    lib.mclst_merge_topk.argtypes = [p, p, p, i32, i64, i32, p, p, p, p]
    lib.mclst_neighbor_weights.argtypes = [p, p, i64, i32, i32, p, p]
    lib.mclst_contrastive_loss_workspace_bytes.argtypes = [i32, i32, i32, i64, C.POINTER(sz)]
    lib.mclst_contrastive_loss_phase.argtypes = [p, i64, p, i64, i32, i32, C.c_float, i32, i64, i64, i32, p,
                                                 p, p, i64, p, i64, p, sz, p]
    lib.mclst_contrastive_loss.argtypes = [p, i64, p, i64, i32, i32, C.c_float, i32, p, p, i64, p, i64,
                                           p, sz, p]
    f32 = C.c_float
    lib.mclst_embed_add.argtypes = [p, i64, p, i64, p, p, i32, i32, i32, p, i64, p, p]
    lib.mclst_embed_add_backward.argtypes = [p, i64, p, i64, i32, i32, i32, p, p, p]
    lib.mclst_embed_add_backward_accumulate.argtypes = lib.mclst_embed_add_backward.argtypes
    lib.mclst_zero_fill_background.argtypes = [p, i64, i32, p]
    lib.mclst_layernorm_forward.argtypes = [p, i64, p, p, i64, i32, f32, p, i64, p, p, p]
    lib.mclst_layernorm_backward.argtypes = [p, i64, p, i64, p, p, p, i64, i32, p, i64, p, p, p, sz, p]
    lib.mclst_gelu_forward.argtypes = [p, p, i64, p]
    lib.mclst_gelu_backward.argtypes = [p, p, p, i64, p]
    lib.mclst_softmax_forward.argtypes = [p, i64, i64, i32, p]
    lib.mclst_softmax_backward.argtypes = [p, p, i64, i64, i32, p]
    lib.mclst_softmax_blockdiag.argtypes = [p, i64, i64, i32, i32, i64, p]
    lib.mclst_col_sum.argtypes = [p, i64, i64, i32, p, p]
    lib.mclst_matmul_workspace_bytes.argtypes = [i64, i64, i64, i32, C.POINTER(sz)]
    lib.mclst_matmul.argtypes = [p, i64, i32, i64, p, i64, i32, i64, p, i64, i64, i64, i64, i64, i32,
                                 C.c_float, p, i32, p, i32, p, sz, p]
    lib.mclst_find_matches_dist.argtypes = [p, i64, i64, p, i64, i64, i32, i32, i64, p, p, p, i32, p, sz,
                                            i32, p]
    lib.mclst_weighted_average.argtypes = [p, i64, i64, p, i64, i32, i32, p, i64, i64, i32, p, p, p,
                                           i32, i64, i32, p, p, i32, p]
    lib.mclst_retrieve_workspace_bytes.argtypes = [i64, i64, i32, i32, i32, C.POINTER(sz)]
    lib.mclst_retrieve.argtypes = [p, i64, i64, p, i64, i32, i32, p, i64, i64, i32, i32, i32, p, p, p, p, i32,
                                   p, sz, i32, p]
    lib.mclst_neighbor_distances.argtypes = [p, i64, i64, p, i64, i64, i32, p, i32, i64, i32, p, p]
    lib.mclst_weighted_gather.argtypes = [p, i64, i64, i32, i32, p, p, i64, i32, i64, p, p]
    f64 = C.c_double
    lib.mclst_debug_spec_rank.argtypes = [i32, f64]
    lib.mclst_debug_lane_plan.argtypes = [i64, i64, i32, i32, p, i64, C.POINTER(i64), C.POINTER(i32)]
    lib.mclst_debug_gemm_variant.argtypes = [i64, i64, i32, C.POINTER(i32), C.POINTER(i32)]
    lib.mclst_adam_coef_bytes.argtypes = [i32]
    lib.mclst_adam_coef_bytes.restype = sz
    lib.mclst_adam_set_step.argtypes = [p, i32, i32, f64, f64, f64, f64, f64, p]
    lib.mclst_adam_dense.argtypes = [p, p, p, p, i64, p, i32, p]
    lib.mclst_adam_lazy_rows.argtypes = [p, p, p, p, p, i32, i32, p, i64, i32, i32, p, i64, p, i32, p, p, p]
    lib.mclst_adam_lazy_flush.argtypes = [p, p, p, p, i32, i32, p, i32, p]
    for name in header_symbols():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        if fn.restype is C.c_int and name not in ("mclst_version",):
            fn.restype = i32
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().mclst_last_error().decode(errors="replace")
        raise MclstError(f"{what or 'libmclst_b200'} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(load().mclst_launch_count())


def profile_enable(on: bool) -> None:
    check(load().mclst_profile_enable(int(on)), "profile_enable")


def profile_collect(cap: int = 65536):
    """[(kernel name, milliseconds)] for every traced launch since the last collect."""
    names = C.create_string_buffer(48 * cap)
    ms = (C.c_float * cap)()
    n = C.c_int()
    check(load().mclst_profile_collect(names, ms, cap, C.byref(n)), "profile_collect")
    raw = names.raw
    return [(raw[48 * i:48 * i + 48].split(b"\0")[0].decode(), float(ms[i])) for i in range(n.value)]


def require_cuda(*tensors) -> None:
    import torch
    if not torch.cuda.is_available():
        raise MclstError("no CUDA device: the mclSTExp hot path runs only on a B200 "
                         "(sm_100a); there is no CPU fallback")
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise MclstError("expected CUDA tensors (no CPU fallback)")


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return C.c_void_p(0 if t is None else t.data_ptr())
