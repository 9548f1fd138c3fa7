"""ctypes binding of libnrms_b200.so (the C-ABI declared in include/nrms_b200.h).

There is NO fallback: if the shared library is missing or a call fails this module raises.
Build it with `python newsrecommendationsystem_b200/csrc/build.py` (or `__graft_entry__.build()`).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnrms_b200.so")

MODE_FP32 = 0
MODE_TF32 = 1
MODES = {"fp32": MODE_FP32, "tf32": MODE_TF32}

_vp, _i64, _i32, _f32, _u64, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_uint64, C.c_size_t

# name -> (restype, argtypes); mirrors include/nrms_b200.h one to one
SIGNATURES = {
    "nrms_last_error": (C.c_char_p, []),
    "nrms_abi_version": (_i32, []),
    "nrms_launch_count": (_i64, []),
    "nrms_set_option": (_i32, [C.c_char_p, _i32]),
    "nrms_get_stat": (C.c_double, [C.c_char_p]),
    "nrms_encoder_stash_bytes": (_sz, [_i64, _i32]),
    "nrms_encoder_fwd_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32, _i64]),
    "nrms_encoder_bwd_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "nrms_news_encoder_fwd": (_i32, [_vp, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                     _f32, _u64, _u64, _i32, _vp]),
    "nrms_news_encoder_i32_fwd": (_i32, [_vp, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nrms_news_encoder_bwd": (_i32, [_vp, _vp, _i64, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _vp, _sz, _f32, _u64, _u64, _i32, _vp]),
    "nrms_user_encoder_fwd": (_i32, [_vp, _i64, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "nrms_user_encoder_bwd": (_i32, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                                     _i32, _vp]),
    "nrms_user_encoder_table16_workspace_bytes": (_sz, [_i64, _i32, _i64]),
    "nrms_user_encoder_table16_fwd": (_i32, [_vp, _i64, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nrms_encoder_ln_stash_bytes": (_sz, [_i64, _i32]),
    "nrms_news_encoder_ln_fwd": (_i32, [_vp, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                        _sz, _f32, _u64, _u64, _i32, _vp]),
    "nrms_news_encoder_ln_bwd": (_i32, [_vp, _vp, _i64, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                        _vp, _vp, _vp, _vp, _sz, _f32, _u64, _u64, _i32, _vp]),
    "nrms_user_encoder_ln_fwd": (_i32, [_vp, _i64, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                        _sz, _i32, _vp]),
    "nrms_user_encoder_ln_bwd": (_i32, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                        _vp, _vp, _sz, _i32, _vp]),
    "nrms_mhsa_fwd": (_i32, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "nrms_mhsa_masked_fwd": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "nrms_mhsa_bwd_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "nrms_mhsa_bwd": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "nrms_mha_fwd_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "nrms_mha_fwd": (_i32, [_vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "nrms_mha_bwd_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32]),
    "nrms_mha_bwd": (_i32, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i32,
                            _vp]),
    "nrms_additive_fwd": (_i32, [_vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "nrms_additive_bwd_workspace_bytes": (_sz, [_i64, _i32, _i32]),
    "nrms_additive_bwd": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _i32, _vp]),
    "nrms_news_encoder_rows_fwd": (_i32, [_vp, _i64, _vp, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _vp, _f32, _u64, _u64, _i32, _vp]),
    "nrms_news_encoder_rows_bwd": (_i32, [_vp, _vp, _i64, _vp, _i64, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _sz, _f32, _u64, _u64, _i32, _vp]),
    "nrms_text_encoder_fwd": (_i32, [_vp, _i64, _vp, _i64, _i32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _vp, _sz, _f32, _u64, _u64, _i32, _vp]),
    "nrms_text_encoder_bwd": (_i32, [_vp, _vp, _i64, _vp, _i64, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _vp, _vp, _vp, _vp, _vp, _sz, _f32, _u64, _u64, _i32, _vp]),
    "nrms_element_encoder_table_bytes": (_sz, [_i64]),
    "nrms_element_encoder_fwd": (_i32, [_vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "nrms_element_encoder_bwd": (_i32, [_vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nrms_add_position_fwd": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "nrms_add_position_bwd_workspace_bytes": (_sz, [_i32]),
    "nrms_add_position_bwd": (_i32, [_vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    "nrms_copy_rows_strided": (_i32, [_vp, _i64, _vp, _i64, _i64, _i32, _vp]),
    "nrms_recommend_workspace_bytes": (_sz, []),
    "nrms_recommend_user": (_i32, [_vp, _i64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "nrms_topk_workspace_bytes": (_sz, [_i64, _i64, _i32, _i32, _i32]),
    "nrms_topk_news": (_i32, [_vp, _i64, _vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _sz, _i32, _vp]),
    "nrms_score_fwd": (_i32, [_vp, _vp, _i64, _i32, _i32, _vp, _vp]),
    "nrms_score_bwd": (_i32, [_vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "nrms_score_csr": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "nrms_pack_rows_f16": (_i32, [_vp, _i64, _vp, _vp]),
    "nrms_score_csr_f16": (_i32, [_vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "nrms_ce_loss_fwd_bwd": (_i32, [_vp, _i64, _i32, _f32, _vp, _vp, _vp]),
    "nrms_adam_step": (_i32, [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _f32, _i32, _i64, _f32, _vp]),
    "nrms_gather_rows": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "nrms_rank_metrics": (_i32, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "nrms_gemm_nt": (_i32, [_vp, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _i32, _i32, _i32, _vp]),
}

_lib = None


def load():
    """Load the shared library once; raise loudly if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the NRMS B200 CUDA library is not built. "
            "Run `python newsrecommendationsystem_b200/csrc/build.py` (nvcc, sm_100a). There is no CPU fallback.")
    import torch  # noqa: F401  (brings libcudart.so.12 into the process before dlopen)
    _prefer_large_page_segments(torch)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _prefer_large_page_segments(torch):
    """Workspaces (the projected q|k|v table above all: 141 MB gathered in random 2,160-byte rows) must sit on 2 MB
    pages.  Measured on B200: carved out of a plain cudaMalloc segment the same evaluate pass took 4.3 ms in the user
    stage instead of 3.2 ms whenever less than ~64 MB had been allocated before it (profiles/k1g_probe.py,
    PROBE_FLUSHBUF_MB sweep); segments mapped through the CUDA virtual-memory API -- torch's `expandable_segments` --
    are 3.2 ms in every order.  Only a default: an explicit PYTORCH_CUDA_ALLOC_CONF or NRMS_B200_KEEP_ALLOCATOR=1 wins."""
    if os.environ.get("PYTORCH_CUDA_ALLOC_CONF") or os.environ.get("NRMS_B200_KEEP_ALLOCATOR"):
        return
    try:
        if torch.cuda.is_available():
            setter = getattr(torch._C, "_accelerator_setAllocatorSettings", None) or torch.cuda.memory._set_allocator_settings
            setter("expandable_segments:True")
    except Exception:      # an allocator backend without the knob: keep its default
        pass


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().nrms_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libnrms_b200 {what} failed (code {rc}): {msg}")


def ptr(t):
    """Raw device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
