"""ctypes loader for libspt_b200.so.  There is NO fallback: if the CUDA library is missing the
import fails loudly (the product path never routes through torch-eager or the oracle)."""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libspt_b200.so")

SPT_OK = 0
SPT_F32 = 0
SPT_BF16 = 1
SPT_F16 = 2          # PQ encode / train, the fused attention and the routed FFN only (include/spt_b200.h)
SPT_ATTN_Y_TRANSPOSED = 1


class SptLibraryMissing(ImportError):
    pass


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise SptLibraryMissing(
            f"{LIB_PATH} not found. Build it with `python -m spt_proto_b200.build` "
            "(or __graft_entry__.build()). spt_proto_b200 has no CPU / eager fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    c = ctypes
    vp, i32, i64, f32, sz = c.c_void_p, c.c_int, c.c_int64, c.c_float, c.c_size_t
    sig = {
        "spt_abi_version": (c.c_int, []),
        "spt_last_error": (c.c_char_p, []),
        "spt_launch_count": (c.c_uint64, []),
        "spt_cdist_fwd": (i32, [vp, vp, vp, vp, i32, i64, i32, i32, i32, vp]),
        "spt_cdist_bwd_workspace_bytes": (sz, [i32, i64, i32, i32]),
        "spt_cdist_bwd": (i32, [vp, vp, vp, vp, vp, vp, i32, i64, i32, i32, vp]),
        "spt_pq_encode": (i32, [vp, vp, vp, i64, i32, i32, i32, i32, vp]),
        "spt_pq_encode_pair": (i32, [vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]),
        "spt_pq_train_blocks": (i32, [i64, i32]),
        "spt_pq_train_fwd": (i32, [vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]),
        "spt_pq_train_bwd": (i32, [vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]),
        "spt_lookup_workspace_bytes": (sz, [i32, i32, i32, i32]),
        "spt_lookup_fwd": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp]),
        "spt_sddmm_fwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i64, f32, f32, i32, vp]),
        "spt_clamp_scale_bwd": (i32, [vp, vp, vp, i64, f32, f32, vp]),
        "spt_spmm_fwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i64, i32, i32, vp]),
        "spt_spmm_t_fwd": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i64, i32, i32, vp]),
        "spt_csr_tiles_supported": (i32, [i32, i64]),
        "spt_csr_tiles_ptr_len": (i64, [i32]),
        "spt_csr_tiles": (i32, [vp, vp, vp, vp, i32, i32, i64, vp]),
        "spt_spmm_t_tiles_fwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i64, i32, i32, vp]),
        "spt_spmm_tiles_fwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i64, i32, i32, i32, vp]),
        "spt_sddmm_tiles_fwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i64, f32, f32, i32, vp]),
        "spt_csr2csc_workspace_bytes": (sz, [i32, i32, i64]),
        "spt_csr2csc": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i64, vp]),
        "spt_softmax_fwd": (i32, [vp, vp, vp, vp, i32, i32, i64, vp]),
        "spt_softmax_bwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i64, vp]),
        "spt_softmax_bwd_ex": (i32, [vp, vp, vp, vp, vp, i32, i32, i64, i32, vp]),
        "spt_lookup_mask_fwd": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
        "spt_lookup_mask_fwd_ex": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]),
        "spt_sparse_attn_fwd": (i32, [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, f32, i32, vp]),
        "spt_sparse_attn_fwd_ex": (i32, [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, f32, i32, i32, vp]),
        "spt_sparse_attn_bwd_ex": (i32, [vp] * 12 + [i32, i32, i32, i32, f32, f32, i32, i32, vp]),
        "spt_sparse_attn_bwd_workspace_bytes": (sz, [i32, i32]),
        "spt_debug_attn_prof": (i32, [vp, i32]),
        "spt_sparse_attn_bwd": (i32, [vp] * 12 + [i32, i32, i32, i32, f32, f32, i32, vp]),
    }
    ll = c.c_longlong
    sig["spt_grouped_gemm_bf16"] = (i32, [i32, vp, ll, ll, ll, i32, vp, ll, ll, ll, i32, vp, i32, vp, i32, i32, i32, i32,
                                          i32, i32, i32, i32, ll, ll, vp, ll, i32, vp, i32, vp, i32, vp, ll, vp])
    sig["spt_grouped_gemm"] = (i32, sig["spt_grouped_gemm_bf16"][1][:-1] + [i32, vp])
    sig["spt_rmsnorm_bwd_blocks"] = (i32, [i64])
    sig["spt_rmsnorm_fwd_bf16"] = (i32, [vp, vp, vp, vp, i64, i32, f32, vp])
    sig["spt_rmsnorm_bwd_bf16"] = (i32, [vp, vp, vp, vp, vp, vp, i64, i32, vp])
    sig["spt_rope_bf16"] = (i32, [vp, vp, vp, vp, i64, i32, i32, i32, i32, vp])
    sig["spt_grouped_gemm_plan"] = (i32, [vp, i32, i32, vp, i32])
    sig["spt_scale_add_fwd"] = (i32, [vp, vp, i32, vp, i32, vp, i32, i64, i32, vp])
    sig["spt_scale_add_bwd"] = (i32, [vp, vp, i32, vp, i32, vp, vp, i64, i32, vp])
    sig["spt_lora_glu_fwd"] = (i32, [vp] * 6 + [i64, i32, vp])
    sig["spt_silu_mul_fwd"] = (i32, [vp] * 3 + [i64, vp])
    sig["spt_silu_mul_bwd"] = (i32, [vp] * 5 + [i64, vp])
    sig["spt_lora_glu_bwd"] = (i32, [vp] * 11 + [i64, i32, vp])
    sig["spt_lora_glu_fwd_ex"] = (i32, [vp] * 6 + [i64, i32, i32, vp])
    sig["spt_lora_glu_bwd_ex"] = (i32, [vp] * 11 + [i64, i32, i32, vp])
    sig["spt_silu_mul_fwd_ex"] = (i32, [vp] * 3 + [i64, i32, vp])
    sig["spt_silu_mul_bwd_ex"] = (i32, [vp] * 5 + [i64, i32, vp])
    sig["spt_route_bucket_workspace_bytes"] = (sz, [i64, i32])
    sig["spt_route_bucket"] = (i32, [vp] * 8 + [i64, i32, i32, i64, vp])
    sig["spt_gather_rows_bf16"] = (i32, [vp, vp, vp, i64, i32, vp])
    sig["spt_ffn_combine"] = (i32, [vp, vp, vp, vp, i64, i32, i32, i32, i32, vp])
    sig["spt_group_colsum_workspace_bytes"] = (sz, [i32, i32])
    sig["spt_group_colsum_bf16"] = (i32, [vp, vp, vp, vp, i32, i32, vp])
    sig["spt_group_colsum"] = (i32, [vp, vp, vp, vp, i32, i32, i32, vp])
    sig["spt_row_coeff_bwd"] = (i32, [vp, vp, vp, vp, i64, i64, i32, vp])
    sig["spt_softmax_clamp_bwd"] = (i32, [vp] * 6 + [i32, i32, i64, f32, f32, i32, vp])
    sig["spt_swap_dims12"] = (i32, [vp, vp, i64, i64, i64, i64, vp])
    sig["spt_transpose_last2"] = (i32, [vp, vp, i64, i32, i32, i32, vp])
    # packed variable-length sequences
    sig["spt_varlen_worklist_bytes"] = (sz, [i32, i32])
    sig["spt_varlen_worklist"] = (i32, [vp, i32, i32, i32, vp, vp])
    sig["spt_lookup_mask_varlen_workspace_bytes"] = (sz, [i32, i32, i32, i32])
    sig["spt_lookup_mask_varlen_max_seqlen"] = (i32, [i32])
    sig["spt_lookup_mask_varlen_fwd"] = (i32, [vp] * 6 + [i32] * 6 + [vp])
    sig["spt_lookup_mask_varlen_fwd_ex"] = (i32, [vp] * 6 + [i32] * 7 + [vp])
    sig["spt_sparse_attn_varlen_fwd"] = (i32, [vp] * 8 + [i32, i32, i32, i32, i32, f32, f32, i32, i32, vp])
    sig["spt_sparse_attn_varlen_bwd_workspace_bytes"] = (sz, [i32, i32])
    sig["spt_sparse_attn_varlen_bwd"] = (i32, [vp] * 13 + [i32, i32, i32, i32, i32, f32, f32, i32, i32, vp])
    # grouped-query attention: H query heads, Hkv key / value heads
    sig["spt_lookup_mask_gqa_fwd"] = (i32, [vp] * 6 + [i32] * 7 + [vp])
    sig["spt_lookup_mask_varlen_gqa_fwd"] = (i32, [vp] * 6 + [i32] * 8 + [vp])
    sig["spt_sparse_attn_fwd_gqa"] = (i32, [vp] * 7 + [i32, i32, i32, i32, i32, f32, f32, i32, i32, vp])
    sig["spt_sparse_attn_bwd_gqa_workspace_bytes"] = (sz, [i32] * 5)
    sig["spt_sparse_attn_bwd_gqa"] = (i32, [vp] * 12 + [i32, i32, i32, i32, i32, f32, f32, i32, i32, vp])
    sig["spt_sparse_attn_varlen_fwd_gqa"] = (i32, [vp] * 8 + [i32] * 6 + [f32, f32, i32, i32, vp])
    sig["spt_sparse_attn_varlen_bwd_gqa_workspace_bytes"] = (sz, [i32] * 4)
    sig["spt_sparse_attn_varlen_bwd_gqa"] = (i32, [vp] * 13 + [i32] * 6 + [f32, f32, i32, i32, vp])
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError => header/library mismatch, fail loudly
        fn.restype = res
        fn.argtypes = args
    # optional symbols added by later ABI revisions are bound lazily in their own modules
    return lib


lib = _load()


def check(rc: int) -> None:
    """Map an spt_status to the exception type the reference raises from TORCH_CHECK (RuntimeError)."""
    if rc != SPT_OK:
        raise RuntimeError(f"spt_b200: {lib.spt_last_error().decode()} (status {rc})")
