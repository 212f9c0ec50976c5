"""Grouped-query attention: the C entry points and the Python layers reject malformed head counts before any CUDA call
(no GPU needed)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ("spt_lookup_mask_gqa_fwd", "spt_lookup_mask_varlen_gqa_fwd", "spt_sparse_attn_fwd_gqa",
               "spt_sparse_attn_bwd_gqa", "spt_sparse_attn_bwd_gqa_workspace_bytes", "spt_sparse_attn_varlen_fwd_gqa",
               "spt_sparse_attn_varlen_bwd_gqa", "spt_sparse_attn_varlen_bwd_gqa_workspace_bytes")


def _lib():
    import __graft_entry__
    __graft_entry__.build()
    lib = ctypes.CDLL(os.path.join(ROOT, "spt_proto_b200", "lib", "libspt_b200.so"))
    vp, i32, f32, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t
    lib.spt_last_error.restype = ctypes.c_char_p
    lib.spt_lookup_mask_gqa_fwd.argtypes = [vp] * 6 + [i32] * 7 + [vp]
    lib.spt_lookup_mask_varlen_gqa_fwd.argtypes = [vp] * 6 + [i32] * 8 + [vp]
    lib.spt_sparse_attn_fwd_gqa.argtypes = [vp] * 7 + [i32] * 5 + [f32, f32, i32, i32, vp]
    lib.spt_sparse_attn_bwd_gqa.argtypes = [vp] * 12 + [i32] * 5 + [f32, f32, i32, i32, vp]
    lib.spt_sparse_attn_varlen_fwd_gqa.argtypes = [vp] * 8 + [i32] * 6 + [f32, f32, i32, i32, vp]
    lib.spt_sparse_attn_varlen_bwd_gqa.argtypes = [vp] * 13 + [i32] * 6 + [f32, f32, i32, i32, vp]
    lib.spt_sparse_attn_bwd_gqa_workspace_bytes.restype = sz
    lib.spt_sparse_attn_bwd_gqa_workspace_bytes.argtypes = [i32] * 5
    lib.spt_sparse_attn_bwd_workspace_bytes.restype = sz
    lib.spt_sparse_attn_bwd_workspace_bytes.argtypes = [i32] * 2
    lib.spt_sparse_attn_varlen_bwd_gqa_workspace_bytes.restype = sz
    lib.spt_sparse_attn_varlen_bwd_gqa_workspace_bytes.argtypes = [i32] * 4
    lib.spt_sparse_attn_varlen_bwd_workspace_bytes.restype = sz
    lib.spt_sparse_attn_varlen_bwd_workspace_bytes.argtypes = [i32] * 2
    return lib


def test_header_declares_the_gqa_entry_points():
    text = open(os.path.join(ROOT, "include", "spt_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    declared = set(re.findall(r"\b(spt_[a-z0-9_]+)\s*\(", text))
    assert set(NEW_SYMBOLS) <= declared


@pytest.mark.parametrize("H,Hkv", [(4, 0), (4, -2), (4, 3), (8, 16)])
def test_entry_points_reject_bad_head_counts(H, Hkv):
    """Hkv < 1 and H % Hkv != 0: status 1 and a message naming Hkv, from every GQA entry point, before any CUDA call."""
    lib = _lib()
    buf = (ctypes.c_uint8 * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p).value
    p = (p + 15) // 16 * 16 if p % 16 else p            # 16-byte aligned (the alignment check would come first)
    bf16 = 1
    calls = [
        lambda: lib.spt_sparse_attn_fwd_gqa(*([p] * 7), 2 * H, 256, 64, H, Hkv, 0.1, 10.0, bf16, 0, None),
        lambda: lib.spt_sparse_attn_bwd_gqa(*([p] * 12), 2 * H, 256, 64, H, Hkv, 0.1, 10.0, bf16, 0, None),
        lambda: lib.spt_sparse_attn_varlen_fwd_gqa(*([p] * 8), 2, 512, 256, 64, H, Hkv, 0.1, 10.0, bf16, 0, None),
        lambda: lib.spt_sparse_attn_varlen_bwd_gqa(*([p] * 13), 2, 512, 256, 64, H, Hkv, 0.1, 10.0, bf16, 0, None),
        lambda: lib.spt_lookup_mask_gqa_fwd(*([p] * 6), 2 * H, 256, 8, 32, H, Hkv, 16, None),
        lambda: lib.spt_lookup_mask_varlen_gqa_fwd(*([p] * 6), 2, 512, 256, H, Hkv, 8, 8, 16, None),
    ]
    for call in calls:
        assert call() == 1
        got = lib.spt_last_error()
        assert b"Hkv=%d" % Hkv in got and (b">= 1" in got or b"multiple" in got), got


def test_workspace_sizes():
    """Multi-head sizes at Hkv = H; plus the dK / dV partials (2 * rows * d * 2 bytes) when Hkv < H."""
    lib = _lib()
    B, S, d, H = 64, 2048, 128, 32
    base = lib.spt_sparse_attn_bwd_workspace_bytes(B, S)
    assert lib.spt_sparse_attn_bwd_gqa_workspace_bytes(B, S, d, H, H) == base
    assert lib.spt_sparse_attn_bwd_gqa_workspace_bytes(B, S, d, H, 8) == base + 2 * B * S * d * 2
    T = 4096
    vbase = lib.spt_sparse_attn_varlen_bwd_workspace_bytes(T, H)
    assert lib.spt_sparse_attn_varlen_bwd_gqa_workspace_bytes(T, d, H, H) == vbase
    assert lib.spt_sparse_attn_varlen_bwd_gqa_workspace_bytes(T, d, H, 1) == vbase + 2 * H * T * d * 2


def test_ext_rejects_mismatched_shapes_before_any_cuda_call():
    _lib()
    from spt_proto_b200 import ext
    q = torch.zeros(1, 256, 8, 64, dtype=torch.bfloat16)
    k = torch.zeros(1, 256, 2, 64, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="k and v must have the same shape"):
        ext.sparse_attn_fwd(q, k, torch.zeros(1, 256, 4, 64, dtype=torch.bfloat16), None, None, 0.1)
    with pytest.raises(RuntimeError, match="H % Hkv == 0"):
        ext.sparse_attn_fwd(q, q[:, :, :3].contiguous(), q[:, :, :3].contiguous(), None, None, 0.1)
    with pytest.raises(RuntimeError, match="H % Hkv == 0"):        # head-major 3-D operands stay multi-head
        ext.sparse_attn_fwd(q[0], k[0], k[0], None, None, 0.1)
    with pytest.raises(RuntimeError, match="H % Hkv == 0"):        # packed: head axis 1 of [T, H, d]
        ext.sparse_attn_varlen_fwd(q[0], q[0, :, :5], q[0, :, :5], None, None, None, 256, 0.1)
    # well-formed GQA shapes pass the shape checks and stop at the device check
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ext.sparse_attn_fwd(q, k, k, None, None, 0.1)
    assert ext._kv_heads(q, k, 2, "t") == 2 and ext._kv_heads(q, q, None, "t") == 1


class _Meta:
    """Shape / dtype / device view of a tensor that pretends to live on the GPU (path choice without a device)."""

    def __init__(self, *shape, dtype=torch.bfloat16):
        self._t = torch.empty(shape, dtype=dtype, device="meta")
        self.is_cuda, self.dtype, self.shape = True, dtype, self._t.shape

    def size(self, *a):
        return self._t.size(*a)

    def dim(self):
        return self._t.dim()


@pytest.mark.parametrize("cls", ["SparseVanillaAttentionV2", "SparseRotaryAttentionV2"])
def test_layer_validation_and_path_choice(cls):
    from spt_proto_b200 import layers
    attn = getattr(layers, cls)(d_head=64, p_dropout=0.0, d_codeword=8, n_codewords=16)
    kv_group = attn._kv_group
    q = torch.zeros(2, 256, 32, 64)
    assert kv_group(q, q, q) == 1
    assert kv_group(q, q[:, :, :8], q[:, :, :8]) == 4
    assert kv_group(q, q[:, :, :1], q[:, :, :1]) == 32
    with pytest.raises(ValueError, match="k and v must have the same shape"):
        kv_group(q, q[:, :, :8], q[:, :, :4])
    with pytest.raises(ValueError, match="must be a multiple of the key / value head count Hkv = 5"):
        kv_group(q, q[:, :, :5], q[:, :, :5])
    with pytest.raises(ValueError, match="same N, S and"):
        kv_group(q, q[:, :128, :8], q[:, :128, :8])
    with pytest.raises(ValueError):
        attn(q, q[:, :, :5], q[:, :, :5])                         # forward validates before choosing a path
    with pytest.raises(ValueError):
        attn.forward_packed(q[:1], q[:1, :, :5], q[:1, :, :5], [0, 256])
    k, v = attn._repeat_kv(q[:, :, :8], q[:, :, :8] + 1, 4)
    assert k.shape == q.shape and torch.equal(k[:, :, 5], q[:, :, 1]) and torch.equal(v[:, :, 31], q[:, :, 7] + 1)
    # the fused envelope depends on q alone: GQA shapes take the fused path wherever multi-head ones do
    assert attn._fused_ok(_Meta(1, 2048, 32, 64))
    assert not attn._fused_ok(_Meta(1, 2048, 32, 96))
    assert attn._packed_fused_ok(_Meta(1, 4096, 32, 64), 2048)
    attn.use_fused = False
    assert not attn._fused_ok(_Meta(1, 2048, 32, 64)) and not attn._packed_fused_ok(_Meta(1, 4096, 32, 64), 2048)
