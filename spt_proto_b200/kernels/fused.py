"""Fused sparse attention autograd Function: the fast path of the V2 layers (bf16 or fp16, d_head 64,
80 or 128).
Equivalent to  spmm(softmax(clamp_(scale * sddmm(q, k), -10, 10)), v)  on the lookup's pattern
(reference layers/sparse/attention.py:122-141 + the three backward passes), computed as masked dense
tiles on the tensor cores from the lookup's bitmask output."""
from torch import autograd

from .. import ext


class SparseAttention(autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, mask, extra0, scale: float, clamp: float, reference_layout: bool = False):
        y, zsum = ext.sparse_attn_fwd(q, k, v, mask, extra0, scale, clamp, reference_layout)
        ctx.save_for_backward(q, k, v, y, mask, extra0, zsum)
        ctx.scale, ctx.clamp, ctx.reference_layout = scale, clamp, reference_layout
        return y

    @staticmethod
    def backward(ctx, grad_y):
        q, k, v, y, mask, extra0, zsum = ctx.saved_tensors
        gq, gk, gv = ext.sparse_attn_bwd(q, k, v, y, grad_y.contiguous(), mask, extra0, zsum, ctx.scale, ctx.clamp,
                                         ctx.reference_layout)
        return gq, gk, gv, None, None, None, None, None


def sparse_attention(q, k, v, mask, extra0, scale: float, clamp: float = 10.0, reference_layout: bool = False):
    """q, k, v [B, S, d] or [N, S, H, d], all bf16 or all fp16; (mask, extra0) from ext.lookup_mask -> y, same shape
    and dtype.  fp16 needs 0 <= clamp <= 10.
    reference_layout=True: y is returned in the shipped reference layer's output layout (the memory of y^T
    [N*H, d, S] viewed with q's shape, attention.py:139-142), written by the kernel itself."""
    return SparseAttention.apply(q, k, v, mask, extra0, scale, clamp, reference_layout)


class SparseAttentionVarlen(autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, mask, extra0, cu_seqlens, max_seqlen: int, scale: float, clamp: float,
                reference_layout: bool = False):
        T = q.size(-3)
        work = ext.varlen_worklist(cu_seqlens, T, max_seqlen)      # built once, reused by the backward
        y, zsum = ext.sparse_attn_varlen_fwd(q, k, v, mask, extra0, cu_seqlens, max_seqlen, scale, clamp, reference_layout,
                                             work=work)
        ctx.save_for_backward(q, k, v, y, mask, extra0, zsum, cu_seqlens, work)
        ctx.max_seqlen, ctx.scale, ctx.clamp, ctx.reference_layout = max_seqlen, scale, clamp, reference_layout
        return y

    @staticmethod
    def backward(ctx, grad_y):
        q, k, v, y, mask, extra0, zsum, cu, work = ctx.saved_tensors
        gq, gk, gv = ext.sparse_attn_varlen_bwd(q, k, v, y, grad_y.contiguous(), mask, extra0, zsum, cu, ctx.max_seqlen,
                                                ctx.scale, ctx.clamp, ctx.reference_layout, work=work)
        return gq, gk, gv, None, None, None, None, None, None, None


def sparse_attention_varlen(q, k, v, mask, extra0, cu_seqlens, max_seqlen: int, scale: float, clamp: float = 10.0,
                            reference_layout: bool = False):
    """Packed variable-length sequences: q, k, v [T, H, d] or [1, T, H, d], cu_seqlens int32 [n + 1] on the device,
    (mask, extra0) from ext.lookup_mask_varlen -> y like q.  Sequence i gets what sparse_attention gives for it alone;
    reference_layout=True: its y memory is its own y_i^T [H, d, S_i] at token offset cu[i]."""
    return SparseAttentionVarlen.apply(q, k, v, mask, extra0, cu_seqlens, int(max_seqlen), scale, clamp, reference_layout)
