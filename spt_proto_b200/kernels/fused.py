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
