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


# ---- long sequences: the mask is recomputed in the backward -------------------------------------------------------
# The bitmask costs S^2 / 8 bytes per head (128 MiB at S 32768), held from the forward to the backward by the Functions
# above.  These take the PQ codes instead (S m 4 bytes per head), run the lookup in the forward and again in the backward:
# the lookup is deterministic, so the gradients are bit for bit those of the saved-mask Functions.
class SparseAttentionRecompute(autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, q_codes, k_codes, sparse_coeff: int, n_codewords, scale: float, clamp: float,
                reference_layout: bool = False):
        mask, extra0, _ = ext.lookup_mask(q_codes, k_codes, sparse_coeff, n_codewords=n_codewords)
        y, zsum = ext.sparse_attn_fwd(q, k, v, mask, extra0, scale, clamp, reference_layout)
        ctx.save_for_backward(q, k, v, y, zsum, q_codes, k_codes)
        ctx.sparse_coeff, ctx.n_codewords = sparse_coeff, n_codewords
        ctx.scale, ctx.clamp, ctx.reference_layout = scale, clamp, reference_layout
        return y

    @staticmethod
    def backward(ctx, grad_y):
        q, k, v, y, zsum, q_codes, k_codes = ctx.saved_tensors
        mask, extra0, _ = ext.lookup_mask(q_codes, k_codes, ctx.sparse_coeff, n_codewords=ctx.n_codewords)
        gq, gk, gv = ext.sparse_attn_bwd(q, k, v, y, grad_y.contiguous(), mask, extra0, zsum, ctx.scale, ctx.clamp,
                                         ctx.reference_layout)
        return gq, gk, gv, None, None, None, None, None, None, None


def sparse_attention_recompute(q, k, v, q_codes, k_codes, sparse_coeff: int, scale: float, clamp: float = 10.0,
                               reference_layout: bool = False, n_codewords=None):
    """sparse_attention on the pattern ext.lookup_mask(q_codes, k_codes, sparse_coeff, n_codewords=n_codewords) gives,
    without keeping the mask between forward and backward (codes int32 [B, S, m] or [N, S, H, m], like q)."""
    return SparseAttentionRecompute.apply(q, k, v, q_codes, k_codes, int(sparse_coeff), n_codewords, scale, clamp,
                                          reference_layout)


class SparseAttentionVarlenRecompute(autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, q_codes, k_codes, cu_seqlens, max_seqlen: int, sparse_coeff: int, n_codewords,
                scale: float, clamp: float, reference_layout: bool = False):
        T = q.size(-3)
        work = ext.varlen_worklist(cu_seqlens, T, max_seqlen)      # built once, reused by both lookups and the backward
        mask, extra0 = ext.lookup_mask_varlen(q_codes, k_codes, cu_seqlens, max_seqlen, sparse_coeff, work=work,
                                              n_codewords=n_codewords)
        y, zsum = ext.sparse_attn_varlen_fwd(q, k, v, mask, extra0, cu_seqlens, max_seqlen, scale, clamp, reference_layout,
                                             work=work)
        ctx.save_for_backward(q, k, v, y, zsum, q_codes, k_codes, cu_seqlens, work)
        ctx.max_seqlen, ctx.sparse_coeff, ctx.n_codewords = max_seqlen, sparse_coeff, n_codewords
        ctx.scale, ctx.clamp, ctx.reference_layout = scale, clamp, reference_layout
        return y

    @staticmethod
    def backward(ctx, grad_y):
        q, k, v, y, zsum, q_codes, k_codes, cu, work = ctx.saved_tensors
        mask, extra0 = ext.lookup_mask_varlen(q_codes, k_codes, cu, ctx.max_seqlen, ctx.sparse_coeff, work=work,
                                              n_codewords=ctx.n_codewords)
        gq, gk, gv = ext.sparse_attn_varlen_bwd(q, k, v, y, grad_y.contiguous(), mask, extra0, zsum, cu, ctx.max_seqlen,
                                                ctx.scale, ctx.clamp, ctx.reference_layout, work=work)
        return (gq, gk, gv) + (None,) * 9


def sparse_attention_varlen_recompute(q, k, v, q_codes, k_codes, cu_seqlens, max_seqlen: int, sparse_coeff: int,
                                      scale: float, clamp: float = 10.0, reference_layout: bool = False,
                                      n_codewords=None):
    """sparse_attention_varlen on the pattern of ext.lookup_mask_varlen, recomputed in the backward (as
    sparse_attention_recompute)."""
    return SparseAttentionVarlenRecompute.apply(q, k, v, q_codes, k_codes, cu_seqlens, int(max_seqlen), int(sparse_coeff),
                                                n_codewords, scale, clamp, reference_layout)
