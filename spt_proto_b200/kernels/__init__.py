"""torch.autograd Functions of the hot path — same names and call signatures as the reference's
`naive_gpt.kernels` (naive_gpt/kernels/__init__.py:1-14)."""
from .cdist import cdist
from .lookup import lookup
from .softmax import softmax
from .sddmm import sddmm, sddmm_scaled, sddmm_softmax
from .spmm import spmm
from .fused import (sparse_attention, sparse_attention_recompute, sparse_attention_varlen,
                    sparse_attention_varlen_recompute)

__all__ = ["cdist", "lookup", "softmax", "sddmm", "sddmm_scaled", "sddmm_softmax", "spmm", "sparse_attention", "sparse_attention_varlen",
           "sparse_attention_recompute", "sparse_attention_varlen_recompute"]
