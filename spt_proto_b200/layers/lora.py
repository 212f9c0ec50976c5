"""LoRA layers (reference naive_gpt/layers/tuning/lora.py, lora_ffn.py).

LoRALinear / LoRAEmbedding: frozen base + rank-r update with nn.Embedding-shaped factors
(`lora.left.weight [in, r]`, `lora.right.weight [out, r]`, right zero-initialised) — thin GEMMs, plain
torch.  LoRARoutedFFN / LoRARoutedLLaMaFFN (lora_ffn.py:6-115, 118-225) are what SparseLoRAHandler
installs for fine-tuning: the routed FFN with frozen base weights, a per-(token, block) scalar
coeff = 2 * prob that carries the router's gradient, and the LoRA paths:

    u  = coeff * (x W1_i^T + b1_i) + (x L1) R1_i^T          h = act(u)
    y += coeff * (h W2_i) + (h L2_i) R2^T                   y += b2

Here every product with a base weight block or a blocked LoRA factor is a grouped GEMM on the tcgen05
tensor cores over the bucketed tokens; the rank-r dense factors (x L1, . R2^T) are torch GEMMs and the
elementwise glue (coeff * base + lora, the SiLU gate) runs in the fused kernels of csrc/lora_fuse.cu
(autograd Functions in kernels/ffn.py), so autograd yields exactly the reference's gradients (router
via coeff, LoRA factors; no gradient for the frozen base)."""
from __future__ import annotations

import torch
from torch import nn

from .. import ext
from ..kernels import ffn as F
from .basic import Feedforward, LLaMaFeedforward
from .routed_ffn import RoutedFFN, RoutedLLaMaFFN, _route


class LoRABase(nn.Module):
    def __init__(self, d_lora: int, in_features: int, out_features: int, device=None, dtype=None):
        super().__init__()
        self.left = nn.Embedding(in_features, embedding_dim=d_lora, device=device, dtype=dtype)
        self.right = nn.Embedding(out_features, embedding_dim=d_lora, device=device, dtype=dtype)
        self.scaling = 1.0 / d_lora          # kept for parity with the reference; unused there too
        nn.init.zeros_(self.right.weight)


class LoRALinear(nn.Linear):
    def __init__(self, d_lora: int, in_features: int, out_features: int, bias: bool = True, *args, **kwargs):
        super().__init__(in_features=in_features, out_features=out_features, bias=bias, *args, **kwargs)
        for p in self.parameters():
            p.requires_grad = False
        self.lora = LoRABase(d_lora=d_lora, in_features=in_features, out_features=out_features)

    @staticmethod
    def from_pretrained(d_lora: int, source: nn.Linear):
        model = LoRALinear(d_lora=d_lora, in_features=source.in_features, out_features=source.out_features,
                           bias=source.bias is not None)
        result = model.load_state_dict(source.state_dict(), strict=False)
        if len(result.missing_keys) != 2:
            raise RuntimeError
        return model

    def forward(self, x):
        y = nn.functional.linear(x, self.weight, self.bias)
        # y + (x L) R^T with the addition in the second product's epilogue (one pass less over y than a separate add)
        # (in place on the fresh product: an out-of-place addmm would first copy y)
        t = x.reshape(-1, x.size(-1)) @ self.lora.left.weight
        y.view(-1, y.size(-1)).addmm_(t, self.lora.right.weight.t())
        return y


class LoRAEmbedding(nn.Embedding):
    def __init__(self, d_lora: int, num_embeddings: int, embedding_dim: int, *args, **kwargs):
        super().__init__(num_embeddings=num_embeddings, embedding_dim=embedding_dim, *args, **kwargs)
        for p in self.parameters():
            p.requires_grad = False
        self.lora = LoRABase(d_lora=d_lora, in_features=num_embeddings, out_features=embedding_dim)

    @staticmethod
    def from_pretrained(d_lora: int, source: nn.Embedding):
        model = LoRAEmbedding(d_lora=d_lora, num_embeddings=source.num_embeddings, embedding_dim=source.embedding_dim)
        result = model.load_state_dict(source.state_dict(), strict=False)
        if len(result.missing_keys) != 2:
            raise RuntimeError
        return model

    def forward(self, x):
        return nn.functional.embedding(x, self.weight) + self.lora.left(x) @ self.lora.right.weight.t()


class _RowCoeff(torch.autograd.Function):
    """coeff[r] = 2 * prob[token(r), block(r)] for real bucket rows, 0 for padding — differentiable in prob (this is how
    the router is trained, lora_ffn.py:92,206).  route_bucket already gathered prob[token, block] per row (row_prob), so
    the forward is one multiply; the backward writes 2 * grad to the row's (token, block) cell with plain stores (every
    pair owns at most one row) instead of torch's index chain and sort-based index_put backward (~25 small kernels)."""

    @staticmethod
    def forward(ctx, prob, bucket):
        ctx.bucket, ctx.p_dtype = bucket, prob.dtype
        return bucket.row_prob * 2.0

    @staticmethod
    def backward(ctx, grad):
        return ext.row_coeff_bwd(grad.float().contiguous(), ctx.bucket).to(ctx.p_dtype), None


def _row_coeff(prob: torch.Tensor, bucket) -> torch.Tensor:
    """prob [T, nb] must hold the values route_bucket() bucketed (its fp32 copy): coeff comes from bucket.row_prob."""
    return _RowCoeff.apply(prob, bucket)


class _MmF32(torch.autograd.Function):
    """16-bit x 16-bit -> fp32 thin matmul, both operands of one type (torch.mm(out_dtype=fp32) has no autograd
    formula)."""

    @staticmethod
    def forward(ctx, a, b):
        ctx.save_for_backward(a, b)
        return torch.mm(a, b, out_dtype=torch.float32)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        g16 = g.to(a.dtype)
        da = torch.mm(g16, b.t()) if ctx.needs_input_grad[0] else None
        db = torch.mm(a.t(), g16, out_dtype=torch.float32).to(b.dtype) if ctx.needs_input_grad[1] else None
        return da, db


def _down_proj_split(xp: torch.Tensor, left: torch.Tensor) -> torch.Tensor:
    """t = xp @ left (rank-r, fp32 accumulate) returned as [hi | lo] halves in xp's 16-bit type, hi + lo ~ t
    to 16 mantissa bits in bf16 (about 22 in fp16).  Fed to the grouped GEMM against [R | R], this keeps the
    LoRA pre-activation at fp32 quality: a single bf16 rounding of t flips ReLU gates when the LoRA term
    dominates (measured: 3 % gradient error vs 0.3 %).  Autograd through hi/lo is exact (d(hi + lo)/dt = 1)."""
    t = _MmF32.apply(xp, left.to(xp.dtype))
    hi = t.to(xp.dtype)
    lo = (t - hi.float()).to(xp.dtype)
    return torch.cat([hi, lo], dim=1)


def _twice(w: torch.Tensor) -> torch.Tensor:
    return torch.cat([w, w], dim=1)


def _pad8(w: torch.Tensor) -> torch.Tensor:
    """Zero-pad the rank dimension of a LoRA factor [*, r] to a multiple of 8 (TMA needs 16-byte rows)."""
    r = w.size(1)
    return w if r % 8 == 0 else nn.functional.pad(w, (0, (-r) % 8))


class LoRARoutedFFN(RoutedFFN):
    def __init__(self, d_lora: int, block_size: int, d_model: int, d_feedforward: int, activation: nn.Module):
        super().__init__(block_size=block_size, d_model=d_model, d_feedforward=d_feedforward, activation=activation,
                         p_dropout=0.0)
        self.fc1 = LoRALinear(d_lora=d_lora, in_features=d_model, out_features=d_feedforward)
        self.fc2 = LoRALinear(d_lora=d_lora, in_features=d_feedforward, out_features=d_model)

    @staticmethod
    def from_pretrained(d_lora: int, block_size: int, source: Feedforward):
        assert isinstance(source, Feedforward)
        model = LoRARoutedFFN(d_lora=d_lora, block_size=block_size, d_model=source.d_model,
                              d_feedforward=source.d_feedforward, activation=source.activation)
        result = model.load_state_dict(source.state_dict(), strict=False)
        if len(result.missing_keys) != 2:
            raise RuntimeError
        return model

    @property
    def k_active(self) -> int:
        return self.n_blocks // 2

    def forward(self, x: torch.Tensor):
        if not x.is_cuda:
            raise RuntimeError("LoRARoutedFFN: spt_proto_b200 has no CPU path (x must be a CUDA tensor)")
        x_size, bs = x.size(), self.block_size
        x2 = x.reshape(-1, self.d_model)
        prob, bucket = _route(self.router, x2, self.k_active)
        coeff = _row_coeff(prob.float(), bucket)                               # [R] fp32
        cdt = F.compute_dtype(x)                                                # bf16, or fp16 for fp16 x
        xp = F.gather(x2.to(cdt).contiguous(), bucket)                          # [R, d]
        f32 = torch.float32   # pre-activations stay fp32 so that activation gates are decided as in the reference
        base = F.blocked_linear_rows(xp, self.fc1.weight, self.fc1.bias, bucket, bs, out_dtype=f32)   # x W1_i^T + b1_i
        t1 = _down_proj_split(xp, _pad8(self.fc1.lora.left.weight))             # [R, 2r] = [hi | lo]
        lora = F.blocked_linear_rows(t1, _twice(_pad8(self.fc1.lora.right.weight)), None, bucket, bs,
                                     out_dtype=f32)                             # (x L1) R1_i^T
        h = self.activation(F.scale_add(coeff, base, lora, f32)).to(cdt)
        y_base = F.blocked_linear_cols(h, self.fc2.weight, bucket, bs)          # h W2_i
        t2 = F.blocked_linear_cols_t(h, _pad8(self.fc2.lora.left.weight), bucket, bs)   # h L2_i   [R, r]
        y_lora = t2 @ _pad8(self.fc2.lora.right.weight).to(cdt).t()             # (h L2_i) R2^T
        yp = F.scale_add(coeff, y_base, y_lora, cdt)
        y = F.combine(yp, bucket, self.fc2.bias, x.dtype)
        return y.view(x_size)


class LoRARoutedLLaMaFFN(RoutedLLaMaFFN):
    def __init__(self, d_lora: int, block_size: int, d_model: int, d_feedforward: int, activation: nn.Module):
        super().__init__(d_model, d_feedforward, block_size=block_size, activation=activation)
        self.gate = LoRALinear(d_lora=d_lora, in_features=d_model, out_features=d_feedforward, bias=False)
        self.side = LoRALinear(d_lora=d_lora, in_features=d_model, out_features=d_feedforward, bias=False)
        self.down = LoRALinear(d_lora=d_lora, in_features=d_feedforward, out_features=d_model, bias=False)

    @staticmethod
    def from_pretrained(d_lora: int, block_size: int, source: LLaMaFeedforward):
        assert isinstance(source, LLaMaFeedforward)
        model = LoRARoutedLLaMaFFN(d_lora=d_lora, block_size=block_size, d_model=source.d_model,
                                   d_feedforward=source.d_feedforward, activation=source.activation)
        result = model.load_state_dict(source.state_dict(), strict=False)
        if len(result.missing_keys) != 2:
            raise RuntimeError
        return model

    @property
    def k_active(self) -> int:
        return self.n_blocks // 2            # the LoRA variant activates half (lora_ffn.py:172)

    def _proj(self, lin: LoRALinear, xp, bucket):
        """-> (x W_i^T, (x L) R_i^T), both fp32 [R, bs]; the caller forms coeff * base + lora."""
        base = F.blocked_linear_rows(xp, lin.weight, None, bucket, self.block_size, out_dtype=torch.float32)
        lora = F.blocked_linear_rows(_down_proj_split(xp, _pad8(lin.lora.left.weight)),
                                     _twice(_pad8(lin.lora.right.weight)), None, bucket, self.block_size,
                                     out_dtype=torch.float32)
        return base, lora

    def forward(self, x: torch.Tensor):
        if not x.is_cuda:
            raise RuntimeError("LoRARoutedLLaMaFFN: spt_proto_b200 has no CPU path (x must be a CUDA tensor)")
        x_size, bs = x.size(), self.block_size
        x2 = x.reshape(-1, self.d_model)
        prob, bucket = _route(self.router, x2, self.k_active)
        coeff = _row_coeff(prob.float(), bucket)
        cdt = F.compute_dtype(x)
        xp = F.gather(x2.to(cdt).contiguous(), bucket)
        bg, lg = self._proj(self.gate, xp, bucket)
        bsd, lsd = self._proj(self.side, xp, bucket)
        if isinstance(self.activation, nn.SiLU):       # the LLaMA case: one fused kernel per direction
            h = F.lora_glu(coeff, bg, lg, bsd, lsd, cdt)
        else:
            h = (self.activation(F.scale_add(coeff, bg, lg, torch.float32))
                 * F.scale_add(coeff, bsd, lsd, torch.float32)).to(cdt)
        y_base = F.blocked_linear_cols(h, self.down.weight, bucket, bs)
        t2 = F.blocked_linear_cols_t(h, _pad8(self.down.lora.left.weight), bucket, bs)
        yp = F.scale_add(coeff, y_base, t2 @ _pad8(self.down.lora.right.weight).to(cdt).t(), cdt)
        y = F.combine(yp, bucket, None, x.dtype)
        return y.view(x_size)
