"""Dense building blocks the sparse layers derive from.  These mirror the *interface* of the
reference's naive_gpt/layers/basic/{attention,position,feedforward,quantizer}.py (constructor
arguments, attribute / parameter names — so reference checkpoints load — and forward contracts);
they are plain PyTorch and out of the hot path except for PQ 'encode', which is one fused kernel."""
from __future__ import annotations

import torch
from torch import nn

from .. import ext, kernels
from ..kernels import norm_rope


class RotaryEmbedding(nn.Module):
    """RoPE with cached cos/sin tables (reference basic/position.py:5-48).  x: [N, S, H, E]."""

    def __init__(self, n_embeddings: int, d_model: int, base: float = 10000.0):
        super().__init__()
        if d_model % 2:
            raise ValueError("d_model must be even")
        self.base, self.d_model = base, d_model
        cos, sin = self._angles(n_embeddings)
        self.register_buffer("cos_cached", cos)
        self.register_buffer("sin_cached", sin)
        # rows n_embeddings .. of longer tables, per (device, dtype): not buffers, so state_dict keeps the reference's
        # keys and shapes and reference checkpoints load unchanged
        self._beyond = {}

    def _angles(self, n: int):
        inv_freq = self.base ** (-torch.arange(0, self.d_model, 2) / self.d_model)
        angles = torch.outer(torch.arange(n), inv_freq).repeat(1, 2)   # [S, E]
        return angles.cos(), angles.sin()

    def tables(self, n: int):
        """(cos, sin) [n', E] with n' >= n rows: the registered buffers, followed past their length by rows of the same
        expression (what RotaryEmbedding(n_embeddings=n) holds there)."""
        L = self.cos_cached.size(0)
        if n <= L:
            return self.cos_cached, self.sin_cached
        key = (self.cos_cached.device, self.cos_cached.dtype)
        hit = self._beyond.get(key)
        if hit is None or hit[0].size(0) < n - L:
            cos, sin = self._angles(n)
            hit = tuple(t[L:].to(device=key[0], dtype=key[1]) for t in (cos, sin))
            self._beyond[key] = hit
        return torch.cat([self.cos_cached, hit[0][: n - L]]), torch.cat([self.sin_cached, hit[1][: n - L]])

    @staticmethod
    def rotate_half(x: torch.Tensor) -> torch.Tensor:
        lo, hi = x.chunk(2, dim=-1)
        return torch.cat((-hi, lo), dim=-1)

    fused = True    # one CUDA kernel per direction for bf16 inputs on the GPU (same roundings as the expression below)

    def forward(self, x: torch.Tensor, ids: torch.Tensor, n_positions=None) -> torch.Tensor:
        """n_positions: ids are < n_positions, which may exceed the registered tables (see tables)."""
        assert x.dim() == 4 and ids.dim() == 1
        cos_t, sin_t = self.tables(n_positions) if n_positions is not None else (self.cos_cached, self.sin_cached)
        cos, sin = cos_t[ids], sin_t[ids]
        if self.fused and ids.numel() == x.size(1) and ext.rope_supported(x, cos):
            return norm_rope.rope(x, cos.contiguous(), sin.contiguous())
        cos = cos.view(1, -1, 1, x.size(-1))
        sin = sin.view(1, -1, 1, x.size(-1))
        return x * cos + self.rotate_half(x) * sin


class VanillaAttention(nn.Module):
    """Dense softmax attention on [N, S, H, E] tensors (reference basic/attention.py:6-57).
    Sub-classes override _get_attn / _apply_attn."""

    def __init__(self, d_head: int, p_dropout: float):
        super().__init__()
        self.d_head = d_head
        self.p_dropout = p_dropout
        self.scaling = float(d_head) ** -0.5
        self.dropout = nn.Dropout(p_dropout)

    def _get_attn(self, q, k, attn_mask):
        scores = torch.einsum("niae,njae->naij", q, k)
        if attn_mask is not None:
            scores = scores + attn_mask
        return self.dropout(torch.softmax(self.scaling * scores, dim=-1))

    def _apply_attn(self, attn, v):
        return torch.einsum("naij,njae->niae", attn, v).contiguous()

    def forward(self, q, k, v, attn_mask=None):
        assert q.dim() == 4 and k.dim() == 4 and v.dim() == 4
        assert q.size(0) == k.size(0) == v.size(0)
        return self._apply_attn(self._get_attn(q, k, attn_mask), v)


class RotaryAttention(VanillaAttention):
    """VanillaAttention with RoPE applied to q and k (reference basic/attention.py:60-92)."""

    def __init__(self, d_head: int, p_dropout: float, max_length: int = 2048):
        super().__init__(d_head=d_head, p_dropout=p_dropout)
        self.max_length = max_length
        self.embedding = RotaryEmbedding(n_embeddings=max_length, d_model=d_head)
        self.register_buffer("cached_ids", torch.arange(max_length))

    def _rotate(self, x):
        S = x.size(1)
        if S <= self.cached_ids.numel():
            return self.embedding(x, ids=self.cached_ids[:S])
        # positions >= max_length: the embedding's tables extended by the same expression
        return self.embedding(x, ids=torch.arange(S, device=self.cached_ids.device), n_positions=S)

    def _get_attn(self, q, k, attn_mask):
        return VanillaAttention._get_attn(self, self._rotate(q), self._rotate(k), attn_mask)


class Feedforward(nn.Module):
    """fc2(act(dropout(fc1(x)))) (reference basic/feedforward.py:5-34)."""

    def __init__(self, d_model: int, d_feedforward: int, p_dropout: float, activation: nn.Module):
        super().__init__()
        self.d_model, self.d_feedforward = d_model, d_feedforward
        self.p_dropout = p_dropout
        self.fc1 = nn.Linear(d_model, d_feedforward)
        self.fc2 = nn.Linear(d_feedforward, d_model)
        self.dropout = nn.Dropout(p_dropout)
        self.activation = activation

    def forward(self, x):
        return self.fc2(self.activation(self.dropout(self.fc1(x))))


class LLaMaFeedforward(nn.Module):
    """down(act(gate(x)) * side(x)) (reference basic/feedforward.py:37-62)."""

    def __init__(self, d_model: int, d_feedforward: int, activation: nn.Module):
        super().__init__()
        self.d_model, self.d_feedforward = d_model, d_feedforward
        self.gate = nn.Linear(d_model, d_feedforward, bias=False)
        self.side = nn.Linear(d_model, d_feedforward, bias=False)
        self.down = nn.Linear(d_feedforward, d_model, bias=False)
        self.activation = activation

    def forward(self, x):
        return self.down(self.activation(self.gate(x)) * self.side(x))


class LlamaRMSNorm(nn.Module):
    """x / rms(x) * weight with the statistics in fp32 (reference basic/utils.py:22-38)."""

    def __init__(self, hidden_size: int, eps: float = 1e-6):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(hidden_size))
        self.variance_epsilon = eps

    fused = True    # one CUDA kernel per direction for bf16 input and weight on the GPU

    def forward(self, x):
        if self.fused and ext.rmsnorm_supported(x, self.weight):
            return norm_rope.rmsnorm(x, self.weight, self.variance_epsilon)
        inv_rms = torch.rsqrt(x.float().pow(2).mean(-1, keepdim=True) + self.variance_epsilon)
        y = x * inv_rms
        if self.weight.dtype in (torch.float16, torch.bfloat16):
            y = y.to(self.weight.dtype)
        return self.weight * y


class MultiheadAttention(nn.Module):
    """q/k/v/o projections around an attention function on [N, S, H, E] (reference basic/transformer.py:6-50).
    Attribute names (`linear_q` ... `linear_o`, `attn_fn`) are the reference's: they are checkpoint keys and the
    paths the module upgrader rewrites."""

    def __init__(self, d_model: int, n_heads: int, attention_fn: nn.Module, bias: bool):
        super().__init__()
        self.d_model, self.n_heads = d_model, n_heads
        self.attn_fn = attention_fn
        self.linear_q, self.linear_k, self.linear_v, self.linear_o = (
            nn.Linear(d_model, d_model, bias=bias) for _ in range(4))

    def forward(self, q, k, v, attn_mask=None):
        assert q.size(0) == k.size(0) == v.size(0)
        split = lambda t: t.view(t.size(0), t.size(1), self.n_heads, -1)
        y = self.attn_fn(split(self.linear_q(q)), split(self.linear_k(k)), split(self.linear_v(v)), attn_mask=attn_mask)
        return self.linear_o(y.reshape(y.size(0), y.size(1), -1))


class TransformerBlock(nn.Module):
    """Pre- or post-norm block: attention + feed-forward with residuals (reference basic/transformer.py:53-97)."""

    def __init__(self, d_model: int, n_heads: int, layernorm_fn: nn.Module, attention_fn: nn.Module,
                 feedforward_fn: nn.Module, attention_bias: bool, pre_norm: bool):
        super().__init__()
        import copy
        self.pre_norm = pre_norm
        self.mha = MultiheadAttention(d_model=d_model, n_heads=n_heads, attention_fn=attention_fn, bias=attention_bias)
        self.ffd = copy.deepcopy(feedforward_fn)
        self.norm1, self.norm2 = copy.deepcopy(layernorm_fn), copy.deepcopy(layernorm_fn)

    def forward(self, x, attn_mask=None):
        assert x.dim() == 3
        if self.pre_norm:
            h = self.norm1(x)
            x = x + self.mha(h, h, h, attn_mask=attn_mask)
            return x + self.ffd(self.norm2(x))
        x = self.norm1(x + self.mha(x, x, x, attn_mask=attn_mask))
        return self.norm2(x + self.ffd(x))


class _PQTrainFused(torch.autograd.Function):
    """PQ 'train' mode as one forward and one backward kernel (csrc/cdist.cu, pq_train_*)."""

    @staticmethod
    def forward(ctx, z, weight):
        w32 = weight.detach().float().contiguous()
        zq, loss = ext.pq_train_fwd(z, w32)
        ctx.save_for_backward(z, w32)
        ctx.w_dtype = weight.dtype
        return zq.view(list(z.shape[:-1]) + [-1]), loss

    @staticmethod
    def backward(ctx, grad_zq, grad_loss):
        z, w32 = ctx.saved_tensors
        if grad_loss is None:
            grad_loss = torch.zeros((), device=z.device)
        gzq = None if grad_zq is None else grad_zq.reshape(-1, z.size(-1)).float().contiguous()
        grad_z, grad_w = ext.pq_train_bwd(z, w32, gzq, grad_loss)
        return grad_z, grad_w.to(ctx.w_dtype)


class PQBase(nn.Module):
    """Product quantizer with one codebook weight[m, c, dc] shared by all heads of a layer
    (reference basic/quantizer.py:6-111).  forward(mode, z), mode in
    {'encode', 'decode', 'quantize', 'train'}:
        encode   z [..., m*dc]  -> codes [..., m]   (int64 for v1 like torch.argmin, int32 for v2)
        decode   codes [..., m] -> centroids [..., m*dc]
        quantize z -> nearest centroids
        train    z -> (nearest centroids, soft/hard centroid MSE loss)
    method 'v1' = torch.cdist(p=1)+argmin (the reference's torch oracle), 'v2' = CUDA kernels."""

    def __init__(self, d_codeword: int, n_codewords: int, n_subspaces: int, method: str):
        super().__init__()
        self.method = method
        self.d_codeword, self.n_codewords, self.n_subspaces = d_codeword, n_codewords, n_subspaces
        self.weight = nn.Parameter(torch.randn(n_subspaces, n_codewords, d_codeword))
        self.loss_fn = nn.MSELoss()
        self.fused_train = True    # v2 on CUDA with 16 codewords x 8: one kernel each way instead of ~10 torch ops

    def _distance_and_codes(self, z_flat):
        if self.method == "v1":
            dist = torch.cdist(z_flat.float(), self.weight.float(), p=1.0).to(z_flat.dtype)
            return dist, dist.argmin(dim=-1, keepdim=True)
        if self.method == "v2":
            dist, codes = kernels.cdist(z_flat, self.weight)
            return dist, codes.unsqueeze(-1)
        raise RuntimeError(f"unknown PQ method {self.method}")

    def forward(self, mode: str, z: torch.Tensor):
        if mode not in ("train", "encode", "decode", "quantize"):
            raise AssertionError(mode)
        assert z.dim() > 1
        m, dc = self.n_subspaces, self.d_codeword
        assert z.size(-1) == (m if mode == "decode" else m * dc)
        out_shape = list(z.shape[:-1]) + [-1]

        if mode == "encode" and self.method == "v2" and z.is_cuda:
            # fused fast path: no [m, n, dc] copy, no distance tensor (SURVEY.md section 8 a-0)
            return ext.pq_encode(z.contiguous(), self.weight)

        if mode == "train" and self.method == "v2" and self.fused_train and ext.pq_train_supported(z, self.weight):
            return _PQTrainFused.apply(z.contiguous(), self.weight)

        z_flat = z.flatten(end_dim=-2).view(-1, m, z.size(-1) // m).transpose(0, 1).contiguous()
        if mode == "decode":
            distance, codes = None, z_flat
        else:
            distance, codes = self._distance_and_codes(z_flat)
        if mode == "encode":
            return codes.transpose(0, 1).reshape(out_shape).contiguous()

        codes = codes.long()
        z_q_flat = torch.gather(self.weight, 1, codes.expand(-1, -1, dc))
        z_q = z_q_flat.transpose(0, 1).reshape(out_shape)
        if mode in ("decode", "quantize"):
            return z_q

        # 'train': soft centroids from inverse distances vs the hard centroid, plus commitment term
        # (computed in fp32 whatever the module dtype: the reference path is fp32 throughout)
        weights = torch.softmax(-torch.log(torch.clamp(distance.float(), min=1e-5)), dim=-1)
        z_w = torch.matmul(weights, self.weight.float())
        loss = self.loss_fn(z_w, z_q_flat.float()) + self.loss_fn(z_flat.float(), z_q_flat.float())
        return z_q, loss


class PQV1(PQBase):
    def __init__(self, d_codeword: int, n_codewords: int, n_subspaces: int):
        super().__init__(d_codeword, n_codewords, n_subspaces, method="v1")


class PQV2(PQBase):
    def __init__(self, d_codeword: int, n_codewords: int, n_subspaces: int):
        super().__init__(d_codeword, n_codewords, n_subspaces, method="v2")
