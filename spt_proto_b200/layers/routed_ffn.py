"""Routed FFN layers (reference naive_gpt/layers/sparse/feedforward.py): a sigmoid router activates
n_blocks // 2 (OPT form) or n_blocks // 4 (LLaMA form) column blocks of the FFN per token.

The reference loops over blocks in Python — mask, gather, addmm, activation, matmul, scatter-add,
and a permuted copy of fc2.weight on every call (feedforward.py:47-103).  Here the tokens are
bucketed once on the device and every product of the forward and backward pass is ONE grouped GEMM
on the tcgen05 tensor cores (spt_proto_b200/csrc/ffn_gemm.cu).  Constructors, parameter names
(`fc1`, `fc2`, `router.0`, `gate`, `side`, `down`) and `from_pretrained` match the reference so its
checkpoints load unchanged."""
from __future__ import annotations

import torch
from torch import nn

from .. import ext
from ..kernels import ffn as F
from .basic import Feedforward, LLaMaFeedforward


def _make_router(d_model: int, n_blocks: int) -> nn.Sequential:
    return nn.Sequential(nn.Linear(d_model, n_blocks), nn.Sigmoid())


def _route(router: nn.Module, x2: torch.Tensor, k_active: int):
    prob = router(x2)
    return prob, ext.route_bucket(prob.detach().float().contiguous(), k_active)


class RoutedFFN(Feedforward):
    def __init__(self, d_model: int, d_feedforward: int, block_size: int, activation: nn.Module,
                 p_dropout: float = 0.0):
        super().__init__(d_model, d_feedforward, p_dropout=p_dropout, activation=activation)
        assert d_feedforward % block_size == 0
        self.block_size = block_size
        self.n_blocks = d_feedforward // block_size
        self.router = _make_router(d_model, self.n_blocks)

    @staticmethod
    def from_pretrained(block_size: int, source: Feedforward):
        assert isinstance(source, Feedforward)
        model = RoutedFFN(d_model=source.d_model, d_feedforward=source.d_feedforward, block_size=block_size,
                          activation=source.activation, p_dropout=source.p_dropout)
        result = model.load_state_dict(source.state_dict(), strict=False)
        if len(result.missing_keys) != 2:   # router.0.weight, router.0.bias
            raise RuntimeError
        return model

    @property
    def k_active(self) -> int:
        return self.n_blocks // 2

    def forward(self, x: torch.Tensor):
        if not x.is_cuda:
            raise RuntimeError("RoutedFFN: spt_proto_b200 has no CPU path (x must be a CUDA tensor)")
        x_size = x.size()
        x2 = x.reshape(-1, self.d_model)
        _, bucket = _route(self.router, x2, self.k_active)
        xp = F.gather(x2.to(F.compute_dtype(x)).contiguous(), bucket)
        relu = isinstance(self.activation, nn.ReLU)
        # ReLU: applied in the fc1 epilogue, its backward mask in the epilogue of the GEMM that produces dH
        h = F.blocked_linear_rows(xp, self.fc1.weight, self.fc1.bias, bucket, self.block_size,
                                  act=F.ACT_RELU if relu else F.ACT_NONE, grad_premasked=relu)
        if not relu:
            h = self.activation(h)
        yp = F.blocked_linear_cols(h, self.fc2.weight, bucket, self.block_size, relu_input=relu)
        y = F.combine(yp, bucket, self.fc2.bias, x.dtype)
        return y.view(x_size)


class RoutedLLaMaFFN(LLaMaFeedforward):
    def __init__(self, d_model: int, d_feedforward: int, block_size: int, activation: nn.Module):
        super().__init__(d_model, d_feedforward, activation)
        assert d_feedforward % block_size == 0
        self.block_size = block_size
        self.n_blocks = d_feedforward // block_size
        self.router = _make_router(d_model, self.n_blocks)

    @staticmethod
    def from_pretrained(block_size: int, source: LLaMaFeedforward):
        assert isinstance(source, LLaMaFeedforward)
        model = RoutedLLaMaFFN(d_model=source.d_model, d_feedforward=source.d_feedforward, block_size=block_size,
                               activation=source.activation)
        result = model.load_state_dict(source.state_dict(), strict=False)
        if len(result.missing_keys) != 2:
            raise RuntimeError
        return model

    @property
    def k_active(self) -> int:
        return self.n_blocks // 4        # the plain LLaMA form activates a quarter (feedforward.py:156)

    def forward(self, x: torch.Tensor):
        if not x.is_cuda:
            raise RuntimeError("RoutedLLaMaFFN: spt_proto_b200 has no CPU path (x must be a CUDA tensor)")
        x_size = x.size()
        x2 = x.reshape(-1, self.d_model)
        _, bucket = _route(self.router, x2, self.k_active)
        xp = F.gather(x2.to(F.compute_dtype(x)).contiguous(), bucket)
        g = F.blocked_linear_rows(xp, self.gate.weight, None, bucket, self.block_size)
        s = F.blocked_linear_rows(xp, self.side.weight, None, bucket, self.block_size)
        if isinstance(self.activation, nn.SiLU) and g.numel() % 8 == 0:
            h = F.silu_mul(g, s)                      # one kernel each way instead of the eager act(g) * s chain
        else:
            h = self.activation(g) * s
        yp = F.blocked_linear_cols(h, self.down.weight, bucket, self.block_size)
        y = F.combine(yp, bucket, None, x.dtype)
        return y.view(x_size)
