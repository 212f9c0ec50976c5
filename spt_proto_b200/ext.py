"""Drop-in replacement for the reference's torch CUDA extension `naive_gpt.ext`
(reference extension/entry.cpp:43-56): the same 7 function names, arity, argument meaning, return
values and error type (RuntimeError, as TORCH_CHECK raises), implemented as a thin ctypes binding
over the C ABI of include/spt_b200.h (libspt_b200.so, hand-written sm_100a kernels).

Differences from the reference, all relaxations:
  * bf16 operands are accepted next to fp32 (outputs that are "values" stay fp32);
  * the shape whitelists are lifted (cdist: any n / n_codewords; lookup: any (m, nnz) with m >= 4,
    nnz % 4 == 0; softmax: any row length);
  * every kernel runs on torch's CURRENT stream (the reference launches its hand kernels on the
    legacy default stream, extension/cdist.cu:214 — a latent ordering hazard, SURVEY.md section 3a).

Extra entry points (SURVEY.md section 8b): pq_encode, csr2csc, spmm_csc, sddmm_scaled, ffn_*.
There is no CPU path: tensors must be CUDA tensors and the library must be built.
"""
from __future__ import annotations

from typing import List, Tuple

import torch

from ._lib import SPT_ATTN_Y_TRANSPOSED, SPT_BF16, SPT_F16, SPT_F32, check, lib

_DTYPES = {torch.float32: SPT_F32, torch.bfloat16: SPT_BF16}
# fp16 is taken by the PQ encode / train kernels, the fused attention and the routed-FFN entry points (grouped_gemm,
# gather_rows, ffn_combine, group_colsum, scale_add_*, silu_mul_*, lora_glu_*), not by the stage entry points
_PQ_DTYPES = {**_DTYPES, torch.float16: SPT_F16}
_ATTN_DTYPES = {torch.bfloat16: SPT_BF16, torch.float16: SPT_F16}
_FFN_DTYPES = {**_DTYPES, torch.float16: SPT_F16}          # fp32 or a 16-bit type (bf16 and fp16 never mix in one call)
_HALF_DTYPES = {torch.bfloat16: SPT_BF16, torch.float16: SPT_F16}   # grouped GEMM operands, gathered rows, ...

# softmax_backward_cuda computes the TRUE softmax gradient.  The shipped reference kernel clamps the row
# dot product sum(y * dy) to >= 1e-9 (extension/softmax.cu:69), which is wrong whenever that sum is
# negative.  Set this flag (or SPT_REFERENCE_SOFTMAX_CLAMP=1 in the environment) to reproduce the shipped
# kernel bit for bit in training-parity A/B runs; it applies to the stage kernel (the fused attention
# path always uses the true gradient: route through the stage path with use_fused=False for such runs).
import os as _os

REFERENCE_SOFTMAX_CLAMP = _os.environ.get("SPT_REFERENCE_SOFTMAX_CLAMP", "0") not in ("", "0")


# ---- validation helpers (mirror CHECK_DIM / CHECK_TYPE, extension/common.h:13-21) -----------------
def _check_dim(x: torch.Tensor, d: int, name: str) -> None:
    if not isinstance(x, torch.Tensor):
        raise RuntimeError(f"{name} must be a tensor")
    if not x.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor")
    if x.dim() != d:
        raise RuntimeError(f"{name} must be of dim {d}")
    if not x.is_contiguous():
        raise RuntimeError(f"{name} custom kernel requires contiguous tensor")


def _check_type(x: torch.Tensor, t: torch.dtype, name: str) -> None:
    if x.dtype != t:
        raise RuntimeError(f"{name} must be type of {t}")


def _float_code(x: torch.Tensor, name: str) -> int:
    code = _DTYPES.get(x.dtype)
    if code is None:
        raise RuntimeError(f"{name} must be type of torch.float32 or torch.bfloat16")
    return code


def _pq_code(x: torch.Tensor, name: str) -> int:
    code = _PQ_DTYPES.get(x.dtype)
    if code is None:
        raise RuntimeError(f"{name} must be type of torch.float32, torch.bfloat16 or torch.float16")
    return code


def _ffn_code(x: torch.Tensor, name: str) -> int:
    code = _FFN_DTYPES.get(x.dtype)
    if code is None:
        raise RuntimeError(f"{name} must be type of torch.float32, torch.bfloat16 or torch.float16 (got {x.dtype})")
    return code


def _half_code(x: torch.Tensor, name: str) -> int:
    code = _HALF_DTYPES.get(x.dtype)
    if code is None:
        raise RuntimeError(f"{name} must be type of torch.bfloat16 or torch.float16 (got {x.dtype})")
    return code


def _stream(x: torch.Tensor) -> int:
    return torch.cuda.current_stream(x.device).cuda_stream


def _p(x) -> int:
    return 0 if x is None else x.data_ptr()


class _on_device:
    """Make x's device current for the duration of a launch (no-op in the common case)."""

    def __init__(self, x: torch.Tensor):
        self.idx = x.device.index
        self.prev = None

    def __enter__(self):
        cur = torch.cuda.current_device()
        if self.idx is not None and self.idx != cur:
            self.prev = cur
            torch.cuda.set_device(self.idx)

    def __exit__(self, *exc):
        if self.prev is not None:
            torch.cuda.set_device(self.prev)


def _workspace(nbytes: int, like: torch.Tensor) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=like.device)


# ---- (1) cdist ---------------------------------------------------------------------------------------
def cdist_forward_cuda(query: torch.Tensor, table: torch.Tensor) -> List[torch.Tensor]:
    """query [m, n, dc], table [m, c, dc] -> [distance [m, n, c] f32, indices [m, n] i32]
    (extension/cdist.cu:185-249)."""
    _check_dim(query, 3, "query")
    _check_dim(table, 3, "table")
    code = _float_code(query, "query")
    if query.size(0) != table.size(0) or query.size(-1) != table.size(-1):
        raise RuntimeError("query and table must agree in n_subspaces and d_code")
    table32 = table if table.dtype == torch.float32 else table.float()
    m, n, dc = query.shape
    c = table.size(1)
    distance = torch.empty((m, n, c), dtype=torch.float32, device=query.device)
    indices = torch.empty((m, n), dtype=torch.int32, device=query.device)
    with _on_device(query):
        check(lib.spt_cdist_fwd(_p(query), _p(table32), _p(distance), _p(indices), m, n, c, dc, code,
                                _stream(query)))
    return [distance, indices]


def cdist_backward_cuda(query: torch.Tensor, table: torch.Tensor, grad_output: torch.Tensor) -> List[torch.Tensor]:
    """-> [grad_query [m,n,dc], grad_table [m,c,dc]] (extension/cdist.cu:251-333)."""
    _check_dim(query, 3, "query")
    _check_dim(table, 3, "table")
    _check_dim(grad_output, 3, "grad_output")
    _check_type(query, torch.float32, "query")
    _check_type(table, torch.float32, "table")
    _check_type(grad_output, torch.float32, "grad_output")
    m, n, dc = query.shape
    c = table.size(1)
    if (table.size(0) != m or table.size(2) != dc or grad_output.size(0) != m
            or grad_output.size(1) != n or grad_output.size(2) != c):
        raise RuntimeError("cdist_backward: shape mismatch")
    grad_query = torch.empty_like(query)
    grad_table = torch.empty_like(table)
    ws = _workspace(lib.spt_cdist_bwd_workspace_bytes(m, n, c, dc), query)
    with _on_device(query):
        check(lib.spt_cdist_bwd(_p(query), _p(table), _p(grad_output), _p(grad_query), _p(grad_table), _p(ws),
                                m, n, c, dc, _stream(query)))
    return [grad_query, grad_table]


def pq_encode(z: torch.Tensor, table: torch.Tensor) -> torch.Tensor:
    """Fused PQBase.forward(mode='encode') (quantizer.py:26-77): z [..., m*dc] -> codes [..., m] int32,
    straight from the head-major layout (no [m, n, dc] transposed copy, no distance tensor)."""
    if not z.is_cuda or not z.is_contiguous():
        raise RuntimeError("z must be a contiguous CUDA tensor")
    _check_dim(table, 3, "table")
    code = _pq_code(z, "z")
    m, c, dc = table.shape
    if z.size(-1) != m * dc:
        raise RuntimeError("z last dim must equal n_subspaces * d_codeword")
    table32 = table if table.dtype == torch.float32 else table.float()
    rows = z.numel() // (m * dc)
    codes = torch.empty(list(z.shape[:-1]) + [m], dtype=torch.int32, device=z.device)
    with _on_device(z):
        check(lib.spt_pq_encode(_p(z), _p(table32), _p(codes), rows, m, c, dc, code, _stream(z)))
    return codes


def pq_encode_pair(z0: torch.Tensor, z1: torch.Tensor, table: torch.Tensor):
    """pq_encode of two same-shaped tensors sharing the codebook (q and k of one attention call) in one
    launch -> (codes0, codes1)."""
    if not (z0.is_cuda and z1.is_cuda and z0.is_contiguous() and z1.is_contiguous()):
        raise RuntimeError("z0 and z1 must be contiguous CUDA tensors")
    if z0.shape != z1.shape or z0.dtype != z1.dtype:
        raise RuntimeError("z0 and z1 must have the same shape and dtype")
    _check_dim(table, 3, "table")
    code = _pq_code(z0, "z0")
    m, c, dc = table.shape
    if z0.size(-1) != m * dc:
        raise RuntimeError("z last dim must equal n_subspaces * d_codeword")
    table32 = table if table.dtype == torch.float32 else table.float()
    rows = z0.numel() // (m * dc)
    shape = list(z0.shape[:-1]) + [m]
    codes0 = torch.empty(shape, dtype=torch.int32, device=z0.device)
    codes1 = torch.empty(shape, dtype=torch.int32, device=z0.device)
    with _on_device(z0):
        check(lib.spt_pq_encode_pair(_p(z0), _p(z1), _p(table32), _p(codes0), _p(codes1), rows, m, c, dc, code,
                                     _stream(z0)))
    return codes0, codes1


def pq_train_supported(z: torch.Tensor, table: torch.Tensor) -> bool:
    return (z.is_cuda and z.dtype in _PQ_DTYPES and table.dim() == 3 and table.size(1) == 16 and table.size(2) == 8
            and table.size(0) <= 64 and z.size(-1) == table.size(0) * 8 and z.numel() > 0)


def pq_train_fwd(z: torch.Tensor, table32: torch.Tensor):
    """Fused PQ 'train' forward: -> (zq [rows, m*dc] fp32 hard centroids, loss scalar fp32)."""
    m, c, dc = table32.shape
    rows = z.numel() // (m * dc)
    zq = torch.empty((rows, m * dc), dtype=torch.float32, device=z.device)
    partial = torch.empty((lib.spt_pq_train_blocks(rows, m),), dtype=torch.float32, device=z.device)
    with _on_device(z):
        check(lib.spt_pq_train_fwd(_p(z), _p(table32), _p(zq), _p(partial), rows, m, c, dc, _pq_code(z, "z"), _stream(z)))
    return zq, partial.sum() / float(rows * m * dc)


def pq_train_bwd(z: torch.Tensor, table32: torch.Tensor, grad_zq, grad_loss: torch.Tensor):
    """-> (grad_z like z, grad_table [m, c, dc] fp32)."""
    m, c, dc = table32.shape
    rows = z.numel() // (m * dc)
    grad_z = torch.empty_like(z)
    partial = torch.empty((lib.spt_pq_train_blocks(rows, m), m, c, dc), dtype=torch.float32, device=z.device)
    gl = grad_loss.reshape(1).float().contiguous()
    with _on_device(z):
        check(lib.spt_pq_train_bwd(_p(z), _p(table32), _p(grad_zq), _p(gl), _p(grad_z), _p(partial), rows, m, c, dc,
                                   _pq_code(z, "z"), _stream(z)))
    return grad_z, partial.sum(0)


# ---- (2) lookup --------------------------------------------------------------------------------------
def lookup_forward_cuda(config: torch.Tensor, query: torch.Tensor, key: torch.Tensor) -> torch.Tensor:
    """config carries sparse_coeff in its SHAPE (kernels/lookup.py:23, lookup.cu:99);
    query, key [B, S, m] int32 codes -> [B, S, S // sparse_coeff] int32 (extension/lookup.cu:87-174)."""
    _check_dim(key, 3, "key")
    _check_dim(query, 3, "query")
    _check_type(key, torch.int32, "key")
    _check_type(query, torch.int32, "query")
    if query.shape != key.shape:
        raise RuntimeError("query and key must have the same shape")
    sparsity = int(config.size(0))
    B, S, m = query.shape
    if sparsity <= 0 or S % sparsity != 0:
        raise RuntimeError("seq_length must be divisible by sparse_coeff")
    nnz = S // sparsity
    output = torch.empty((B, S, nnz), dtype=torch.int32, device=query.device)
    ws = _workspace(lib.spt_lookup_workspace_bytes(B, S, m, nnz), query)
    with _on_device(query):
        check(lib.spt_lookup_fwd(_p(query), _p(key), _p(output), _p(ws), B, S, m, nnz, _stream(query)))
    return output


# ---- (3) sddmm ---------------------------------------------------------------------------------------
def _flag(t) -> bool:
    return bool(t.item()) if isinstance(t, torch.Tensor) else bool(t)


def _check_csr(indptr, indices, S: int) -> None:
    _check_dim(indptr, 1, "indptr")
    _check_dim(indices, 2, "indices")
    _check_type(indptr, torch.int32, "indptr")
    _check_type(indices, torch.int32, "indices")
    if indptr.size(-1) != S + 1:
        raise RuntimeError("indptr must have seq_length + 1 entries")


def sddmm_scaled(indptr, indices, query, key, scale: float = 1.0, clamp: float = 0.0) -> torch.Tensor:
    _check_dim(key, 3, "key")
    _check_dim(query, 3, "query")
    if query.shape != key.shape or query.dtype != key.dtype:
        raise RuntimeError("query and key must have the same shape and dtype")
    B, S, d = query.shape
    _check_csr(indptr, indices, S)
    if indices.size(0) != B:
        raise RuntimeError("indices batch must match query batch")
    code = _float_code(query, "query")
    nnz = indices.size(-1)
    values = torch.empty((B, nnz), dtype=torch.float32, device=query.device)
    with _on_device(query):
        check(lib.spt_sddmm_fwd(_p(indptr), _p(indices), _p(query), _p(key), _p(values), B, S, d, nnz,
                                float(scale), float(clamp), code, _stream(query)))
    return values


def clamp_scale_bwd(grad: torch.Tensor, clamped: torch.Tensor, scale: float, clamp: float) -> torch.Tensor:
    """Gradient of clamp(scale * raw, -clamp, clamp) w.r.t. raw, given the clamped values (one pass)."""
    _check_type(grad, torch.float32, "grad")
    _check_type(clamped, torch.float32, "clamped")
    if grad.shape != clamped.shape or not grad.is_contiguous() or not clamped.is_contiguous():
        raise RuntimeError("grad and clamped must be contiguous tensors of the same shape")
    out = torch.empty_like(grad)
    with _on_device(grad):
        check(lib.spt_clamp_scale_bwd(_p(grad), _p(clamped), _p(out), grad.numel(), float(scale), float(clamp), _stream(grad)))
    return out


def sddmm_forward_cuda(trans_lhs, trans_rhs, indptr, indices, query, key) -> torch.Tensor:
    """values[b, e] = <query[b, row(e)], key[b, indices[b, e]]> (extension/sddmm.cpp:3-73).  Only the
    (N, T) operand layout the reference ever uses (kernels/sddmm.py:19-22, kernels/spmm.py:37-40)."""
    if _flag(trans_lhs) or not _flag(trans_rhs):
        raise RuntimeError("sddmm_forward_cuda: only trans_lhs=False, trans_rhs=True is supported")
    return sddmm_scaled(indptr, indices, query, key)


# ---- (a-7) csr2csc + (5) spmm ------------------------------------------------------------------------
def csr2csc(indptr: torch.Tensor, indices: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """-> (col_ptr [B, S+1], row_idx [B, nnz], perm [B, nnz]); stable (rows ascending per column)."""
    S = indptr.size(-1) - 1
    _check_csr(indptr, indices, S)
    B, nnz = indices.shape
    dev = indices.device
    col_ptr = torch.empty((B, S + 1), dtype=torch.int32, device=dev)
    row_idx = torch.empty((B, nnz), dtype=torch.int32, device=dev)
    perm = torch.empty((B, nnz), dtype=torch.int32, device=dev)
    ws = _workspace(lib.spt_csr2csc_workspace_bytes(B, S, nnz), indices)
    with _on_device(indices):
        check(lib.spt_csr2csc(_p(indptr), _p(indices), _p(col_ptr), _p(row_idx), _p(perm), _p(ws), B, S, nnz,
                              _stream(indices)))
    return col_ptr, row_idx, perm


def _check_spmm(indptr, indices, values, x):
    _check_dim(x, 3, "x")
    _check_dim(values, 2, "values")
    B, S, d = x.shape
    _check_csr(indptr, indices, S)
    _check_type(values, torch.float32, "values")
    if indices.size(0) != B or indices.shape != values.shape:
        raise RuntimeError("indices / values / x shape mismatch")
    return B, S, d, indices.size(-1), _float_code(x, "x")


def spmm_csc(csc, values: torch.Tensor, x: torch.Tensor, out_dtype=None) -> torch.Tensor:
    """y = A^T x using a CSC from csr2csc(); values stay in CSR order (gathered through perm)."""
    col_ptr, row_idx, perm = csc
    _check_dim(x, 3, "x")
    _check_dim(values, 2, "values")
    _check_type(values, torch.float32, "values")
    B, S, d = x.shape
    nnz = values.size(-1)
    code = _float_code(x, "x")
    if out_dtype is None:
        out_dtype = x.dtype
    y = torch.empty((B, S, d), dtype=out_dtype, device=x.device)
    with _on_device(x):
        check(lib.spt_spmm_t_fwd(_p(col_ptr), _p(row_idx), _p(perm), _p(values), _p(x), _p(y), B, S, d, nnz,
                                 code, _DTYPES[out_dtype], _stream(x)))
    return y


def csr_tiles_supported(indices: torch.Tensor, x: torch.Tensor) -> bool:
    """Can the transposed product A^T x run on the tile index (csr_tiles / spmm_tiles)?  bf16 x, head dim 64 / 128,
    at most 2^20 entries per head, S <= 8192."""
    return bool(x.dtype == torch.bfloat16 and x.dim() == 3 and x.size(-1) in (64, 128) and x.is_contiguous()
                and lib.spt_csr_tiles_supported(x.size(1), indices.size(-1)))


def csr_tiles(indptr: torch.Tensor, indices: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """-> (tile_ptr [B, n*n + 1] int32, tile_ent [B, nnz] int32 bit patterns): the entries of every head bucketed by
    (64-column tile, 64-row chunk) — what the transposed product needs of a CSC, at a fraction of its cost."""
    S = indptr.size(-1) - 1
    _check_csr(indptr, indices, S)
    B, nnz = indices.shape
    if not lib.spt_csr_tiles_supported(S, nnz):
        raise RuntimeError(f"csr_tiles: S={S} / nnz={nnz} beyond the tile index format (S <= 8192, nnz <= 2^20 per head)")
    tile_ptr = torch.empty((B, lib.spt_csr_tiles_ptr_len(S)), dtype=torch.int32, device=indices.device)
    tile_ent = torch.empty((B, nnz), dtype=torch.int32, device=indices.device)
    with _on_device(indices):
        check(lib.spt_csr_tiles(_p(indptr), _p(indices), _p(tile_ptr), _p(tile_ent), B, S, nnz, _stream(indices)))
    return tile_ptr, tile_ent


def sddmm_tiles(tiles, query: torch.Tensor, key: torch.Tensor, scale: float = 1.0, clamp: float = 0.0) -> torch.Tensor:
    """values[b, e] = clamp(scale * <query[b, row(e)], key[b, col(e)]>) for the entries of a tile index (bf16, d 64 / 128)."""
    tile_ptr, tile_ent = tiles
    _check_dim(key, 3, "key")
    _check_dim(query, 3, "query")
    if query.shape != key.shape or query.dtype != key.dtype:
        raise RuntimeError("query and key must have the same shape and dtype")
    B, S, d = query.shape
    nnz = tile_ent.size(-1)
    if tile_ent.size(0) != B:
        raise RuntimeError("sddmm_tiles: tile index batch must match query batch")
    code = _float_code(query, "query")
    values = torch.empty((B, nnz), dtype=torch.float32, device=query.device)   # every entry of a valid pattern is in the index
    with _on_device(query):
        check(lib.spt_sddmm_tiles_fwd(_p(tile_ptr), _p(tile_ent), _p(query), _p(key), _p(values), B, S, d, nnz,
                                      float(scale), float(clamp), code, _stream(query)))
    return values


def spmm_tiles(tiles, values: torch.Tensor, x: torch.Tensor, out_dtype=None, trans: bool = True) -> torch.Tensor:
    """y = A^T x (trans, the default) or y = A x on a tile index from csr_tiles(); values stay in CSR order."""
    tile_ptr, tile_ent = tiles
    _check_dim(x, 3, "x")
    _check_dim(values, 2, "values")
    _check_type(values, torch.float32, "values")
    B, S, d = x.shape
    nnz = values.size(-1)
    if tile_ent.shape != values.shape or tile_ptr.size(0) != B:
        raise RuntimeError("spmm_tiles: tile index / values / x shape mismatch")
    code = _float_code(x, "x")
    if out_dtype is None:
        out_dtype = x.dtype
    y = torch.empty((B, S, d), dtype=out_dtype, device=x.device)
    with _on_device(x):
        check(lib.spt_spmm_tiles_fwd(_p(tile_ptr), _p(tile_ent), _p(values), _p(x), _p(y), B, S, d, nnz, code,
                                     _DTYPES[out_dtype], 1 if trans else 0, _stream(x)))
    return y


def spmm_forward_cuda(trans_lhs, trans_rhs, indptr, indices, values, x) -> torch.Tensor:
    """y = op(A) x, A = batched CSR with shared indptr (extension/spmm.cpp:3-72).  trans_lhs=True is
    the transposed product of the backward passes; it builds the CSC on the fly (callers that need
    it twice should use csr2csc() + spmm_csc(), as spt_proto_b200.kernels does)."""
    if _flag(trans_rhs):
        raise RuntimeError("spmm_forward_cuda: trans_rhs=True is not supported")
    B, S, d, nnz, code = _check_spmm(indptr, indices, values, x)
    if _flag(trans_lhs):
        if csr_tiles_supported(indices, x):      # bf16, head dim 64 / 128: tile index instead of a CSC
            return spmm_tiles(csr_tiles(indptr, indices), values, x, out_dtype=x.dtype)
        return spmm_csc(csr2csc(indptr, indices), values, x, out_dtype=x.dtype)
    y = torch.empty_like(x)
    with _on_device(x):
        check(lib.spt_spmm_fwd(_p(indptr), _p(indices), _p(values), _p(x), _p(y), B, S, d, nnz, code, code,
                               _stream(x)))
    return y


# ---- (4) softmax -------------------------------------------------------------------------------------
def softmax_forward_cuda(indptr, indices, values) -> torch.Tensor:
    """Causal CSR row softmax (extension/softmax.cu:84-114)."""
    _check_dim(values, 2, "values")
    _check_csr(indptr, indices, indptr.size(-1) - 1)
    _check_type(values, torch.float32, "values")
    if indices.shape != values.shape:
        raise RuntimeError("indices and values must have the same shape")
    B, nnz = indices.shape
    S = indptr.size(-1) - 1
    output = torch.empty_like(values)
    with _on_device(values):
        check(lib.spt_softmax_fwd(_p(indptr), _p(indices), _p(values), _p(output), B, S, nnz, _stream(values)))
    return output


def softmax_backward_cuda(indptr, indices, output, grad_output) -> torch.Tensor:
    """True softmax gradient on the kept entries (extension/softmax.cu:116-148 without its clamp bug;
    REFERENCE_SOFTMAX_CLAMP = True reproduces the shipped kernel, clamp included)."""
    _check_dim(output, 2, "output")
    _check_dim(grad_output, 2, "grad_output")
    _check_csr(indptr, indices, indptr.size(-1) - 1)
    _check_type(output, torch.float32, "output")
    _check_type(grad_output, torch.float32, "grad_output")
    if grad_output.shape != output.shape or indices.shape != output.shape:
        raise RuntimeError("indices / output / grad_output shape mismatch")
    B, nnz = indices.shape
    S = indptr.size(-1) - 1
    grad_values = torch.empty_like(output)
    with _on_device(output):
        check(lib.spt_softmax_bwd_ex(_p(indptr), _p(indices), _p(output), _p(grad_output), _p(grad_values), B, S, nnz,
                                     int(REFERENCE_SOFTMAX_CLAMP), _stream(output)))
    return grad_values


def softmax_clamp_bwd(indptr, indices, output, grad_output, clamped, scale: float, clamp: float) -> torch.Tensor:
    """softmax_backward_cuda followed by clamp_scale_bwd in one pass: the gradient w.r.t. the raw sddmm scores of
    softmax(clamp(scale * raw, -clamp, clamp)), bit-identical to the two-kernel chain."""
    _check_csr(indptr, indices, indptr.size(-1) - 1)
    for name, t in (("output", output), ("grad_output", grad_output), ("clamped", clamped)):
        _check_dim(t, 2, name)
        _check_type(t, torch.float32, name)
        if t.shape != indices.shape or not t.is_contiguous():
            raise RuntimeError(f"{name} must be contiguous with the shape of indices")
    B, nnz = indices.shape
    S = indptr.size(-1) - 1
    grad_raw = torch.empty_like(output)
    with _on_device(output):
        check(lib.spt_softmax_clamp_bwd(_p(indptr), _p(indices), _p(output), _p(grad_output), _p(clamped), _p(grad_raw), B, S,
                                        nnz, float(scale), float(clamp), int(REFERENCE_SOFTMAX_CLAMP), _stream(output)))
    return grad_raw


def launch_count() -> int:
    """Kernel launches issued through libspt_b200 by this process so far."""
    return int(lib.spt_launch_count())


# ---- fused sparse attention (masked dense tiles on the tensor cores) ------------------------------------
def _heads(t: torch.Tensor, name: str):
    """(B, S, H): 3-D [B, S, *] is head-major (H = 1); 4-D [N, S, H, *] has the heads interleaved."""
    if t.dim() == 3:
        return t.size(0), t.size(1), 1
    if t.dim() == 4:
        return t.size(0) * t.size(2), t.size(1), t.size(2)
    raise RuntimeError(f"{name} must be of dim 3 ([B,S,*]) or 4 ([N,S,H,*])")


LOOKUP_MAX_SEQ = 65536    # longest S of lookup_mask (include/spt_b200.h): the key indices of the reference fit uint16


def lookup_mask(query: torch.Tensor, key: torch.Tensor, sparse_coeff: int, want_indices: bool = False,
                n_codewords=None):
    """Same selection as lookup_forward_cuda, emitted as (mask [B,S,S/32] int32 bit-words in the
    lane-major layout: word 4g+t bit i <=> key 128g+4i+t, extra0 [B,S] int32 zero-padding multiplicity
    of key 0, indices [B,S,nnz] or None).
    Codes: [B,S,m] head-major or [N,S,H,m] (heads interleaved, B = N*H).
    n_codewords: the caller's promise that every code is < n_codewords (the codebook size).  At lengths where
    the fallback for codes >= 16 cannot run (beyond about 16 k tokens at sparse_coeff 8) only n_codewords <= 16
    lets the call run; None makes no promise (include/spt_b200.h, spt_lookup_mask_fwd_ex)."""
    _check_dim(key, query.dim(), "key")
    _check_type(key, torch.int32, "key")
    _check_type(query, torch.int32, "query")
    if query.shape != key.shape or not query.is_cuda or not query.is_contiguous():
        raise RuntimeError("query and key must be contiguous CUDA tensors of the same shape")
    B, S, H = _heads(query, "query")
    m = query.size(-1)
    if sparse_coeff <= 0 or S % sparse_coeff != 0 or S % 128 != 0:
        raise RuntimeError("seq_length must be divisible by sparse_coeff and by 128")
    nnz = S // sparse_coeff
    dev = query.device
    mask = torch.empty((B, S, S // 32), dtype=torch.int32, device=dev)
    extra0 = torch.empty((B, S), dtype=torch.int32, device=dev)
    indices = torch.empty((B, S, nnz), dtype=torch.int32, device=dev) if want_indices else None
    ws = _workspace(lib.spt_lookup_workspace_bytes(B, S, m, nnz), query)
    with _on_device(query):
        if n_codewords is None:
            check(lib.spt_lookup_mask_fwd(_p(query), _p(key), _p(indices), _p(mask), _p(extra0), _p(ws), B, S, m, nnz, H,
                                          _stream(query)))
        else:
            check(lib.spt_lookup_mask_fwd_ex(_p(query), _p(key), _p(indices), _p(mask), _p(extra0), _p(ws), B, S, m, nnz,
                                             H, int(n_codewords), _stream(query)))
    return mask, extra0, indices


def _check_attn(q, k, v):
    """-> (B, S, d, H, dtype code): q, k, v of one shape and one dtype, bf16 or fp16."""
    if q.dtype not in _ATTN_DTYPES:
        raise RuntimeError("q must be type of torch.bfloat16 or torch.float16")
    for name, t in (("q", q), ("k", k), ("v", v)):
        _check_dim(t, q.dim(), name)
        _check_type(t, q.dtype, name)
    if q.shape != k.shape or q.shape != v.shape:
        raise RuntimeError("q, k, v must have the same shape")
    B, S, H = _heads(q, "q")
    return B, S, q.size(-1), H, _ATTN_DTYPES[q.dtype]


def sparse_attn_fwd(q, k, v, mask, extra0, scale: float, clamp: float = 10.0, reference_layout: bool = False):
    """q, k, v: [B,S,d] head-major or [N,S,H,d] (native layer layout, no transposes), all bf16 or all fp16
    -> (y, same shape and dtype as q; zsum [B,S] fp32).  fp16 needs 0 <= clamp <= 10.  reference_layout: y's MEMORY is the shipped layer's y^T [B, d, S]
    (attention.py:139-142), returned viewed with q's shape.  See include/spt_b200.h."""
    B, S, d, H, code = _check_attn(q, k, v)
    y = torch.empty_like(q)
    zsum = torch.empty((B, S), dtype=torch.float32, device=q.device)
    with _on_device(q):
        check(lib.spt_sparse_attn_fwd_ex(_p(q), _p(k), _p(v), _p(mask), _p(extra0), _p(y), _p(zsum), B, S, d, H,
                                         float(scale), float(clamp), code,
                                         SPT_ATTN_Y_TRANSPOSED if reference_layout else 0, _stream(q)))
    return y, zsum


def sparse_attn_bwd(q, k, v, y, grad_y, mask, extra0, zsum, scale: float, clamp: float = 10.0,
                    reference_layout: bool = False):
    """-> (grad_q, grad_k, grad_v) in q's dtype.  reference_layout: y and grad_y are in the layout
    sparse_attn_fwd(..., reference_layout=True) returned."""
    B, S, d, H, code = _check_attn(q, k, v)
    _check_dim(grad_y, q.dim(), "grad_y")
    _check_type(grad_y, q.dtype, "grad_y")
    _check_type(y, q.dtype, "y")
    gq, gk, gv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    ws = _workspace(lib.spt_sparse_attn_bwd_workspace_bytes(B, S), q)
    with _on_device(q):
        check(lib.spt_sparse_attn_bwd_ex(_p(q), _p(k), _p(v), _p(y), _p(grad_y), _p(mask), _p(extra0), _p(zsum),
                                         _p(gq), _p(gk), _p(gv), _p(ws), B, S, d, H, float(scale), float(clamp), code,
                                         SPT_ATTN_Y_TRANSPOSED if reference_layout else 0, _stream(q)))
    return gq, gk, gv


# ---- packed variable-length sequences (include/spt_b200.h, DESIGN.md section 4.5) ------------------------------
def check_cu_seqlens(cu_seqlens, T: int, sparse_coeff: int, max_seqlen=None) -> int:
    """Validate host-side sequence offsets of a packed batch of T tokens; returns the longest length.
    Raises ValueError naming the broken rule."""
    cu = [int(x) for x in (cu_seqlens.tolist() if isinstance(cu_seqlens, torch.Tensor) else cu_seqlens)]
    if len(cu) < 2 or cu[0] != 0:
        raise ValueError("cu_seqlens must start with 0 and hold at least one sequence")
    lengths = [b - a for a, b in zip(cu[:-1], cu[1:])]
    if any(n <= 0 for n in lengths):
        raise ValueError("cu_seqlens must be strictly increasing (non-monotonic offsets)")
    if cu[-1] != T:
        raise ValueError(f"the last offset of cu_seqlens ({cu[-1]}) must equal the token count T = {T}")
    step = 4 * sparse_coeff
    for i, n in enumerate(lengths):
        if n % step or n % 32:
            raise ValueError(f"sequence {i} has length {n}: lengths must be multiples of 4 * sparse_coeff = {step} and of 32")
        if n < 8 * sparse_coeff:
            raise ValueError(f"sequence {i} has length {n}: lengths must be at least 8 * sparse_coeff = {8 * sparse_coeff}")
    longest = max(lengths)
    if max_seqlen is not None and int(max_seqlen) < longest:
        raise ValueError(f"max_seqlen {max_seqlen} is smaller than the longest sequence ({longest})")
    return longest


def _tokens(t: torch.Tensor, name: str):
    """(T, H) of a packed [T, H, *] or [1, T, H, *] tensor."""
    if t.dim() == 4 and t.size(0) == 1:
        return t.size(1), t.size(2)
    if t.dim() == 3:
        return t.size(0), t.size(1)
    raise RuntimeError(f"{name} must be [T, H, *] or [1, T, H, *]")


def _cu_device(cu_seqlens, like: torch.Tensor) -> torch.Tensor:
    if not (isinstance(cu_seqlens, torch.Tensor) and cu_seqlens.is_cuda and cu_seqlens.dtype == torch.int32
            and cu_seqlens.dim() == 1 and cu_seqlens.is_contiguous()):
        raise RuntimeError("cu_seqlens must be a contiguous 1-D int32 CUDA tensor")
    if cu_seqlens.device != like.device:
        raise RuntimeError("cu_seqlens must be on the operands' device")
    return cu_seqlens


def varlen_worklist(cu_seqlens: torch.Tensor, T: int, max_seqlen: int) -> torch.Tensor:
    """Work list of a packed batch (one item per sequence and 128-row tile, heaviest first), built on the device from
    cu_seqlens without a host synchronisation; pass it to lookup_mask_varlen / sparse_attn_varlen_*."""
    n_seq = cu_seqlens.numel() - 1
    work = torch.empty(max(int(lib.spt_varlen_worklist_bytes(n_seq, T)), 16) // 4, dtype=torch.int32,
                       device=cu_seqlens.device)
    with _on_device(cu_seqlens):
        check(lib.spt_varlen_worklist(_p(cu_seqlens), n_seq, T, int(max_seqlen), _p(work), _stream(cu_seqlens)))
    return work


def lookup_mask_varlen_max_seqlen(m: int) -> int:
    """Longest max_seqlen lookup_mask_varlen takes at m subspaces (0: m not supported)."""
    return int(lib.spt_lookup_mask_varlen_max_seqlen(m))


def lookup_mask_varlen(query: torch.Tensor, key: torch.Tensor, cu_seqlens: torch.Tensor, max_seqlen: int,
                       sparse_coeff: int, work=None, n_codewords=None):
    """lookup_mask of every sequence of a packed batch alone, in one launch per kernel.  Codes [T, H, m] or [1, T, H, m]
    int32; cu_seqlens int32 [n + 1] on the device -> (mask [H, T, 4 ceil(max_seqlen / 128)] int32 lane-major words
    relative to each sequence's start, extra0 [H, T] int32).  n_codewords: as in lookup_mask."""
    _check_type(query, torch.int32, "query")
    _check_type(key, torch.int32, "key")
    if query.shape != key.shape or not query.is_cuda or not query.is_contiguous() or not key.is_contiguous():
        raise RuntimeError("query and key must be contiguous CUDA tensors of the same shape")
    T, H = _tokens(query, "query")
    m = query.size(-1)
    cu = _cu_device(cu_seqlens, query)
    n_seq = cu.numel() - 1
    if work is None:
        work = varlen_worklist(cu, T, max_seqlen)
    words = 4 * ((int(max_seqlen) + 127) // 128)
    mask = torch.empty((H, T, words), dtype=torch.int32, device=query.device)
    extra0 = torch.empty((H, T), dtype=torch.int32, device=query.device)
    ws = _workspace(lib.spt_lookup_mask_varlen_workspace_bytes(n_seq, T, H, m), query)
    with _on_device(query):
        if n_codewords is None:
            check(lib.spt_lookup_mask_varlen_fwd(_p(query), _p(key), _p(work), _p(mask), _p(extra0), _p(ws), n_seq, T,
                                                 int(max_seqlen), H, m, int(sparse_coeff), _stream(query)))
        else:
            check(lib.spt_lookup_mask_varlen_fwd_ex(_p(query), _p(key), _p(work), _p(mask), _p(extra0), _p(ws), n_seq, T,
                                                    int(max_seqlen), H, m, int(sparse_coeff), int(n_codewords),
                                                    _stream(query)))
    return mask, extra0


def sparse_attn_varlen_fwd(q, k, v, mask, extra0, cu_seqlens, max_seqlen: int, scale: float, clamp: float = 10.0,
                           reference_layout: bool = False, work=None):
    """sparse_attn_fwd of every sequence of a packed batch: q, k, v [T, H, d] or [1, T, H, d] -> (y like q, zsum [H, T]).
    reference_layout: sequence i's y memory is its own y_i^T [H, d, S_i] at token offset cu[i]."""
    _B, _S, d, _H, code = _check_attn(q, k, v)
    T, H = _tokens(q, "q")
    cu = _cu_device(cu_seqlens, q)
    if work is None:
        work = varlen_worklist(cu, T, max_seqlen)
    y = torch.empty_like(q)
    zsum = torch.empty((H, T), dtype=torch.float32, device=q.device)
    with _on_device(q):
        check(lib.spt_sparse_attn_varlen_fwd(_p(q), _p(k), _p(v), _p(mask), _p(extra0), _p(y), _p(zsum), _p(work),
                                             cu.numel() - 1, T, int(max_seqlen), d, H, float(scale), float(clamp), code,
                                             SPT_ATTN_Y_TRANSPOSED if reference_layout else 0, _stream(q)))
    return y, zsum


def sparse_attn_varlen_bwd(q, k, v, y, grad_y, mask, extra0, zsum, cu_seqlens, max_seqlen: int, scale: float,
                           clamp: float = 10.0, reference_layout: bool = False, work=None):
    """-> (grad_q, grad_k, grad_v) of sparse_attn_varlen_fwd."""
    _B, _S, d, _H, code = _check_attn(q, k, v)
    T, H = _tokens(q, "q")
    _check_type(grad_y, q.dtype, "grad_y")
    _check_type(y, q.dtype, "y")
    if grad_y.shape != q.shape or not grad_y.is_contiguous():
        raise RuntimeError("grad_y must be contiguous with q's shape")
    cu = _cu_device(cu_seqlens, q)
    if work is None:
        work = varlen_worklist(cu, T, max_seqlen)
    gq, gk, gv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
    ws = _workspace(lib.spt_sparse_attn_varlen_bwd_workspace_bytes(T, H), q)
    with _on_device(q):
        check(lib.spt_sparse_attn_varlen_bwd(_p(q), _p(k), _p(v), _p(y), _p(grad_y), _p(mask), _p(extra0), _p(zsum),
                                             _p(gq), _p(gk), _p(gv), _p(ws), _p(work), cu.numel() - 1, T, int(max_seqlen),
                                             d, H, float(scale), float(clamp), code,
                                             SPT_ATTN_Y_TRANSPOSED if reference_layout else 0, _stream(q)))
    return gq, gk, gv


# ---- (6) routed FFN: grouped GEMM on tcgen05 ------------------------------------------------------------
def grouped_gemm(mode: int, A: torch.Tensor, a_mn_major: bool, B: torch.Tensor, b_mn_major: bool, *,
                 tile_group=None, group_ptr=None, M: int = 0, N: int, K: int = 0,
                 a_k_off: int = 0, a_mn_off: int = 0, b_k_off: int = 0, b_mn_off: int = 0,
                 c_row_off: int = 0, c_col_off: int = 0, out: torch.Tensor, bias=None, bias_stride: int = 0,
                 row_scale=None, act: int = 0, gate=None) -> torch.Tensor:
    """Thin binding of spt_grouped_gemm (see include/spt_b200.h).  A, B: 2-D tensors as stored (row-major, possibly
    with a row stride), both bf16 or both fp16; `gate` of the same type; `out`: 2-D fp32 tensor or one of the operand
    type, written in place."""
    for name, t in (("A", A), ("B", B)):
        if not (t.is_cuda and t.dim() == 2 and t.dtype in _HALF_DTYPES and t.stride(1) == 1):
            raise RuntimeError(f"{name} must be a 2-D bf16 or fp16 CUDA tensor with unit inner stride")
    if A.dtype != B.dtype:
        raise RuntimeError(f"A and B must have the same dtype (A is {A.dtype}, B is {B.dtype})")
    if gate is not None and gate.dtype != A.dtype:
        raise RuntimeError(f"gate must have the operands' dtype {A.dtype} (got {gate.dtype})")
    if not (out.is_cuda and out.dim() == 2 and out.stride(1) == 1):
        raise RuntimeError("out must be a 2-D CUDA tensor with unit inner stride")
    if out.dtype not in (torch.float32, A.dtype):
        raise RuntimeError(f"out must be torch.float32 or the operand type {A.dtype} (got {out.dtype})")
    n_groups = 0 if group_ptr is None else group_ptr.numel() - 1
    n_m_tiles = 0 if tile_group is None else tile_group.numel()
    with _on_device(A):
        check(lib.spt_grouped_gemm(
            mode, _p(A), A.size(0), A.size(1), A.stride(0), int(a_mn_major), _p(B), B.size(0), B.size(1), B.stride(0),
            int(b_mn_major), _p(tile_group), n_m_tiles, _p(group_ptr), n_groups, M, N, K, a_k_off, a_mn_off, b_k_off,
            b_mn_off, c_row_off, c_col_off, _p(out), out.stride(0), _FFN_DTYPES[out.dtype], _p(bias), bias_stride,
            _p(row_scale), act, _p(gate), 0 if gate is None else gate.stride(0), _HALF_DTYPES[A.dtype], _stream(A)))
    return out


class Bucket:
    """Device-side token -> block bucketing produced by route_bucket() (see include/spt_b200.h)."""
    __slots__ = ("T", "nb", "k", "R", "bucket_ptr", "bucket_rows", "tile_group", "row_token", "row_prob", "token_rows")


def route_bucket(prob: torch.Tensor, k_active: int) -> Bucket:
    """prob [T, nb] fp32 router probabilities -> padded bucket layout.  No host synchronisation: the
    row capacity R is the static upper bound round_up(T*k + 127*nb, 128)."""
    _check_dim(prob, 2, "prob")
    _check_type(prob, torch.float32, "prob")
    T, nb = prob.shape
    dev = prob.device
    b = Bucket()
    b.T, b.nb, b.k = T, nb, k_active
    b.R = (T * k_active + 127 * nb + 127) // 128 * 128
    i32 = dict(dtype=torch.int32, device=dev)
    b.bucket_ptr = torch.empty(nb + 1, **i32)
    b.bucket_rows = torch.empty(nb, **i32)
    b.tile_group = torch.empty(b.R // 128, **i32)
    b.row_token = torch.empty(b.R, **i32)
    b.row_prob = torch.empty(b.R, dtype=torch.float32, device=dev)
    b.token_rows = torch.empty(T, k_active, **i32)
    ws = _workspace(lib.spt_route_bucket_workspace_bytes(T, nb), prob)
    with _on_device(prob):
        check(lib.spt_route_bucket(_p(prob), _p(b.bucket_ptr), _p(b.bucket_rows), _p(b.tile_group), _p(b.row_token),
                                   _p(b.row_prob), _p(b.token_rows), _p(ws), T, nb, k_active, b.R, _stream(prob)))
    return b


def row_coeff_bwd(grad_coeff: torch.Tensor, bucket: "Bucket") -> torch.Tensor:
    """grad_prob [T, nb] fp32 of coeff[r] = 2 * prob[token(r), block(r)] (zeros where a (token, block) pair is inactive)."""
    _check_type(grad_coeff, torch.float32, "grad_coeff")
    if grad_coeff.numel() != bucket.R or not grad_coeff.is_contiguous():
        raise RuntimeError("grad_coeff must be a contiguous [R] tensor")
    grad_prob = torch.empty(bucket.T, bucket.nb, dtype=torch.float32, device=grad_coeff.device)
    with _on_device(grad_coeff):
        check(lib.spt_row_coeff_bwd(_p(grad_coeff), _p(bucket.row_token), _p(bucket.tile_group), _p(grad_prob), bucket.R,
                                    bucket.T, bucket.nb, _stream(grad_coeff)))
    return grad_prob


def gather_rows(src: torch.Tensor, row_token: torch.Tensor) -> torch.Tensor:
    """dst[r] = src[row_token[r]] (zeros for padding rows); src [T, C] bf16 or fp16, dst of the same type."""
    _check_dim(src, 2, "src")
    _half_code(src, "src")
    R, C = row_token.numel(), src.size(1)
    dst = torch.empty(R, C, dtype=src.dtype, device=src.device)
    with _on_device(src):
        check(lib.spt_gather_rows_bf16(_p(src), _p(row_token), _p(dst), R, C, _stream(src)))
    return dst


def ffn_combine(partial: torch.Tensor, token_rows: torch.Tensor, bias, out_dtype) -> torch.Tensor:
    """y[t] = bias + sum_j partial[token_rows[t, j]] in ascending block order (fp32 accumulation).  partial and y are
    fp32, bf16 or fp16; a 16-bit partial goes with its own type or fp32, bf16 and fp16 do not mix."""
    _check_dim(partial, 2, "partial")
    T, k = token_rows.shape
    C = partial.size(1)
    y = torch.empty(T, C, dtype=out_dtype, device=partial.device)
    bias32 = None if bias is None else bias.float().contiguous()
    with _on_device(partial):
        check(lib.spt_ffn_combine(_p(partial), _p(token_rows), _p(bias32), _p(y), T, C, k, _ffn_code(partial, "partial"),
                                  _ffn_code(y, "out"), _stream(partial)))
    return y


def group_colsum(x: torch.Tensor, bucket_ptr: torch.Tensor) -> torch.Tensor:
    """out[g, c] = sum of x[row, c] over bucket g's rows; x [R, C] bf16 or fp16 -> [G, C] fp32."""
    _check_dim(x, 2, "x")
    code = _half_code(x, "x")
    G, C = bucket_ptr.numel() - 1, x.size(1)
    out = torch.empty(G, C, dtype=torch.float32, device=x.device)
    ws = _workspace(lib.spt_group_colsum_workspace_bytes(G, C), x)
    with _on_device(x):
        check(lib.spt_group_colsum(_p(x), _p(bucket_ptr), _p(out), _p(ws), G, C, code, _stream(x)))
    return out


# ---- fused elementwise stages of the LoRA-routed FFN (csrc/lora_fuse.cu) ---------------------------------------------
def _rows_cols(a: torch.Tensor, name: str):
    _check_dim(a, 2, name)
    if not a.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")
    return a.size(0), a.size(1)


def scale_add_fwd(coeff: torch.Tensor, a: torch.Tensor, b: torch.Tensor, out_dtype) -> torch.Tensor:
    """out[r, :] = coeff[r] * a[r, :] + b[r, :];  coeff [R] fp32, a / b / out each fp32 or one 16-bit type (bf16 or
    fp16: the two do not mix)."""
    R, C = _rows_cols(a, "a")
    _check_type(coeff, torch.float32, "coeff")
    if b.shape != a.shape or coeff.numel() != R or not b.is_contiguous() or not coeff.is_contiguous():
        raise RuntimeError("scale_add: shape mismatch")
    out = torch.empty(R, C, dtype=out_dtype, device=a.device)
    with _on_device(a):
        check(lib.spt_scale_add_fwd(_p(coeff), _p(a), _ffn_code(a, "a"), _p(b), _ffn_code(b, "b"), _p(out),
                                    _ffn_code(out, "out"), R, C, _stream(a)))
    return out


def scale_add_bwd(coeff: torch.Tensor, a: torch.Tensor, grad: torch.Tensor):
    """-> (da = coeff * grad in a's dtype, dcoeff [R] fp32 = rowsum(grad * a))."""
    R, C = _rows_cols(a, "a")
    if grad.shape != a.shape or not grad.is_contiguous():
        raise RuntimeError("scale_add_bwd: shape mismatch")
    da = torch.empty_like(a)
    dcoeff = torch.empty(R, dtype=torch.float32, device=a.device)
    with _on_device(a):
        check(lib.spt_scale_add_bwd(_p(coeff), _p(a), _ffn_code(a, "a"), _p(grad), _ffn_code(grad, "grad"), _p(da),
                                    _p(dcoeff), R, C, _stream(a)))
    return da, dcoeff


def silu_mul_fwd(gate: torch.Tensor, side: torch.Tensor) -> torch.Tensor:
    """h = silu(gate) * side, tensors of the same shape and type, bf16 or fp16 (fp32 math, one rounding)."""
    code = _half_code(gate, "gate")
    _check_type(side, gate.dtype, "side")
    if gate.shape != side.shape or not gate.is_contiguous() or not side.is_contiguous() or gate.numel() % 8:
        raise RuntimeError("silu_mul: gate / side must be contiguous, equal-shaped, with a multiple of 8 elements")
    h = torch.empty_like(gate)
    with _on_device(gate):
        check(lib.spt_silu_mul_fwd_ex(_p(gate), _p(side), _p(h), gate.numel(), code, _stream(gate)))
    return h


def silu_mul_bwd(gate: torch.Tensor, side: torch.Tensor, grad_h: torch.Tensor):
    """-> (grad_gate, grad_side) in gate's type."""
    code = _half_code(gate, "gate")
    for t, n in ((side, "side"), (grad_h, "grad_h")):
        _check_type(t, gate.dtype, n)
    if grad_h.shape != gate.shape or not grad_h.is_contiguous():
        raise RuntimeError("silu_mul_bwd: shape mismatch")
    dg, ds = torch.empty_like(gate), torch.empty_like(side)
    with _on_device(gate):
        check(lib.spt_silu_mul_bwd_ex(_p(gate), _p(side), _p(grad_h), _p(dg), _p(ds), gate.numel(), code, _stream(gate)))
    return dg, ds


def lora_glu_fwd(coeff, bg, lg, bs, ls, out_dtype=torch.bfloat16) -> torch.Tensor:
    """h (out_dtype: bf16 or fp16) = silu(coeff * bg + lg) * (coeff * bs + ls); all inputs fp32 [R, C], coeff [R]."""
    R, C = _rows_cols(bg, "bg")
    for t, n in ((bg, "bg"), (lg, "lg"), (bs, "bs"), (ls, "ls"), (coeff, "coeff")):
        _check_type(t, torch.float32, n)
        if n != "coeff" and (t.shape != bg.shape or not t.is_contiguous()):
            raise RuntimeError("lora_glu: shape mismatch")
    h = torch.empty(R, C, dtype=out_dtype, device=bg.device)
    code = _half_code(h, "h")
    with _on_device(bg):
        check(lib.spt_lora_glu_fwd_ex(_p(coeff), _p(bg), _p(lg), _p(bs), _p(ls), _p(h), R, C, code, _stream(bg)))
    return h


def lora_glu_bwd(coeff, bg, lg, bs, ls, grad_h):
    """-> (d_bg, d_lg, d_bs, d_ls fp32 [R, C], dcoeff [R] fp32); grad_h bf16 or fp16."""
    R, C = _rows_cols(bg, "bg")
    code = _half_code(grad_h, "grad_h")
    if grad_h.shape != bg.shape or not grad_h.is_contiguous():
        raise RuntimeError("lora_glu_bwd: shape mismatch")
    outs = [torch.empty_like(bg) for _ in range(4)]
    dcoeff = torch.empty(R, dtype=torch.float32, device=bg.device)
    with _on_device(bg):
        check(lib.spt_lora_glu_bwd_ex(_p(coeff), _p(bg), _p(lg), _p(bs), _p(ls), _p(grad_h), *[_p(o) for o in outs],
                                      _p(dcoeff), R, C, code, _stream(bg)))
    return (*outs, dcoeff)


# ---- RMSNorm / RoPE of the block around the SPT operators (csrc/norm_rope.cu) ------------------------------------
def rmsnorm_supported(x: torch.Tensor, weight: torch.Tensor) -> bool:
    C = x.size(-1)
    return (x.is_cuda and x.dtype == torch.bfloat16 and weight.dtype == torch.bfloat16 and weight.is_cuda
            and C % 8 == 0 and 8 <= C <= 8192 and x.numel() > 0)


def rmsnorm_fwd(x: torch.Tensor, weight: torch.Tensor, eps: float):
    """-> (out like x, inv_rms [rows] fp32); x [..., C] bf16 contiguous, weight [C] bf16."""
    C = x.size(-1)
    rows = x.numel() // C
    out = torch.empty_like(x)
    inv = torch.empty(rows, dtype=torch.float32, device=x.device)
    with _on_device(x):
        check(lib.spt_rmsnorm_fwd_bf16(_p(x), _p(weight), _p(out), _p(inv), rows, C, float(eps), _stream(x)))
    return out, inv


def rmsnorm_bwd(grad: torch.Tensor, x: torch.Tensor, weight: torch.Tensor, inv: torch.Tensor):
    """-> (dx like x, dw [C] fp32)."""
    C = x.size(-1)
    rows = x.numel() // C
    dx = torch.empty_like(x)
    partial = torch.empty(lib.spt_rmsnorm_bwd_blocks(rows), C, dtype=torch.float32, device=x.device)
    with _on_device(x):
        check(lib.spt_rmsnorm_bwd_bf16(_p(grad), _p(x), _p(weight), _p(inv), _p(dx), _p(partial), rows, C, _stream(x)))
    return dx, partial.sum(0)


def rope_supported(x: torch.Tensor, cos: torch.Tensor) -> bool:
    return (x.is_cuda and x.dim() == 4 and x.dtype == torch.bfloat16 and cos.dtype == torch.bfloat16
            and x.size(-1) % 16 == 0 and x.numel() > 0)


def rope(x: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, transpose: bool = False) -> torch.Tensor:
    """x [N, S, H, E] bf16 contiguous; cos / sin [S, E] bf16 contiguous (gathered by position)."""
    N, S, H, E = x.shape
    if cos.shape != (S, E) or sin.shape != (S, E):
        raise RuntimeError("rope: cos / sin must be [S, E]")
    out = torch.empty_like(x)
    with _on_device(x):
        check(lib.spt_rope_bf16(_p(x), _p(cos), _p(sin), _p(out), N * S * H, S, H, E, int(transpose), _stream(x)))
    return out


def swap12_supported(x: torch.Tensor) -> bool:
    return (x.is_cuda and x.dim() == 4 and x.is_contiguous() and x.numel() > 0
            and (x.size(3) * x.element_size()) % 16 == 0 and x.data_ptr() % 16 == 0)


def swap12(x: torch.Tensor) -> torch.Tensor:
    """x [A, B, C, E] contiguous -> x.transpose(1, 2).contiguous() = [A, C, B, E] (16-byte-word row moves)."""
    if not swap12_supported(x):
        raise RuntimeError("swap12: need a contiguous 4-D CUDA tensor with rows of a multiple of 16 bytes")
    A, B, C, E = x.shape
    out = torch.empty(A, C, B, E, dtype=x.dtype, device=x.device)
    with _on_device(x):
        check(lib.spt_swap_dims12(_p(x), _p(out), A, B, C, E * x.element_size(), _stream(x)))
    return out


def transpose_last2_supported(x: torch.Tensor) -> bool:
    return x.is_cuda and x.dim() == 3 and x.is_contiguous() and x.numel() > 0 and x.element_size() in (2, 4) \
        and x.size(0) <= 65535


def transpose_last2(x: torch.Tensor) -> torch.Tensor:
    """x [B, R, C] contiguous -> x.transpose(1, 2).contiguous() = [B, C, R]."""
    if not transpose_last2_supported(x):
        raise RuntimeError("transpose_last2: need a contiguous 3-D CUDA tensor of 2- or 4-byte elements")
    B, R, C = x.shape
    out = torch.empty(B, C, R, dtype=x.dtype, device=x.device)
    with _on_device(x):
        check(lib.spt_transpose_last2(_p(x), _p(out), B, R, C, x.element_size(), _stream(x)))
    return out
