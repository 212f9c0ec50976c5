"""Autograd building blocks of the routed FFN (reference naive_gpt/layers/sparse/feedforward.py:47-85
and its torch-autograd backward), on the tcgen05 grouped GEMM:

    bucket   = route(prob)                              tokens bucketed by active block (no grad)
    Xp       = gather(x, bucket)                        [R, d]    backward: block-ordered combine
    H        = blocked_linear_rows(Xp, W1, b1, act)     [R, bs]   block g uses W1[g*bs:(g+1)*bs, :]
    Yp       = blocked_linear_cols(H, W2)               [R, d]    block g uses W2[:, g*bs:(g+1)*bs]
    y        = combine(Yp, bucket, b2)                  [T, d]    backward: gather

All GEMM operands share one 16-bit compute type (compute_dtype: fp16 for fp16 inputs, bf16 for everything else) with
fp32 accumulation; weight gradients come out in the parameter's dtype, straight from the GEMM epilogue when that is the
compute type."""
import torch
from torch import autograd
from torch.utils.weak import WeakIdKeyDictionary

from .. import ext

ACT_NONE, ACT_RELU, ACT_SILU = 0, 1, 2


def compute_dtype(x: torch.Tensor) -> torch.dtype:
    """The 16-bit type the routed FFN computes in for input x: fp16 for fp16 x (an fp16 model keeps its own precision
    and needs no second copy of its weights), bf16 for every other input (bf16 and fp32 models)."""
    return torch.float16 if x.dtype == torch.float16 else torch.bfloat16


def _grad_buffer(shape, dtype, device, ab_dtype):
    """Weight-gradient output of the K-grouped GEMM on ab_dtype operands: a parameter of that type gets its gradient
    written in it by the GEMM epilogue (fp32 accumulation in TMEM), every other one an fp32 buffer (converted by the
    caller)."""
    return torch.empty(shape, dtype=dtype if dtype == ab_dtype else torch.float32, device=device)


# parameter -> {dtype: (version, copy of that dtype)}.  Keyed by identity: tensor `==` is elementwise, so a dictionary
# that compares its keys by equality (weakref.WeakKeyDictionary) cannot look a tensor up.
_W16 = WeakIdKeyDictionary()


def _operand(weight: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """GEMM operand of a weight in the compute type `dtype`.  A weight already of that type is used in place (no cache
    entry); any other (an fp32 parameter: the reference trains in fp32, script/4-sparse-tuning-0.py:184) is converted
    ONCE per parameter version instead of on every call — the frozen base weights of the LoRA FFN are never converted
    again, trained ones once per optimizer step.  Copies are kept per (parameter, dtype)."""
    if weight.dtype == dtype:
        return weight
    if weight.requires_grad and weight.is_cuda and torch.cuda.is_current_stream_capturing():
        # a trained fp32 weight inside a captured step: the conversion must be part of the graph (replays do not re-run
        # Python, so a cached copy would go stale after the captured optimizer update)
        return weight.detach().to(dtype)
    copies = _W16.get(weight)
    hit = None if copies is None else copies.get(dtype)
    if hit is not None and hit[0] == weight._version and hit[1].device == weight.device:
        return hit[1]
    w16 = weight.detach().to(dtype)
    if copies is None:
        copies = _W16[weight] = {}
    copies[dtype] = (weight._version, w16)
    return w16


_WHOLE_PTR = {}


def _whole_ptr(rows: int, device) -> torch.Tensor:
    """[0, rows] int32 on `device`: the one-group row pointer that turns group_colsum into a plain column sum."""
    key = (rows, str(device))
    t = _WHOLE_PTR.get(key)
    if t is None:
        t = _WHOLE_PTR[key] = torch.tensor([0, rows], dtype=torch.int32, device=device)
    return t


class GatherRows(autograd.Function):
    @staticmethod
    def forward(ctx, x, bucket):
        ctx.bucket = bucket
        return ext.gather_rows(x, bucket.row_token)

    @staticmethod
    def backward(ctx, grad):
        b = ctx.bucket
        return ext.ffn_combine(grad.contiguous(), b.token_rows, None, grad.dtype), None


class CombineRows(autograd.Function):
    @staticmethod
    def forward(ctx, partial, bucket, bias, out_dtype):
        ctx.bucket, ctx.has_bias, ctx.p_dtype = bucket, bias is not None, partial.dtype
        ctx.bias_dtype = None if bias is None else bias.dtype
        return ext.ffn_combine(partial, bucket.token_rows, bias, out_dtype)

    @staticmethod
    def backward(ctx, grad):
        g16 = grad.contiguous().to(compute_dtype(grad))
        d_partial = ext.gather_rows(g16, ctx.bucket.row_token).to(ctx.p_dtype)
        d_bias = None
        # column sum of the 16-bit gradient in fp32, one pass; skipped when the bias is frozen (LoRARoutedFFN's fc2.bias)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            d_bias = ext.group_colsum(g16, _whole_ptr(g16.size(0), g16.device)).reshape(-1).to(ctx.bias_dtype)
        return d_partial, None, d_bias, None


class BlockedLinearRows(autograd.Function):
    """y[i, :] = act(x[i, :] @ W[g*bs:(g+1)*bs, :].T + b[g*bs:(g+1)*bs]) * row_scale[i],  g = block of row i.
    W [F, K] (fc1 / gate / side layout).  act in {none, relu}; other activations are applied by the caller."""

    @staticmethod
    def forward(ctx, x, weight, bias, bucket, bs, act, out_dtype, grad_premasked=False):
        w16 = _operand(weight, x.dtype)
        out_dtype = x.dtype if out_dtype is None else out_dtype
        y = torch.empty(x.size(0), bs, dtype=out_dtype, device=x.device)
        b32 = None if bias is None else bias.float().contiguous()
        ext.grouped_gemm(0, x, False, w16, False, tile_group=bucket.tile_group, N=bs, K=x.size(1), b_mn_off=bs,
                         out=y, bias=b32, bias_stride=bs, act=act)
        ctx.save_for_backward(x, w16, y if act == ACT_RELU else None)
        ctx.bucket, ctx.bs, ctx.act = bucket, bs, act
        ctx.grad_premasked = grad_premasked   # the consumer's backward already applied the ReLU mask (fused epilogue)
        ctx.w_dtype, ctx.w_shape = weight.dtype, weight.shape
        ctx.b_dtype = None if bias is None else bias.dtype
        return y

    @staticmethod
    def backward(ctx, grad):
        x, w16, y = ctx.saved_tensors
        b, bs = ctx.bucket, ctx.bs
        grad = grad.contiguous()
        if ctx.act == ACT_RELU and not ctx.grad_premasked:
            grad = grad * (y > 0)
        if grad.dtype != x.dtype:
            grad = grad.to(x.dtype)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:   # dx[i, :] = grad[i, :] @ W_g : W consumed MN-major, K offset g*bs
            dx = torch.empty_like(x)
            ext.grouped_gemm(0, grad, False, w16, True, tile_group=b.tile_group, N=x.size(1), K=bs, b_k_off=bs, out=dx)
        if ctx.needs_input_grad[1]:   # dW_g = grad_g^T x_g over the bucket's rows
            dw = _grad_buffer(ctx.w_shape, ctx.w_dtype, x.device, x.dtype)   # in the parameter's dtype if it is x's
            ext.grouped_gemm(1, grad, True, x, True, group_ptr=b.bucket_ptr, M=bs, N=x.size(1), c_row_off=bs, out=dw)
            dw = dw.to(ctx.w_dtype)
        if ctx.b_dtype is not None and ctx.needs_input_grad[2]:
            db = ext.group_colsum(grad, b.bucket_ptr).reshape(-1).to(ctx.b_dtype)
        return dx, dw, db, None, None, None, None, None


class BlockedLinearCols(autograd.Function):
    """y[i, :] = (x[i, :] @ W[:, g*bs:(g+1)*bs].T) * row_scale[i],  W [d, F] (fc2 / down layout)."""

    @staticmethod
    def forward(ctx, x, weight, bucket, bs, relu_input=False):
        ctx.relu_input = relu_input   # x is a ReLU output used only here: mask dx by (x > 0) in the GEMM epilogue
        w16 = _operand(weight, x.dtype)
        d = weight.size(0)
        y = torch.empty(x.size(0), d, dtype=x.dtype, device=x.device)
        ext.grouped_gemm(0, x, False, w16, False, tile_group=bucket.tile_group, N=d, K=bs, b_k_off=bs, out=y)
        ctx.save_for_backward(x, w16)
        ctx.bucket, ctx.bs, ctx.w_dtype, ctx.w_shape = bucket, bs, weight.dtype, weight.shape
        return y

    @staticmethod
    def backward(ctx, grad):
        x, w16 = ctx.saved_tensors
        b, bs = ctx.bucket, ctx.bs
        grad = grad.contiguous()
        dx = dw = None
        if ctx.needs_input_grad[0]:   # dx[i, f] = sum_n grad[i, n] W[n, g*bs + f] : W MN-major, N offset g*bs
            dx = torch.empty_like(x)
            ext.grouped_gemm(0, grad, False, w16, True, tile_group=b.tile_group, N=bs, K=grad.size(1), b_mn_off=bs,
                             out=dx, gate=x if ctx.relu_input else None)
        if ctx.needs_input_grad[1]:   # dW[:, g*bs:(g+1)*bs] = grad_g^T x_g
            dw = _grad_buffer(ctx.w_shape, ctx.w_dtype, x.device, x.dtype)
            ext.grouped_gemm(1, grad, True, x, True, group_ptr=b.bucket_ptr, M=grad.size(1), N=bs, c_col_off=bs,
                             out=dw)
            dw = dw.to(ctx.w_dtype)
        return dx, dw, None, None, None


def gather(x, bucket):
    return GatherRows.apply(x, bucket)


def combine(partial, bucket, bias, out_dtype):
    return CombineRows.apply(partial, bucket, bias, out_dtype)


def blocked_linear_rows(x, weight, bias, bucket, bs, act=ACT_NONE, out_dtype=None, grad_premasked=False):
    """x is in the compute type (bf16 or fp16); out_dtype None gives x's type, torch.float32 keeps the fp32 accumulator (used where the result feeds an activation gate
    after further additions, so that gates are decided in fp32 like in the reference).
    grad_premasked: with act=relu, the incoming gradient already carries the (y > 0) mask — set together
    with blocked_linear_cols(relu_input=True) when y feeds that product and nothing else."""
    return BlockedLinearRows.apply(x, weight, bias, bucket, bs, act, out_dtype, grad_premasked)


def blocked_linear_cols(x, weight, bucket, bs, relu_input=False):
    return BlockedLinearCols.apply(x, weight, bucket, bs, relu_input)


class BlockedLinearColsT(autograd.Function):
    """y[i, :] = x[i, :] @ W[g*bs:(g+1)*bs, :],  W [F, n] row-blocked, reduction over the block's rows
    (h L2_i of the LoRA FFN: W = fc2.lora.left.weight [F, r]).  W is consumed MN-major in place."""

    @staticmethod
    def forward(ctx, x, weight, bucket, bs):
        w16 = _operand(weight, x.dtype)
        n = weight.size(1)
        y = torch.empty(x.size(0), n, dtype=x.dtype, device=x.device)
        ext.grouped_gemm(0, x, False, w16, True, tile_group=bucket.tile_group, N=n, K=bs, b_k_off=bs, out=y)
        ctx.save_for_backward(x, w16)
        ctx.bucket, ctx.bs, ctx.w_dtype, ctx.w_shape = bucket, bs, weight.dtype, weight.shape
        return y

    @staticmethod
    def backward(ctx, grad):
        x, w16 = ctx.saved_tensors
        b, bs = ctx.bucket, ctx.bs
        grad = grad.contiguous()
        dx = dw = None
        if ctx.needs_input_grad[0]:   # dx[i, f] = sum_n grad[i, n] W[g*bs + f, n] : W K-major, N offset g*bs
            dx = torch.empty_like(x)
            ext.grouped_gemm(0, grad, False, w16, False, tile_group=b.tile_group, N=bs, K=grad.size(1), b_mn_off=bs,
                             out=dx)
        if ctx.needs_input_grad[1]:   # dW[g*bs:(g+1)*bs, :] = x_g^T grad_g
            dw = _grad_buffer(ctx.w_shape, ctx.w_dtype, x.device, x.dtype)
            ext.grouped_gemm(1, x, True, grad, True, group_ptr=b.bucket_ptr, M=bs, N=grad.size(1), c_row_off=bs,
                             out=dw)
            dw = dw.to(ctx.w_dtype)
        return dx, dw, None, None


def blocked_linear_cols_t(x, weight, bucket, bs):
    return BlockedLinearColsT.apply(x, weight, bucket, bs)


class ScaleAdd(autograd.Function):
    """out = coeff[:, None] * a + b in one pass (coeff [R] fp32 carries the router gradient of the LoRA FFN)."""

    @staticmethod
    def forward(ctx, coeff, a, b, out_dtype):
        coeff = coeff.contiguous()
        ctx.save_for_backward(coeff, a)
        ctx.b_dtype = b.dtype
        return ext.scale_add_fwd(coeff, a, b, out_dtype)

    @staticmethod
    def backward(ctx, grad):
        coeff, a = ctx.saved_tensors
        grad = grad.contiguous()
        da, dcoeff = ext.scale_add_bwd(coeff, a, grad)
        db = grad if grad.dtype == ctx.b_dtype else grad.to(ctx.b_dtype)
        return dcoeff, da, db, None


class LoraGLU(autograd.Function):
    """h = silu(coeff * bg + lg) * (coeff * bs + ls) -> bf16 / fp16 in one pass; backward in one pass as well."""

    @staticmethod
    def forward(ctx, coeff, bg, lg, bs, ls, out_dtype):
        coeff = coeff.contiguous()
        ctx.save_for_backward(coeff, bg, lg, bs, ls)
        return ext.lora_glu_fwd(coeff, bg, lg, bs, ls, out_dtype)

    @staticmethod
    def backward(ctx, grad):
        coeff, bg, lg, bs, ls = ctx.saved_tensors
        d_bg, d_lg, d_bs, d_ls, dcoeff = ext.lora_glu_bwd(coeff, bg, lg, bs, ls, grad.contiguous())
        return dcoeff, d_bg, d_lg, d_bs, d_ls, None


class SiluMul(autograd.Function):
    """h = silu(gate) * side in one pass each way (the plain RoutedLLaMaFFN's `act(gate) * side`)."""

    @staticmethod
    def forward(ctx, gate, side):
        ctx.save_for_backward(gate, side)
        return ext.silu_mul_fwd(gate, side)

    @staticmethod
    def backward(ctx, grad):
        gate, side = ctx.saved_tensors
        return ext.silu_mul_bwd(gate, side, grad.contiguous())


def silu_mul(gate, side):
    return SiluMul.apply(gate, side)


def scale_add(coeff, a, b, out_dtype):
    return ScaleAdd.apply(coeff, a, b, out_dtype)


def lora_glu(coeff, bg, lg, bs, ls, out_dtype=torch.bfloat16):
    return LoraGLU.apply(coeff, bg, lg, bs, ls, out_dtype)
