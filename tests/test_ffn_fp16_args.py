"""Argument checks of the fp16 routed-FFN entry points: they run without a GPU (every dtype check precedes the first
CUDA call, so a rejected call returns SPT_ERR_INVALID_ARGUMENT even where there is no device)."""
import ctypes
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32, BF16, F16 = 0, 1, 2


def _lib():
    import __graft_entry__
    __graft_entry__.build()
    lib = ctypes.CDLL(os.path.join(ROOT, "spt_proto_b200", "lib", "libspt_b200.so"))
    lib.spt_last_error.restype = ctypes.c_char_p
    vp, i32, i64, ll = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_longlong
    lib.spt_grouped_gemm.argtypes = [i32, vp, ll, ll, ll, i32, vp, ll, ll, ll, i32, vp, i32, vp, i32, i32, i32, i32, i32,
                                     i32, i32, i32, ll, ll, vp, ll, i32, vp, i32, vp, i32, vp, ll, i32, vp]
    lib.spt_group_colsum.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp]
    lib.spt_ffn_combine.argtypes = [vp, vp, vp, vp, i64, i32, i32, i32, i32, vp]
    lib.spt_scale_add_fwd.argtypes = [vp, vp, i32, vp, i32, vp, i32, i64, i32, vp]
    lib.spt_scale_add_bwd.argtypes = [vp, vp, i32, vp, i32, vp, vp, i64, i32, vp]
    lib.spt_lora_glu_fwd_ex.argtypes = [vp] * 6 + [i64, i32, i32, vp]
    lib.spt_lora_glu_bwd_ex.argtypes = [vp] * 11 + [i64, i32, i32, vp]
    lib.spt_silu_mul_fwd_ex.argtypes = [vp] * 3 + [i64, i32, vp]
    lib.spt_silu_mul_bwd_ex.argtypes = [vp] * 5 + [i64, i32, vp]
    return lib


def _buf():
    mem = (ctypes.c_uint8 * 256)()
    return mem, (ctypes.addressof(mem) + 15) & ~15       # non-null, 16-byte aligned; never dereferenced


def _gemm(lib, p, c_dtype, ab_dtype):
    """A valid mode-0 call (one 128-row tile, N 128, K 64) in every argument but the dtypes."""
    return lib.spt_grouped_gemm(0, p, 128, 64, 64, 0, p, 128, 64, 64, 0, p, 1, None, 0, 0, 128, 64, 0, 0, 0, 0, 0, 0,
                                p, 128, c_dtype, None, 0, None, 0, None, 0, ab_dtype, None)


@pytest.mark.parametrize("ab_dtype", [F32, 3, -1])
def test_grouped_gemm_rejects_unknown_operand_type(ab_dtype):
    lib = _lib()
    _mem, p = _buf()
    assert _gemm(lib, p, F32, ab_dtype) == 1
    msg = lib.spt_last_error()
    assert b"ab_dtype %d unknown" % ab_dtype in msg and b"SPT_BF16 (1) or SPT_F16 (2)" in msg, msg


@pytest.mark.parametrize("ab_dtype,c_dtype", [(F16, BF16), (BF16, F16), (F16, 3)])
def test_grouped_gemm_rejects_output_of_another_type(ab_dtype, c_dtype):
    lib = _lib()
    _mem, p = _buf()
    assert _gemm(lib, p, c_dtype, ab_dtype) == 1
    msg = lib.spt_last_error()
    assert b"c_dtype %d not allowed" % c_dtype in msg and b"SPT_F32 (0) or the operand type" in msg, msg


def test_dtype_entry_points_reject_unknown_types():
    lib = _lib()
    _mem, p = _buf()
    cases = [
        (lambda d: lib.spt_group_colsum(p, p, p, p, 2, 64, d, None), b"group_colsum: dtype"),
        (lambda d: lib.spt_lora_glu_fwd_ex(p, p, p, p, p, p, 4, 64, d, None), b"lora_glu_fwd: dtype"),
        (lambda d: lib.spt_lora_glu_bwd_ex(*([p] * 11), 4, 64, d, None), b"lora_glu_bwd: dtype"),
        (lambda d: lib.spt_silu_mul_fwd_ex(p, p, p, 64, d, None), b"silu_mul_fwd: dtype"),
        (lambda d: lib.spt_silu_mul_bwd_ex(p, p, p, p, p, 64, d, None), b"silu_mul_bwd: dtype"),
    ]
    for call, text in cases:
        for d in (F32, 3):
            assert call(d) == 1
            msg = lib.spt_last_error()
            assert text in msg and b"SPT_BF16 (1) or SPT_F16 (2)" in msg, msg


@pytest.mark.parametrize("pair", [(BF16, F16), (F16, BF16), (F16, 3), (3, F32)])
def test_ffn_combine_rejects_mixed_16_bit_types(pair):
    lib = _lib()
    _mem, p = _buf()
    assert lib.spt_ffn_combine(p, p, None, p, 4, 64, 2, pair[0], pair[1], None) == 1
    msg = lib.spt_last_error()
    assert b"dtype pair (partial %d, y %d)" % pair in msg and b"bf16 and fp16 do not mix" in msg, msg


def test_scale_add_rejects_mixed_16_bit_types():
    lib = _lib()
    _mem, p = _buf()
    for a, b, o in ((BF16, F16, F32), (F16, F32, BF16), (F32, F32, 3)):
        assert lib.spt_scale_add_fwd(p, p, a, p, b, p, o, 4, 64, None) == 1
        assert b"bf16 and fp16 do not mix" in lib.spt_last_error()
    for a, g in ((BF16, F16), (F16, BF16), (3, F16)):
        assert lib.spt_scale_add_bwd(p, p, a, p, g, p, p, 4, 64, None) == 1
        assert b"bf16 and fp16 do not mix" in lib.spt_last_error()


def test_weight_copy_cache_keys_by_parameter_and_dtype():
    """A weight already in the compute type is used in place with no cache entry; any other is converted once per
    parameter version and per dtype, and repeated lookups of the same parameter return the cached copy."""
    _lib()
    import torch
    from spt_proto_b200.kernels import ffn as F
    w = torch.nn.Parameter(torch.randn(64, 32))
    b16 = F._operand(w, torch.bfloat16)
    assert b16.dtype == torch.bfloat16 and F._operand(w, torch.bfloat16) is b16
    h16 = F._operand(w, torch.float16)
    assert h16.dtype == torch.float16 and F._operand(w, torch.float16) is h16 and F._operand(w, torch.bfloat16) is b16
    with torch.no_grad():
        w.mul_(2.0)                                            # a new parameter version: both copies are redone
    assert torch.equal(F._operand(w, torch.float16), (w.detach() * 1).half())
    assert F._operand(w, torch.bfloat16) is not b16
    for dt in (torch.float16, torch.bfloat16):
        p = torch.nn.Parameter(torch.randn(8, 8).to(dt))
        assert F._operand(p, dt) is p and p not in F._W16
    assert F.compute_dtype(torch.zeros(1, dtype=torch.float16)) == torch.float16
    assert F.compute_dtype(torch.zeros(1)) == F.compute_dtype(torch.zeros(1, dtype=torch.bfloat16)) == torch.bfloat16
