"""Argument checks of the packed variable-length entry points: they run without a GPU (the C checks precede every CUDA
call, the offsets are validated on the host)."""
import ctypes
import re
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    import __graft_entry__
    __graft_entry__.build()
    lib = ctypes.CDLL(os.path.join(ROOT, "spt_proto_b200", "lib", "libspt_b200.so"))
    lib.spt_last_error.restype = ctypes.c_char_p
    vp, i32, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
    lib.spt_sparse_attn_varlen_fwd.argtypes = [vp] * 8 + [i32, i32, i32, i32, i32, f32, f32, i32, i32, vp]
    lib.spt_sparse_attn_varlen_bwd.argtypes = [vp] * 13 + [i32, i32, i32, i32, i32, f32, f32, i32, i32, vp]
    lib.spt_lookup_mask_varlen_fwd.argtypes = [vp] * 6 + [i32] * 6 + [vp]
    lib.spt_varlen_worklist.argtypes = [vp, i32, i32, i32, vp, vp]
    return lib


def _buf():
    mem = (ctypes.c_uint8 * 256)()
    return mem, (ctypes.addressof(mem) + 15) & ~15       # non-null, 16-byte aligned; never dereferenced


def _fwd(lib, p, n_seq=2, T=256, max_s=128, d=64, H=2):
    return lib.spt_sparse_attn_varlen_fwd(*([p] * 8), n_seq, T, max_s, d, H, 0.1, 10.0, 1, 0, None)


def _bwd(lib, p, n_seq=2, T=256, max_s=128, d=64, H=2):
    return lib.spt_sparse_attn_varlen_bwd(*([p] * 13), n_seq, T, max_s, d, H, 0.1, 10.0, 1, 0, None)


def test_varlen_attention_rejects_head_dim_96():
    lib = _lib()
    _mem, p = _buf()
    for call in (_fwd, _bwd):
        assert call(lib, p, d=96) != 0
        msg = lib.spt_last_error()
        assert b"head dim 96" in msg and b"64, 80 or 128" in msg, msg


@pytest.mark.parametrize("field,value,text", [("n_seq", 0, b"n_seq >= 1"), ("T", 0, b"T >= 1"), ("H", 0, b"H >= 1"),
                                              ("max_s", 0, b"max_seqlen 0"), ("max_s", 70000, b"max_seqlen 70000")])
def test_varlen_attention_rejects_bad_sizes(field, value, text):
    lib = _lib()
    _mem, p = _buf()
    for call in (_fwd, _bwd):
        assert call(lib, p, **{field: value}) != 0
        assert text in lib.spt_last_error(), lib.spt_last_error()


def test_varlen_entry_points_reject_null_and_misaligned_pointers():
    lib = _lib()
    _mem, p = _buf()
    assert lib.spt_sparse_attn_varlen_fwd(*([p] * 7), None, 2, 256, 128, 64, 2, 0.1, 10.0, 1, 0, None) != 0
    assert b"null pointer" in lib.spt_last_error()
    assert lib.spt_sparse_attn_varlen_bwd(None, *([p] * 12), 2, 256, 128, 64, 2, 0.1, 10.0, 1, 0, None) != 0
    assert b"null pointer" in lib.spt_last_error()
    assert _fwd(lib, p + 2) != 0 and b"16-byte aligned" in lib.spt_last_error()
    assert lib.spt_lookup_mask_varlen_fwd(p, p, None, p, p, p, 2, 256, 128, 2, 8, 8, None) != 0
    assert b"null pointer" in lib.spt_last_error()
    assert lib.spt_lookup_mask_varlen_fwd(p, p, p, p, p, p, 0, 256, 128, 2, 8, 8, None) != 0
    assert b"n_seq >= 1" in lib.spt_last_error()
    assert lib.spt_lookup_mask_varlen_fwd(p, p, p, p, p, p, 2, 256, 128, 2, 12, 8, None) != 0
    assert b"8, 10 or 16" in lib.spt_last_error()
    assert lib.spt_varlen_worklist(None, 2, 256, 128, p, None) != 0
    assert b"null pointer" in lib.spt_last_error()


@pytest.mark.parametrize("cu,T,max_s,rule", [
    ([0, 128, 64, 256], 256, None, "non-monotonic"),
    ([0, 128, 256], 320, None, "must equal the token count"),
    ([0, 128, 176], 176, None, "multiples of 4 * sparse_coeff"),
    ([0, 128, 160], 160, None, "at least 8 * sparse_coeff"),
    ([0, 128, 384], 384, 128, "smaller than the longest sequence"),
])
def test_host_cu_seqlens_validation_names_the_rule(cu, T, max_s, rule):
    _lib()
    from spt_proto_b200 import ext
    with pytest.raises(ValueError, match=re.escape(rule)):
        ext.check_cu_seqlens(cu, T, 8, max_s)


def test_host_cu_seqlens_accepts_a_valid_pack():
    _lib()
    from spt_proto_b200 import ext
    assert ext.check_cu_seqlens([0, 64, 160, 416], 416, 8) == 256
