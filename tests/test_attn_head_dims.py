"""Head-dim validation of the fused attention entry points: runs without a GPU (the check precedes every CUDA call)."""
import ctypes
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    import __graft_entry__
    __graft_entry__.build()
    lib = ctypes.CDLL(os.path.join(ROOT, "spt_proto_b200", "lib", "libspt_b200.so"))
    lib.spt_last_error.restype = ctypes.c_char_p
    vp, i32, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
    lib.spt_sparse_attn_fwd_ex.argtypes = [vp] * 7 + [i32, i32, i32, i32, f32, f32, i32, i32, vp]
    lib.spt_sparse_attn_bwd_ex.argtypes = [vp] * 12 + [i32, i32, i32, i32, f32, f32, i32, i32, vp]
    return lib


def _fwd(lib, buf, S, d):
    return lib.spt_sparse_attn_fwd_ex(*([buf] * 7), 2, S, d, 1, 0.1, 10.0, 1, 0, None)


def _bwd(lib, buf, S, d):
    return lib.spt_sparse_attn_bwd_ex(*([buf] * 12), 2, S, d, 1, 0.1, 10.0, 1, 0, None)


def test_attention_rejects_head_dim_96_naming_the_supported_ones():
    lib = _lib()
    mem = (ctypes.c_uint8 * 256)()
    buf = (ctypes.addressof(mem) + 15) & ~15      # non-null, 16-byte aligned; never dereferenced
    for call in (_fwd, _bwd):
        rc = call(lib, buf, 256, 96)
        msg = lib.spt_last_error()
        assert rc != 0 and b"head dim 96" in msg and b"64, 80 or 128" in msg, msg


def test_attention_accepts_head_dim_80():
    """d = 80 passes the head-dim check: the first complaint about a bad call is then its sequence length."""
    lib = _lib()
    mem = (ctypes.c_uint8 * 256)()
    buf = (ctypes.addressof(mem) + 15) & ~15
    for call in (_fwd, _bwd):
        rc = call(lib, buf, 100, 80)
        msg = lib.spt_last_error()
        assert rc != 0 and b"head dim" not in msg and b"multiple of 128" in msg, msg
