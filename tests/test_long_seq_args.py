"""Long sequences without a GPU: the codebook-size promise of the _ex lookup entry points, the S envelope of the fused
layers, and the rotary tables past max_length."""
import ctypes
import os
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPT_ERR_UNSUPPORTED = 2


def _lib():
    import __graft_entry__
    __graft_entry__.build()
    lib = ctypes.CDLL(os.path.join(ROOT, "spt_proto_b200", "lib", "libspt_b200.so"))
    lib.spt_last_error.restype = ctypes.c_char_p
    vp, i32 = ctypes.c_void_p, ctypes.c_int
    lib.spt_lookup_mask_fwd.argtypes = [vp] * 6 + [i32] * 5 + [vp]
    lib.spt_lookup_mask_fwd_ex.argtypes = [vp] * 6 + [i32] * 6 + [vp]
    lib.spt_lookup_mask_varlen_fwd.argtypes = [vp] * 6 + [i32] * 6 + [vp]
    lib.spt_lookup_mask_varlen_fwd_ex.argtypes = [vp] * 6 + [i32] * 7 + [vp]
    return lib


def _buf():
    mem = (ctypes.c_uint8 * 256)()
    return mem, (ctypes.addressof(mem) + 15) & ~15       # non-null, 16-byte aligned; never dereferenced


@pytest.mark.parametrize("m", [8, 10, 16])
@pytest.mark.parametrize("S", [32768, 65536])
def test_ex_rejects_large_codebooks_beyond_the_fallback(S, m):
    """S 32768 / 65536 at sparse_coeff 8: the codes >= 16 fallback's row images exceed its limit, so n_codewords > 16
    is unsupported (status 2, before any CUDA call) and the message names the limit; the old entry point fails as it
    did (invalid argument)."""
    lib = _lib()
    _mem, p = _buf()
    nnz = S // 8
    assert lib.spt_lookup_mask_fwd_ex(p, p, None, p, p, p, 1, S, m, nnz, 1, 64, None) == SPT_ERR_UNSUPPORTED
    msg = lib.spt_last_error()
    assert b"n_codewords <= 16" in msg and b"(got 64)" in msg and b"204800" in msg, msg
    assert lib.spt_lookup_mask_fwd(p, p, None, p, p, p, 1, S, m, nnz, 1, None) == 1
    assert b"too large for the shared-memory row images" in lib.spt_last_error()
    # packed: one sequence of S tokens
    assert lib.spt_lookup_mask_varlen_fwd_ex(p, p, p, p, p, p, 1, S, S, 1, m, 8, 17, None) == SPT_ERR_UNSUPPORTED
    msg = lib.spt_last_error()
    assert b"n_codewords <= 16" in msg and b"(got 17)" in msg and b"204800" in msg, msg
    assert lib.spt_lookup_mask_varlen_fwd(p, p, p, p, p, p, 1, S, S, 1, m, 8, None) == 1
    assert b"too large for the row images" in lib.spt_last_error()


def test_ex_rejects_index_output_and_other_m_beyond_the_fallback():
    """Without the fallback only the mask-only lookup at m 8, 10, 16 runs: index output or m 12 is unsupported there
    even with n_codewords <= 16."""
    lib = _lib()
    _mem, p = _buf()
    assert lib.spt_lookup_mask_fwd_ex(p, p, p, p, p, p, 1, 32768, 16, 4096, 1, 16, None) == SPT_ERR_UNSUPPORTED
    assert lib.spt_lookup_mask_fwd_ex(p, p, None, p, p, p, 1, 32768, 12, 4096, 1, 16, None) == SPT_ERR_UNSUPPORTED
    assert b"mask-only" in lib.spt_last_error()


def test_ex_checks_n_codewords():
    lib = _lib()
    _mem, p = _buf()
    assert lib.spt_lookup_mask_fwd_ex(p, p, None, p, p, p, 1, 1024, 8, 128, 1, 0, None) == 1
    assert b"n_codewords must be >= 1" in lib.spt_last_error()
    assert lib.spt_lookup_mask_varlen_fwd_ex(p, p, p, p, p, p, 1, 1024, 1024, 1, 8, 8, 0, None) == 1
    assert b"n_codewords must be >= 1" in lib.spt_last_error()


def test_varlen_max_seqlen_is_the_lookup_limit():
    from spt_proto_b200 import ext
    for m in range(1, 40):
        assert ext.lookup_mask_varlen_max_seqlen(m) == (65536 if m in (8, 10, 16) else 0), m


def _fake_q(S, d, H=4):
    """What _fused_ok / _packed_fused_ok read of q: a CUDA bf16 tensor [1, S, H, d]."""
    shape = (1, S, H, d)
    return types.SimpleNamespace(is_cuda=True, dtype=torch.bfloat16, size=lambda i=None: shape if i is None else shape[i])


@pytest.mark.parametrize("d", [64, 80, 128])
def test_fused_envelope_reaches_65536(d):
    from spt_proto_b200 import layers
    for cls in (layers.SparseVanillaAttentionV2, layers.SparseRotaryAttentionV2):
        attn = cls(d_head=d, d_codeword=8, n_codewords=16, p_dropout=0.0)
        for S, want in ((3840, True), (4224, True), (5376, True), (8192, True), (8576, True), (10752, True),
                        (13312, True), (13440, True), (16384, True), (32768, True), (65536, True), (65536 + 128, False),
                        (131072, False), (16384 + 64, False)):
            assert attn._fused_ok(_fake_q(S, d)) == want, (cls.__name__, d, S)
        for max_seqlen, want in ((5376, True), (5504, True), (13440, True), (16384, True), (65536, True),
                                 (65537, False)):
            assert attn._packed_fused_ok(_fake_q(1024, d), max_seqlen) == want, (cls.__name__, d, max_seqlen)


def test_recompute_threshold_is_8192():
    from spt_proto_b200 import layers
    assert layers.SparseVanillaAttentionV2.recompute_mask_above == 8192
    assert layers.SparseRotaryAttentionV2.recompute_mask_above == 8192


@pytest.mark.parametrize("S", [2049, 4096, 9000])
def test_rotary_extension_equals_a_longer_table(S):
    """Rows >= 2048 equal RotaryEmbedding(n_embeddings=S) bit for bit, rows below are the registered buffers; a long
    forward leaves state_dict's keys, shapes and values as they were."""
    from spt_proto_b200.layers.basic import RotaryAttention, RotaryEmbedding
    d = 64
    attn = RotaryAttention(d_head=d, p_dropout=0.0)
    before = {k: v.clone() for k, v in attn.state_dict().items()}
    ref = RotaryEmbedding(n_embeddings=S, d_model=d)
    cos, sin = attn.embedding.tables(S)
    assert cos.shape == (S, d) and sin.shape == (S, d)
    assert torch.equal(cos[2048:], ref.cos_cached[2048:]) and torch.equal(sin[2048:], ref.sin_cached[2048:])
    assert torch.equal(cos[:2048], attn.embedding.cos_cached) and torch.equal(sin[:2048], attn.embedding.sin_cached)
    g = torch.Generator().manual_seed(S)
    x = torch.randn(1, S, 2, d, generator=g)
    got = attn._rotate(x)
    want = ref(x, ids=torch.arange(S))
    assert torch.equal(got, want)
    # positions below max_length are untouched by the extension
    assert torch.equal(got[:, :2048], attn._rotate(x[:, :2048]))
    after = attn.state_dict()
    assert list(after) == list(before)
    for k, v in before.items():
        assert after[k].shape == v.shape and torch.equal(after[k], v), k
    assert after["embedding.cos_cached"].shape == (2048, d)


def test_rotary_packed_positions_past_max_length():
    """_rotate_packed with max_seqlen > 2048: every sequence rotated as _rotate rotates it alone (CPU tensors; the
    layer computes the positions on the device of cu)."""
    from spt_proto_b200 import layers
    d = 64
    attn = layers.SparseRotaryAttentionV2(d_head=d, p_dropout=0.0, d_codeword=8, n_codewords=16)
    lengths = [3072, 512, 2304]
    cu = torch.tensor([0, 3072, 3584, 5888], dtype=torch.int32)
    x = torch.randn(1, sum(lengths), 2, d, generator=torch.Generator().manual_seed(3))
    got = attn._rotate_packed(x, cu, max(lengths))
    for a, b in zip(cu[:-1].tolist(), cu[1:].tolist()):
        assert torch.equal(got[:, a:b], attn._rotate(x[:, a:b])), (a, b)
