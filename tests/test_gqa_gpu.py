"""Grouped-query / multi-query attention on the fused path (B200).  The definition: the multi-head call on k and v
repeated G = H / Hkv times along the head axis (torch.repeat_interleave(k, G, 2), HF repeat_kv).  The lookup, y, zsum and
dq equal that call bit for bit; dk and dv equal its dk and dv summed over each group in fp32, g ascending, rounded once."""
import pytest
import torch

from oracle import spt_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rep(x, G):
    return x.repeat_interleave(G, dim=-2)


def _group_sum(x, G):
    """[..., H, d] -> [..., H / G, d]: fp32 sum over each group of G heads, g ascending, one rounding."""
    x = x.view(*x.shape[:-2], x.size(-2) // G, G, x.size(-1))
    acc = x[..., 0, :].float()
    for g in range(1, G):
        acc = acc + x[..., g, :].float()
    return acc.to(x.dtype)


def _codes(shape, n, g):
    return torch.randint(0, n, shape, generator=g, dtype=torch.int32).to(DEV)


# ---- 1. lookup ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m,S,H,Hkv,n_codes,n_codewords", [
    (8, 2048, 4, 2, 16, 16),          # plane kernel
    (10, 2048, 8, 1, 16, 16),         # MQA
    (16, 2048, 32, 4, 16, 16),        # G 8
    (16, 16384, 2, 1, 16, 16),        # long S: the streaming kernel (fallback skipped on the codebook promise)
    (8, 2048, 4, 1, 40, None),        # codes >= 16: the flag-guarded fallback
    (12, 1024, 4, 2, 16, None),       # m outside 8 / 10 / 16: the generic kernel
])
def test_lookup_from_kv_head_codes(m, S, H, Hkv, n_codes, n_codewords):
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(S + H + m)
    N = 2 if S <= 2048 else 1
    qc, kc = _codes((N, S, H, m), n_codes, g), _codes((N, S, Hkv, m), n_codes, g)
    mask, extra0, _ = ext.lookup_mask(qc, kc, 8, n_codewords=n_codewords)
    want_m, want_e, _ = ext.lookup_mask(qc, _rep(kc, H // Hkv).contiguous(), 8, n_codewords=n_codewords)
    assert torch.equal(mask, want_m) and torch.equal(extra0, want_e)


@pytest.mark.parametrize("m,H,Hkv,n_codes", [(8, 4, 2, 16), (16, 8, 1, 16), (10, 4, 1, 40)])
def test_lookup_varlen_from_kv_head_codes(m, H, Hkv, n_codes):
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(7 * m + H)
    cu = torch.tensor([0, 256, 1024, 1536, 2048], dtype=torch.int32, device=DEV)
    qc, kc = _codes((2048, H, m), n_codes, g), _codes((2048, Hkv, m), n_codes, g)
    mask, extra0 = ext.lookup_mask_varlen(qc, kc, cu, 768, 8)
    want_m, want_e = ext.lookup_mask_varlen(qc, _rep(kc, H // Hkv).contiguous(), cu, 768, 8)
    assert torch.equal(mask, want_m) and torch.equal(extra0, want_e)


# ---- 2. fixed-length attention, both output layouts -----------------------------------------------------------------
def _operands(N, S, H, Hkv, d, dtype, g, scale=1.0):
    q = (torch.randn(N, S, H, d, generator=g) * scale).to(dtype)
    k = (torch.randn(N, S, Hkv, d, generator=g) * scale).to(dtype)
    v = torch.randn(N, S, Hkv, d, generator=g).to(dtype)
    dy = torch.randn(N, S, H, d, generator=g).to(dtype)
    w = torch.randn(d // 8, 16, 8, generator=g)
    return q, k, v, dy, w


def _check_against_repeated(got, want, G):
    (y, z, gq, gk, gv), (yr, zr, gqr, gkr, gvr) = got, want
    assert torch.equal(y, yr) and torch.equal(z, zr) and torch.equal(gq, gqr)
    assert torch.equal(gk, _group_sum(gkr, G)) and torch.equal(gv, _group_sum(gvr, G))


def _fused_call(q, k, v, dy, mask, extra0, layout, scale):
    from spt_proto_b200 import ext
    y, z = ext.sparse_attn_fwd(q, k, v, mask, extra0, scale, 10.0, layout)
    gq, gk, gv = ext.sparse_attn_bwd(q, k, v, y, dy, mask, extra0, z, scale, 10.0, layout)
    return y, z, gq, gk, gv


ATTN_CASES = [  # (N, S, H, Hkv, d, dtype): every d, dtype and G in {2, 4, 8} and MQA appear
    (2, 1024, 8, 4, 64, torch.bfloat16),
    (1, 512, 4, 1, 64, torch.float16),
    (1, 512, 8, 2, 80, torch.float16),
    (1, 512, 4, 1, 80, torch.bfloat16),
    (1, 512, 8, 1, 128, torch.bfloat16),
    (1, 512, 16, 2, 128, torch.float16),
]


@pytest.mark.parametrize("layout", [False, True])
@pytest.mark.parametrize("N,S,H,Hkv,d,dtype", ATTN_CASES)
def test_attention_equals_repeated_kv_and_oracle(N, S, H, Hkv, d, dtype, layout):
    from spt_proto_b200 import ext
    G = H // Hkv
    g = torch.Generator().manual_seed(S + H + d)
    q, k, v, dy, w = _operands(N, S, H, Hkv, d, dtype, g)
    qd, kd, vd, dyd, wd = (t.to(DEV) for t in (q, k, v, dy, w))
    mask, extra0, _ = ext.lookup_mask(ext.pq_encode(qd, wd), ext.pq_encode(kd, wd), 8, n_codewords=16)
    scale = d ** -0.5
    got = _fused_call(qd, kd, vd, dyd, mask, extra0, layout, scale)
    want = _fused_call(qd, _rep(kd, G).contiguous(), _rep(vd, G).contiguous(), dyd, mask, extra0, layout, scale)
    _check_against_repeated(got, want, G)
    # the oracle layer (gathered form, fp32) on the repeated operands, within the relative bound smoke() holds the
    # multi-head fused path to
    qf, kf, vf = (t.float().requires_grad_() for t in (q, k, v))
    y_ref = O.sparse_mha_layer(qf, _rep(kf, G), _rep(vf, G), w, 8, reference_output_layout=layout)
    y_ref.backward(dy.float())
    rel = lambda a, b: ((a.float().cpu() - b).norm() / b.norm()).item()
    assert rel(got[0], y_ref.detach()) < 1e-2
    for mine, ref in ((got[2], qf.grad), (got[3], kf.grad), (got[4], vf.grad)):
        assert rel(mine, ref) < 1e-2


# ---- 3. G = 1 through the new entry points ----------------------------------------------------------------------------
@pytest.mark.parametrize("d,dtype", [(64, torch.bfloat16), (80, torch.float16), (128, torch.bfloat16)])
def test_gqa_entry_points_at_g1_equal_the_multi_head_ones(d, dtype):
    from spt_proto_b200 import ext
    from spt_proto_b200._lib import check, lib
    g = torch.Generator().manual_seed(d)
    N, S, H = 2, 512, 4
    q, k, v, dy, w = (t.to(DEV) for t in _operands(N, S, H, H, d, dtype, g))
    qc, kc = ext.pq_encode(q, w), ext.pq_encode(k, w)
    B, nnz, code = N * H, S // 8, ext._ATTN_DTYPES[dtype]
    mask, extra0, _ = ext.lookup_mask(qc, kc, 8, n_codewords=16)              # the GQA entry point, Hkv = H
    mask1, extra1 = torch.empty_like(mask), torch.empty_like(extra0)
    ws = ext._workspace(lib.spt_lookup_workspace_bytes(B, S, qc.size(-1), nnz), q)
    check(lib.spt_lookup_mask_fwd_ex(qc.data_ptr(), kc.data_ptr(), None, mask1.data_ptr(), extra1.data_ptr(), ws.data_ptr(),
                                     B, S, qc.size(-1), nnz, H, 16, ext._stream(q)))
    assert torch.equal(mask, mask1) and torch.equal(extra0, extra1)
    for flags in (0, 1):
        y, z, gq, gk, gv = _fused_call(q, k, v, dy, mask, extra0, bool(flags), 0.125)
        y1, z1 = torch.empty_like(q), torch.empty_like(z)
        check(lib.spt_sparse_attn_fwd_ex(q.data_ptr(), k.data_ptr(), v.data_ptr(), mask.data_ptr(), extra0.data_ptr(),
                                         y1.data_ptr(), z1.data_ptr(), B, S, d, H, 0.125, 10.0, code, flags, ext._stream(q)))
        g1 = [torch.empty_like(q) for _ in range(3)]
        ws = ext._workspace(lib.spt_sparse_attn_bwd_workspace_bytes(B, S), q)
        check(lib.spt_sparse_attn_bwd_ex(q.data_ptr(), k.data_ptr(), v.data_ptr(), y1.data_ptr(), dy.data_ptr(),
                                         mask.data_ptr(), extra0.data_ptr(), z1.data_ptr(), *(t.data_ptr() for t in g1),
                                         ws.data_ptr(), B, S, d, H, 0.125, 10.0, code, flags, ext._stream(q)))
        torch.cuda.synchronize()
        assert torch.equal(y, y1) and torch.equal(z, z1)
        assert all(torch.equal(a, b) for a, b in zip((gq, gk, gv), g1))


# ---- 4. recompute path ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", [False, True])
def test_recompute_path_equals_repeated_kv(layout):
    from spt_proto_b200 import ext, kernels
    N, S, H, Hkv, d, G = 1, 16384, 2, 1, 64, 2
    g = torch.Generator().manual_seed(16384)
    q, k, v, dy, w = (t.to(DEV) for t in _operands(N, S, H, Hkv, d, torch.bfloat16, g))
    qc, kc = ext.pq_encode(q, w), ext.pq_encode(k, w)

    def run(k0, v0, kc0):
        qq, kk, vv = (t.clone().requires_grad_() for t in (q, k0, v0))
        y = kernels.sparse_attention_recompute(qq, kk, vv, qc, kc0, 8, d ** -0.5, reference_layout=layout, n_codewords=16)
        y.backward(dy)
        return y.detach(), qq.grad, kk.grad, vv.grad

    y, gq, gk, gv = run(k, v, kc)
    yr, gqr, gkr, gvr = run(_rep(k, G).contiguous(), _rep(v, G).contiguous(), _rep(kc, G).contiguous())
    assert torch.equal(y, yr) and torch.equal(gq, gqr)
    assert torch.equal(gk, _group_sum(gkr, G)) and torch.equal(gv, _group_sum(gvr, G))


# ---- 5. packed batches ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", [False, True])
@pytest.mark.parametrize("H,Hkv,d,dtype", [(4, 2, 80, torch.float16), (8, 1, 128, torch.bfloat16), (8, 2, 64, torch.bfloat16)])
def test_varlen_equals_repeated_kv(H, Hkv, d, dtype, layout):
    from spt_proto_b200 import ext, kernels
    G = H // Hkv
    g = torch.Generator().manual_seed(H * d)
    cu = torch.tensor([0, 256, 1024, 1536, 2048], dtype=torch.int32, device=DEV)
    q, k, v, dy, w = (t.to(DEV) for t in _operands(1, 2048, H, Hkv, d, dtype, g))
    q, k, v, dy = q[0], k[0], v[0], dy[0]
    mask, extra0 = ext.lookup_mask_varlen(ext.pq_encode(q, w), ext.pq_encode(k, w), cu, 768, 8, n_codewords=16)

    def run(k0, v0):
        qq, kk, vv = (t.clone().requires_grad_() for t in (q, k0, v0))
        y = kernels.sparse_attention_varlen(qq, kk, vv, mask, extra0, cu, 768, d ** -0.5, reference_layout=layout)
        y.backward(dy)
        return y.detach(), qq.grad, kk.grad, vv.grad

    y, gq, gk, gv = run(k, v)
    yr, gqr, gkr, gvr = run(_rep(k, G).contiguous(), _rep(v, G).contiguous())
    assert torch.equal(y, yr) and torch.equal(gq, gqr)
    assert torch.equal(gk, _group_sum(gkr, G)) and torch.equal(gv, _group_sum(gvr, G))


# ---- 6. persistent d 64 kernels past one scheduling round -------------------------------------------------------------
def test_persistent_d64_kernels_past_one_round():
    """N 8, H 32, Hkv 8, S 2048: 4096 (head, tile) items per 128 x 128 kernel, many rounds of the persistent grid."""
    from spt_proto_b200 import ext
    N, S, H, Hkv, d, G = 8, 2048, 32, 8, 64, 4
    g = torch.Generator().manual_seed(2048)
    q, k, v, dy, w = (t.to(DEV) for t in _operands(N, S, H, Hkv, d, torch.bfloat16, g))
    mask, extra0, _ = ext.lookup_mask(ext.pq_encode(q, w), ext.pq_encode(k, w), 8, n_codewords=16)
    got = _fused_call(q, k, v, dy, mask, extra0, True, 0.125)
    want = _fused_call(q, _rep(k, G).contiguous(), _rep(v, G).contiguous(), dy, mask, extra0, True, 0.125)
    _check_against_repeated(got, want, G)


# ---- 7. layers --------------------------------------------------------------------------------------------------------
def _layer_step(attn, q, k, v, dy, packed):
    qq, kk, vv = (t.clone().requires_grad_() for t in (q, k, v))
    attn.host_trigger = True
    y = attn.forward_packed(qq, kk, vv, [0, 256, 768, 1024]) if packed else attn(qq, kk, vv)
    y.backward(dy)
    return y.detach(), qq.grad, kk.grad, vv.grad, attn.loss.item(), attn.last_path


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("cls", ["SparseVanillaAttentionV2", "SparseRotaryAttentionV2"])
def test_layers_equal_repeated_kv(cls, packed, fused):
    from spt_proto_b200 import layers
    N, S, H, Hkv, E = (1, 1024, 8, 2, 64) if packed else (2, 512, 8, 4, 64)
    G = H // Hkv
    dtype = torch.bfloat16 if fused else torch.float32
    attn = getattr(layers, cls)(d_head=E, p_dropout=0.0, d_codeword=8, n_codewords=16).to(DEV)
    attn.use_fused = fused
    g = torch.Generator().manual_seed(N * S + H + fused)
    q, k, v, dy, _ = (t.to(DEV) for t in _operands(N, S, H, Hkv, E, dtype, g))
    y, gq, gk, gv, loss, path = _layer_step(attn, q, k, v, dy, packed)
    yr, gqr, gkr, gvr, loss_r, path_r = _layer_step(attn, q, _rep(k, G).contiguous(), _rep(v, G).contiguous(), dy, packed)
    assert path == path_r == ({True: "fused_packed", False: "per_sequence"}[fused] if packed else
                              {True: "fused", False: "stage"}[fused])
    assert torch.equal(y, yr) and torch.equal(gq, gqr)
    if fused and cls == "SparseRotaryAttentionV2":
        # k's gradient passes the rotation backward after the group sum here, before it on the repeated k: the same
        # linear map applied to the sum or to each term, so equal up to the bf16 rounding of the rotated gradients
        assert torch.equal(gv, _group_sum(gvr, G))
        want = _group_sum(gkr, G).float()
        torch.testing.assert_close(gk.float(), want, rtol=2e-2, atol=2e-2 * want.abs().max().item())
    elif fused:
        assert torch.equal(gk, _group_sum(gkr, G)) and torch.equal(gv, _group_sum(gvr, G))
    else:   # the stage path repeats k, v under autograd: the group sum is autograd's (fp32 operands, reordered sum)
        torch.testing.assert_close(gk, _group_sum(gkr, G), rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(gv, _group_sum(gvr, G), rtol=1e-5, atol=1e-6)
    assert loss == pytest.approx(loss_r, rel=1e-5)     # a mean over duplicated rows is the same mean


# ---- 8. graph capture -------------------------------------------------------------------------------------------------
def test_graph_capture_replays_equal_to_eager():
    from spt_proto_b200 import ext, kernels
    N, S, H, Hkv, d, G = 1, 1024, 8, 2, 128, 4
    g = torch.Generator().manual_seed(99)
    q, k, v, dy, w = (t.to(DEV) for t in _operands(N, S, H, Hkv, d, torch.bfloat16, g))
    qq, kk, vv = (t.clone().requires_grad_() for t in (q, k, v))

    def step():
        for t in (qq, kk, vv):
            t.grad = None
        mask, extra0, _ = ext.lookup_mask(ext.pq_encode(qq.detach(), w), ext.pq_encode(kk.detach(), w), 8, n_codewords=16)
        y = kernels.sparse_attention(qq, kk, vv, mask, extra0, d ** -0.5, reference_layout=True)
        y.backward(dy)
        return y.detach()

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = [step().clone()] + [t.grad.clone() for t in (qq, kk, vv)]
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        y_static = step()
    g_static = [t.grad for t in (qq, kk, vv)]
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(y_static, eager[0])
    assert all(torch.equal(a, b) for a, b in zip(g_static, eager[1:]))
    assert g_static[1].shape == k.shape
