"""Head dim 80 (OPT-2.7B: 2560 / 32 heads, PQ 10 subspaces x d_codeword 8) on the fused path: the mask-only lookup at
m = 10, the 128 x 64 attention kernels at D = 80 (padded to 128 in shared memory and TMEM only), the layers, and the
2.7B-shaped routed FFN."""
import os

import pytest
import torch

from oracle import spt_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
E = 80


def _mask_from_indices(indices, S):
    B = indices.shape[0]
    dense = torch.zeros(B, S, S, dtype=torch.int32)
    dense.scatter_add_(2, indices.long(), torch.ones_like(indices))
    # lane-major layout: word 4 g + t, bit i  <=>  key 128 g + 4 i + t
    bits = (dense > 0).view(B, S, S // 128, 32, 4).permute(0, 1, 2, 4, 3).reshape(B, S, S // 32, 32).long()
    words = (bits << torch.arange(32)).sum(-1)
    words = torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32)
    extra0 = dense[:, :, 0] - (dense[:, :, 0] > 0).int()
    assert ((dense[:, :, 1:] <= 1).all())        # only key 0 is ever duplicated (zero padding)
    return words, extra0


def _check_mask(got_mask, got_extra, want_idx, S, coeff):
    """The assertions of test_lookup_mask_matches_index_output: every bit but key 0's exactly, key 0's multiplicity
    (bit + extra0), and rows shorter than the list exactly."""
    want_words, want_extra = _mask_from_indices(want_idx, S)
    got, extra0 = got_mask.cpu(), got_extra.cpu()
    assert torch.equal(got[..., 1:], want_words[..., 1:]) and torch.equal(got[..., 0] & ~1, want_words[..., 0] & ~1)
    assert torch.equal((got[..., 0] & 1) + extra0, (want_words[..., 0] & 1) + want_extra)
    first = min(S, S // coeff)
    assert torch.equal(got[:, :first], want_words[:, :first]) and torch.equal(extra0[:, :first], want_extra[:, :first])


# (2, 512, 4, 8) is the recorded golden's shape; S 2048 runs the plane kernel, S 4096 / 8192 the long-sequence kernel;
# c = 1, 2 overflow the bucket capacities (clobber fix-up)
@pytest.mark.parametrize("B,S,c,coeff", [(2, 512, 4, 8), (2, 2048, 16, 8), (1, 4096, 16, 8), (1, 8192, 16, 32),
                                         (2, 256, 1, 8), (1, 8192, 2, 64)])
def test_lookup_mask_m10_matches_index_output(B, S, c, coeff):
    from spt_proto_b200 import ext
    m = 10
    g = torch.Generator().manual_seed(S + c + m)
    q = torch.randint(0, c, (B, S, m), generator=g, dtype=torch.int32)
    k = torch.randint(0, c, (B, S, m), generator=g, dtype=torch.int32)
    want_idx = O.lookup_forward(q, k, coeff)
    mask, extra0, idx = ext.lookup_mask(q.to(DEV), k.to(DEV), coeff, want_indices=True)
    assert torch.equal(idx.cpu(), want_idx)
    _check_mask(mask, extra0, want_idx, S, coeff)
    # the mask-only kernels (no index output) give the same words
    mask2, extra2, none = ext.lookup_mask(q.to(DEV), k.to(DEV), coeff)
    assert none is None and torch.equal(mask2, mask) and torch.equal(extra2, extra0)


def test_lookup_mask_m10_matches_recorded_reference_kernel():
    """The m = 10 entry of the unmodified reference kernel's recorded output, in mask form, equals the mask-only
    kernel's words."""
    from spt_proto_b200 import ext
    cases = torch.load(os.path.join(os.path.dirname(__file__), "golden", "lookup_ref_kernel_b200.pt"))
    cases = [cs for cs in cases if cs["q"].size(-1) == 10]
    assert cases
    for cs in cases:
        q, k, ref, coeff = cs["q"].int(), cs["k"].int(), cs["ref"].int(), cs["sparse_coeff"]
        S = q.size(1)
        mask, extra0, _ = ext.lookup_mask(q.to(DEV), k.to(DEV), coeff)
        _check_mask(mask, extra0, ref, S, coeff)


def _attn_case(B, S, scale_mul, seed):
    g = torch.Generator().manual_seed(seed)
    q = (torch.randn(B, S, E, generator=g) * scale_mul ** 0.5).bfloat16()
    k = (torch.randn(B, S, E, generator=g) * scale_mul ** 0.5).bfloat16()
    v = torch.randn(B, S, E, generator=g).bfloat16()
    dy = torch.randn(B, S, E, generator=g).bfloat16()
    w = torch.randn(E // 8, 16, 8, generator=g)
    return q, k, v, dy, w


@pytest.mark.parametrize("B,S,scale_mul", [(2, 128, 1.0), (3, 256, 1.0), (2, 256, 6.0), (1, 1024, 1.0), (1, 2048, 1.0),
                                           (1, 2048, 6.0)])
def test_fused_attention_d80_matches_oracle(B, S, scale_mul):
    """As test_fused_attention_matches_oracle, at d = 80; scale_mul = 6 exercises the clamp and its zero gradient.
    The allclose tolerances are those of the d = 128 case."""
    from spt_proto_b200 import ext, kernels
    q, k, v, dy, w = _attn_case(B, S, scale_mul, S + B)
    indptr, indices = O.sparse_attention_indices(q.float(), k.float(), w, 8)
    qf, kf, vf = (t.float().requires_grad_() for t in (q, k, v))
    y_ref, _ = O.sparse_attention_values(indptr, indices, qf, kf, vf, E ** -0.5)
    y_ref.backward(dy.float())

    qd, kd, vd = (t.to(DEV).requires_grad_() for t in (q, k, v))
    q_c, k_c = ext.pq_encode_pair(qd.detach(), kd.detach(), w.to(DEV))
    mask, extra0, idx = ext.lookup_mask(q_c, k_c, 8, want_indices=True)
    assert torch.equal(idx.flatten(1).cpu(), indices)
    y = kernels.sparse_attention(qd, kd, vd, mask, extra0, E ** -0.5)
    y.backward(dy.to(DEV))
    assert torch.allclose(y.float().cpu(), y_ref.detach(), atol=2e-2, rtol=2e-2)
    for got, want in ((vd.grad, vf.grad), (qd.grad, qf.grad), (kd.grad, kf.grad)):
        g_atol = max(8e-2, 1.5e-2 * want.abs().max().item())
        assert torch.allclose(got.float().cpu(), want, atol=g_atol, rtol=3e-2)
    for got, want in ((y, y_ref.detach()), (qd.grad, qf.grad), (kd.grad, kf.grad), (vd.grad, vf.grad)):
        err = (got.float().cpu() - want).norm() / want.norm()
        assert err < 1e-2, err


@pytest.mark.parametrize("reference_layout", [False, True])
def test_fused_d80_interleaved_layout_equals_head_major(reference_layout):
    """[N, S, H, 80] (rows of neighbouring heads 160 bytes apart) gives bit-identical y, dq, dk, dv to the head-major
    call on the same heads: no store of one head touches another head's row."""
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(21)
    N, S, H = 2, 256, 3
    q4, k4, v4, dy4 = (torch.randn(N, S, H, E, generator=g).bfloat16().to(DEV) for _ in range(4))
    w = torch.randn(E // 8, 16, 8, generator=g).to(DEV)
    to_heads = lambda t: t.transpose(1, 2).contiguous().view(N * H, S, -1)
    m4, e4, _ = ext.lookup_mask(*ext.pq_encode_pair(q4, k4, w), 8)
    m3, e3, _ = ext.lookup_mask(to_heads(ext.pq_encode(q4, w)), to_heads(ext.pq_encode(k4, w)), 8)
    assert torch.equal(m4, m3) and torch.equal(e4, e3)
    y4, z4 = ext.sparse_attn_fwd(q4, k4, v4, m4, e4, E ** -0.5, reference_layout=reference_layout)
    y3, z3 = ext.sparse_attn_fwd(to_heads(q4), to_heads(k4), to_heads(v4), m3, e3, E ** -0.5,
                                 reference_layout=reference_layout)
    assert torch.equal(z4, z3)
    if reference_layout:        # the memory of y^T [B, 80, S] either way
        assert torch.equal(y4.reshape(-1), y3.reshape(-1))
        dy3 = dy4.reshape(N * H, S, E)
    else:
        assert torch.equal(to_heads(y4), y3)
        dy3 = to_heads(dy4)
    g4 = ext.sparse_attn_bwd(q4, k4, v4, y4, dy4, m4, e4, z4, E ** -0.5, reference_layout=reference_layout)
    g3 = ext.sparse_attn_bwd(to_heads(q4), to_heads(k4), to_heads(v4), y3, dy3, m3, e3, z3, E ** -0.5,
                             reference_layout=reference_layout)
    for a, b in zip(g4, g3):
        assert torch.equal(to_heads(a), b)


@pytest.mark.parametrize("reference_layout", [False, True])
def test_fused_d80_writes_stay_inside_outputs(reference_layout):
    """Through the C ABI: y, grad_q, grad_k, grad_v sit at the front of larger sentinel-filled buffers and are pre-filled
    with NaN.  After forward and backward every output element is finite (all were written) and every sentinel is
    unchanged (nothing past the last head's 80 columns, or past y^T's 80 feature rows, was written)."""
    from spt_proto_b200 import ext
    from spt_proto_b200._lib import SPT_ATTN_Y_TRANSPOSED, SPT_BF16, check, lib
    g = torch.Generator().manual_seed(33)
    N, S, H = 2, 256, 3
    B = N * H
    q, k, v, dy = (torch.randn(N, S, H, E, generator=g).bfloat16().to(DEV) for _ in range(4))
    w = torch.randn(E // 8, 16, 8, generator=g).to(DEV)
    mask, extra0, _ = ext.lookup_mask(*ext.pq_encode_pair(q, k, w), 8)
    n, tail = q.numel(), 48 * S + 4096
    sentinel = 1536.0                # exactly representable in bf16
    bufs = [torch.full((n + tail,), sentinel, dtype=torch.bfloat16, device=DEV) for _ in range(4)]
    for b in bufs:
        b[:n] = float("nan")
    y, gq, gk, gv = bufs
    zsum = torch.empty(B, S, dtype=torch.float32, device=DEV)
    flags = SPT_ATTN_Y_TRANSPOSED if reference_layout else 0
    st = torch.cuda.current_stream().cuda_stream
    scale = E ** -0.5
    check(lib.spt_sparse_attn_fwd_ex(q.data_ptr(), k.data_ptr(), v.data_ptr(), mask.data_ptr(), extra0.data_ptr(),
                                     y.data_ptr(), zsum.data_ptr(), B, S, E, H, scale, 10.0, SPT_BF16, flags, st))
    ws = torch.empty(lib.spt_sparse_attn_bwd_workspace_bytes(B, S), dtype=torch.uint8, device=DEV)
    check(lib.spt_sparse_attn_bwd_ex(q.data_ptr(), k.data_ptr(), v.data_ptr(), y.data_ptr(), dy.data_ptr(),
                                     mask.data_ptr(), extra0.data_ptr(), zsum.data_ptr(), gq.data_ptr(), gk.data_ptr(),
                                     gv.data_ptr(), ws.data_ptr(), B, S, E, H, scale, 10.0, SPT_BF16, flags, st))
    torch.cuda.synchronize()
    for name, b in zip(("y", "grad_q", "grad_k", "grad_v"), bufs):
        assert torch.isfinite(b[:n].float()).all(), name
        assert (b[n:].float() == sentinel).all(), name
    # and they are the values the torch-facing call computes
    y2, z2 = ext.sparse_attn_fwd(q, k, v, mask, extra0, scale, reference_layout=reference_layout)
    assert torch.equal(y[:n].view_as(q), y2) and torch.equal(zsum, z2)
    for got, want in zip((gq, gk, gv), ext.sparse_attn_bwd(q, k, v, y2, dy, mask, extra0, z2, scale,
                                                           reference_layout=reference_layout)):
        assert torch.equal(got[:n].view_as(q), want)


def _layer_run(attn, q, k, v, dy):
    q.grad = k.grad = v.grad = None
    y = attn(q, k, v)
    y.backward(dy)
    return [t.detach().float().clone() for t in (y, q.grad, k.grad, v.grad)]


def test_vanilla_layer_d80_fused_matches_stage_path():
    """SparseVanillaAttentionV2 at d_head 80 takes the fused path; fused and stage chain (use_fused = False) agree in both
    output layouts."""
    from spt_proto_b200 import layers
    torch.manual_seed(5)
    N, S, H = 2, 256, 4
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0).to(DEV)
    q, k, v = (torch.randn(N, S, H, E, device=DEV).bfloat16().requires_grad_() for _ in range(3))
    dy = torch.randn(N, S, H, E, device=DEV).bfloat16()
    for ref_layout in (True, False):
        attn.reference_output_layout = ref_layout
        out = {}
        for fused in (True, False):
            attn.use_fused = fused
            out[fused] = _layer_run(attn, q, k, v, dy)
            assert attn.last_path == ("fused" if fused else "stage")
        for a, b in zip(out[True], out[False]):
            assert (a - b).norm() / b.norm() < 1.5e-2


def _rope_cpu(x, cos, sin):
    lo, hi = x.chunk(2, dim=-1)
    return x * cos.view(1, -1, 1, x.size(-1)) + torch.cat((-hi, lo), dim=-1) * sin.view(1, -1, 1, x.size(-1))


@pytest.mark.parametrize("reference_layout", [False, True])
def test_rotary_layer_d80_matches_oracle(reference_layout):
    """SparseRotaryAttentionV2 at d_head 80 takes the fused path and matches the oracle layer applied to the rotated
    operands, in both output layouts.  It is compared with the oracle rather than with its own stage chain: the stage
    chain PQ-encodes the fp32 rotation (the reference's dtype promotion) while the fused path encodes the bf16-rounded
    rotation its kernels consume, so the two select different keys wherever a code flips between them."""
    from spt_proto_b200 import layers
    torch.manual_seed(3)
    N, S, H = 2, 256, 4
    attn = layers.SparseRotaryAttentionV2(d_head=E, p_dropout=0.0, d_codeword=8, n_codewords=16,
                                          reference_output_layout=reference_layout).to(DEV)
    q, k, v, dy = (torch.randn(N, S, H, E).bfloat16() for _ in range(4))
    qd, kd, vd = (t.to(DEV).requires_grad_() for t in (q, k, v))
    y = attn(qd, kd, vd)
    assert attn.last_path == "fused"
    y.backward(dy.to(DEV))
    emb = attn.embedding
    cos, sin = emb.cos_cached[:S].float().cpu(), emb.sin_cached[:S].float().cpu()
    qf, kf, vf = (t.float().requires_grad_() for t in (q, k, v))
    qr, kr = _rope_cpu(qf, cos, sin), _rope_cpu(kf, cos, sin)
    qr_b = qr + (qr.detach().bfloat16().float() - qr.detach())     # bf16-rounded, straight-through gradient
    kr_b = kr + (kr.detach().bfloat16().float() - kr.detach())
    y_ref = O.sparse_mha_layer(qr_b, kr_b, vf, attn.quantizer.weight.detach().float().cpu(), 8,
                               reference_output_layout=reference_layout)
    y_ref.backward(dy.float())
    rel = lambda a, b: ((a.float().cpu() - b).norm() / b.norm()).item()
    assert rel(y.detach(), y_ref.detach()) < 1e-2
    assert rel(vd.grad, vf.grad) < 1.5e-2
    assert rel(qd.grad, qf.grad) < 2e-2
    assert rel(kd.grad, kf.grad) < 2e-2


def test_layer_d80_headline_shape_matches_oracle_and_is_deterministic():
    """OPT-2.7B attention at N 1, S 2048, H 32, E 80: forward and backward against the oracle on a subset of heads (heads
    are independent), and two backward passes give bitwise-equal gradients."""
    from spt_proto_b200 import layers
    torch.manual_seed(13)
    N, S, H = 1, 2048, 32
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0,
                                           reference_output_layout=False).to(DEV)
    q, k, v, dy = (torch.randn(N, S, H, E).bfloat16() for _ in range(4))
    qd, kd, vd = (t.to(DEV).requires_grad_() for t in (q, k, v))
    first = _layer_run(attn, qd, kd, vd, dy.to(DEV))
    assert attn.last_path == "fused"
    second = _layer_run(attn, qd, kd, vd, dy.to(DEV))
    for a, b in zip(first, second):
        assert torch.equal(a, b)
    heads = [0, 17, 31]
    sub = lambda t: t[:, :, heads].contiguous()
    qf, kf, vf = (sub(t).float().requires_grad_() for t in (q, k, v))
    y_ref = O.sparse_mha_layer(qf, kf, vf, attn.quantizer.weight.detach().float().cpu(), 8)
    y_ref.backward(sub(dy).float())
    rel = lambda a, b: ((sub(a).cpu() - b).norm() / b.norm()).item()
    y, gq, gk, gv = first
    assert rel(y, y_ref.detach()) < 1e-2
    for got, want in ((gq, qf.grad), (gk, kf.grad), (gv, vf.grad)):
        assert rel(got, want) < 2e-2


def _bf(t):
    return t.bfloat16().float()


def test_routed_ffn_opt27b_shape_matches_oracle():
    """The rest of an OPT-2.7B block: RoutedFFN at d 2560, F 10240, block 2560 (= d_ff / 4, as the adapter sets it), 2048
    tokens, against the oracle (as test_routed_ffn_bench_shape_matches_oracle)."""
    from spt_proto_b200 import layers
    torch.manual_seed(27)
    d, Fdim, bs, T = 2560, 10240, 2560, 2048
    ffn = layers.RoutedFFN(d_model=d, d_feedforward=Fdim, block_size=bs, activation=torch.nn.ReLU()).to(DEV)
    with torch.no_grad():       # router logits are single products: CPU and GPU pick the same blocks
        w = ffn.router[0].weight
        w.zero_()
        for i in range(w.size(0)):
            w[i, i] = 4.0
        ffn.router[0].bias.zero_()
        for p in ffn.parameters():
            p.copy_(_bf(p))
    x = _bf(torch.randn(4, T // 4, d)).to(DEV).requires_grad_()
    y = ffn(x)
    dy = _bf(torch.randn_like(y))
    y.backward(dy)
    sd = {n: t.detach().cpu() for n, t in ffn.state_dict().items()}
    xc = x.detach().cpu().requires_grad_()
    ps = {n: sd[n].clone().requires_grad_() for n in ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias")}
    y_ref = O.routed_ffn(xc, sd["router.0.weight"], sd["router.0.bias"], ps["fc1.weight"], ps["fc1.bias"],
                         ps["fc2.weight"], ps["fc2.bias"], bs, (Fdim // bs) // 2)
    y_ref.backward(dy.cpu())
    rel = lambda a, b: ((a.float().cpu() - b).norm() / b.norm()).item()
    assert rel(y, y_ref.detach()) < 1e-2
    assert rel(x.grad, xc.grad) < 1e-2
    got = dict(ffn.named_parameters())
    for n, p in ps.items():
        assert rel(got[n].grad, p.grad) < 1e-2, (n, rel(got[n].grad, p.grad))
