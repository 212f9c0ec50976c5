"""Long sequences on the fused path: the mask-only lookup from S 16384 to 65536 at m 8, 10 and 16 (the streaming kernel),
the attention kernels on its masks, the V2 layers with the mask recomputed in the backward, and the writes of the lookup
staying inside its outputs.

Lookup rows are checked against a row-subset restatement of the oracle's lookup specification (_spec_row), which is pinned
to the C oracle on whole small problems first.  A row depends only on the codes of keys <= r and on nnz, so single rows
of S 65536 cost O(S m) each.  Attention values are checked against a float64 dense reference computed on the GPU in
query-row chunks from the kernels' own mask and extra0."""
import numpy as np
import pytest
import torch

from oracle import spt_oracle as O

DEV = "cuda"
CLAMP = 10.0
gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# lookup rows: the specification of oracle/spt_oracle.py::lookup_spec for one row
# ---------------------------------------------------------------------------------------------------------------------
def _spec_row(qrow, keys, r, nnz):
    """qrow [m], keys [>= r + 1, m] int64 codes (already reduced mod 2^16) -> (selected keys, extra0) of row r."""
    m = qrow.shape[0]
    div, quarter = m // 4, nnz // 4
    cap = [quarter, quarter, quarter - 1, quarter - 1]
    bucket = np.minimum(3, (keys[: r + 1] == qrow[None, :]).sum(-1) // div)
    j = np.arange(r + 1)
    lists = [[j[(j % 4 == t) & (bucket == s)] for s in range(4)] for t in range(4)]
    lim = min(r + 1, nnz)
    selected, filled = [], 0
    for t in range(4):
        chain = []
        for s in (3, 2, 1, 0):
            own = lists[t][s]
            stored = own[: cap[t]].tolist()
            if t < 2 and len(own) >= quarter:
                partner = lists[3 - t][s]
                if len(partner) >= quarter and partner[-1] // 4 > stored[quarter - 1] // 4:
                    stored[quarter - 1] = int(partner[-1])
            chain.extend(stored)
        chain = chain[: len(range(t, lim, 4))]
        selected += chain
        filled += len(chain)
    return selected, nnz - filled


def _words_of(selected, n_words):
    """Selected keys -> lane-major words (uint32 values in int64): word 4 g + t, bit i <=> key 128 g + 4 i + t."""
    w = np.zeros(n_words, dtype=np.int64)
    for j in selected:
        w[4 * (j >> 7) | (j & 3)] |= 1 << ((j & 127) >> 2)
    return w


def _sample_rows(S, seed, groups=4, extra=8):
    """First and last row of the first, second and last 128-row groups and of `groups` seeded ones, plus seeded rows."""
    g = np.random.default_rng(seed)
    G = S // 128
    picked = {0, 1, G - 1} | set(g.integers(0, G, groups).tolist())
    rows = {r for t in picked for r in (128 * t, 128 * t + 127)}
    rows |= set(g.integers(0, S, extra).tolist())
    return sorted(rows)


def _check_rows(mask_rows, extra_rows, q_codes, k_codes, rows, nnz, n_words, what):
    """mask_rows [len(rows), >= n_words] int32, extra_rows [len(rows)]; codes [S, m] int64 (host)."""
    got = mask_rows.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    ext0 = extra_rows.cpu().numpy()
    for i, r in enumerate(rows):
        sel, e0 = _spec_row(q_codes[r], k_codes, r, nnz)
        want = _words_of(sel, n_words)
        assert np.array_equal(got[i, :n_words], want), (what, r)
        assert not got[i, n_words:].any(), (what, r)
        assert int(ext0[i]) == e0, (what, r, int(ext0[i]), e0)


def test_spec_row_matches_the_c_oracle():
    """The row restatement equals the C oracle's literal emulation on every row of small problems, overflowing
    codebooks (c = 1, 2) included."""
    g = torch.Generator().manual_seed(5)
    for S, m, c, coeff in ((512, 8, 16, 8), (512, 16, 2, 8), (384, 10, 1, 4), (640, 16, 16, 32), (256, 8, 2, 16)):
        q, k = (torch.randint(0, c, (1, S, m), generator=g, dtype=torch.int32) for _ in range(2))
        idx = O.lookup_forward(q, k, coeff)[0].numpy()
        qn, kn = q[0].numpy().astype(np.int64), k[0].numpy().astype(np.int64)
        nnz = S // coeff
        for r in range(S):
            sel, e0 = _spec_row(qn[r], kn, r, nnz)
            want = sorted(set(int(x) for x in idx[r] if x != 0) | ({0} if 0 in sel else set()))
            assert sorted(sel) == want, (S, m, c, r)
            assert len(sel) + e0 == nnz, (S, m, c, r)
            assert (idx[r] == 0).sum() == e0 + (1 if 0 in sel else 0), (S, m, c, r)


def _codes(shape, c, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randint(0, c, shape, generator=g, dtype=torch.int32) for _ in range(2))


def _lookup_kernels(fn):
    """Names of the lookup kernels fn() launches (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.name for e in prof.events() if "lookup_" in e.name and "kernel" in e.name})


@gpu
@pytest.mark.parametrize("c", [16, 2, 1])
@pytest.mark.parametrize("m", [8, 10, 16])
@pytest.mark.parametrize("S", [16384, 32768, 65536])
def test_stream_lookup_rows_match_the_spec(S, m, c):
    """Fixed-length mask-only lookup, one head, sparse_coeff 8, n_codewords = c: the streaming kernel runs (and no
    fallback where it does not fit), and sampled rows equal the specification."""
    from spt_proto_b200 import ext
    q, k = _codes((1, S, m), c, S + m + c)
    qd, kd = q.to(DEV), k.to(DEV)
    run = lambda: ext.lookup_mask(qd, kd, 8, n_codewords=c)
    names = _lookup_kernels(run)
    assert any(f"lookup_maskonly_big_kernel<{m}, false, true>" in n for n in names), names
    mask, extra0, _ = run()
    rows = _sample_rows(S, S + m)
    idx = torch.tensor(rows, device=DEV)
    _check_rows(mask[0, idx], extra0[0, idx], q[0].numpy().astype(np.int64), k[0].numpy().astype(np.int64), rows,
                S // 8, S // 32, (S, m, c))


@gpu
@pytest.mark.parametrize("S,m,coeff", [(8192, 16, 8), (12288, 8, 8), (32768, 8, 128), (32768, 16, 128)])
def test_stream_lookup_matches_the_index_kernel(S, m, coeff):
    """Whole masks against the index-emitting bitmap kernel (want_indices=True writes the mask from its own selection)
    where that still fits; d 128 at S 8192 now runs the streaming kernel on the mask-only call."""
    from spt_proto_b200 import ext
    q, k = _codes((2, S, m), 16, S + m + coeff)
    qd, kd = q.to(DEV), k.to(DEV)
    mask, extra0, _ = ext.lookup_mask(qd, kd, coeff)
    mask_i, extra0_i, idx = ext.lookup_mask(qd, kd, coeff, want_indices=True)
    assert idx is not None
    # every bit but key 0's exactly; key 0's multiplicity (its bit + extra0)
    assert torch.equal(mask[..., 1:], mask_i[..., 1:]) and torch.equal(mask[..., 0] & ~1, mask_i[..., 0] & ~1)
    assert torch.equal((mask[..., 0] & 1) + extra0, (mask_i[..., 0] & 1) + extra0_i)
    names = _lookup_kernels(lambda: ext.lookup_mask(qd, kd, coeff))
    if (S, m) == (8192, 16):
        assert any("lookup_maskonly_big_kernel<16, false, true>" in n for n in names), names
    assert torch.equal(ext.lookup_mask(qd, kd, coeff, n_codewords=16)[0], mask)


PACKED = [16384, 4096, 1056]


@gpu
@pytest.mark.parametrize("c", [16, 2])
@pytest.mark.parametrize("m", [8, 10, 16])
def test_stream_lookup_packed(m, c):
    """Packed sequences of 16384, 4096 and 1056 tokens (max_seqlen 16384, two heads): sampled rows of every sequence
    equal the specification; sequences whose length is a multiple of 128 equal the fixed-length lookup alone."""
    from spt_proto_b200 import ext
    H, T = 2, sum(PACKED)
    q, k = _codes((T, H, m), c, 7 * m + c)
    qd, kd = q.to(DEV), k.to(DEV)
    cu_h = [0]
    for n in PACKED:
        cu_h.append(cu_h[-1] + n)
    cu = torch.tensor(cu_h, dtype=torch.int32, device=DEV)
    run = lambda: ext.lookup_mask_varlen(qd, kd, cu, max(PACKED), 8, n_codewords=c)
    names = _lookup_kernels(run)
    assert any(f"lookup_maskonly_big_kernel<{m}, true, true>" in n for n in names), names
    mask, extra0 = run()
    Wm = mask.shape[-1]
    assert Wm == 4 * max(PACKED) // 128
    for i, (a, b) in enumerate(zip(cu_h[:-1], cu_h[1:])):
        S = b - a
        n_words = 4 * ((S + 127) // 128)
        for h in range(H):
            rows = [r for r in _sample_rows(-(-S // 128) * 128, S + h) if r < S]
            idx = torch.tensor([a + r for r in rows], device=DEV)
            _check_rows(mask[h, idx], extra0[h, idx], q[a:b, h].numpy().astype(np.int64),
                        k[a:b, h].numpy().astype(np.int64), rows, S // 8, n_words, (S, h))
        if S % 128 == 0:
            mf, ef, _ = ext.lookup_mask(qd[a:b].unsqueeze(0).contiguous(), kd[a:b].unsqueeze(0).contiguous(), 8)
            assert torch.equal(mask[:, a:b, : S // 32], mf) and not mask[:, a:b, S // 32:].any()
            assert torch.equal(extra0[:, a:b], ef)


# ---------------------------------------------------------------------------------------------------------------------
# float64 dense reference on the GPU, from (mask, extra0): the formulas in the header of attn_tc.cu
# ---------------------------------------------------------------------------------------------------------------------
def _unpack(words):
    """Lane-major words [R, W] -> selection bits [R, 32 W] (float64)."""
    R, W = words.shape
    shifts = torch.arange(32, device=words.device)
    bits = ((words.long() & 0xFFFFFFFF).view(R, W // 4, 4, 1) >> shifts) & 1      # [R, g, t, i]
    return bits.transpose(2, 3).reshape(R, W * 32).double()


def _reference(q, k, v, dy, words, extra0, scale, clamp=CLAMP, chunk=512):
    """One head on the GPU.  q, k, v, dy [S, d]; words [S, S / 32]; extra0 [S] -> y, dq, dk, dv [S, d] float64:
        w[r][j] = bit + (j == 0) extra0[r],  e = w exp(clamp(scale q k^T, -c, c)) [j <= r],  Z = max(sum e, 1e-9),
        y = e V / Z,  dS = (e / Z)(dO V^T - rowsum(dO y)) [|scale s| <= c],  dQ = scale dS K,  dK = scale dS^T Q,
        dV = (e / Z)^T dO."""
    q, k, v, dy = (t.double() for t in (q, k, v, dy))
    S, d = q.shape
    y, dq = torch.empty_like(q), torch.empty_like(q)
    dk, dv = torch.zeros_like(q), torch.zeros_like(q)
    for r0 in range(0, S, chunk):
        r1 = min(S, r0 + chunk)
        n_w = -(-r1 // 128) * 4                         # keys beyond r1 - 1 are above the diagonal of every row here
        w = _unpack(words[r0:r1, :n_w])[:, :r1]
        w[:, 0] += extra0[r0:r1].double()
        w *= torch.arange(r1, device=q.device).unsqueeze(0) <= torch.arange(r0, r1, device=q.device).unsqueeze(1)
        s = scale * (q[r0:r1] @ k[:r1].T)
        e = w * torch.exp(s.clamp(-clamp, clamp))
        p = e / e.sum(1, keepdim=True).clamp_min(1e-9)
        y[r0:r1] = p @ v[:r1]
        ds = p * (dy[r0:r1] @ v[:r1].T - (dy[r0:r1] * y[r0:r1]).sum(1, keepdim=True)) * (s.abs() <= clamp)
        dq[r0:r1] = scale * (ds @ k[:r1])
        dk[:r1] += scale * (ds.T @ q[r0:r1])
        dv[:r1] += p.T @ dy[r0:r1]
    return y, dq, dk, dv


def _heads(t):
    """[N, S, H, d] -> [N * H, S, d]."""
    N, S, H, d = t.shape
    return t.permute(0, 2, 1, 3).reshape(N * H, S, d)


def _y_heads(y, reference_layout):
    N, S, H, d = y.shape
    return y.reshape(N * H, d, S).transpose(1, 2) if reference_layout else _heads(y)


def _dy_memory(dy, reference_layout):
    return _heads(dy).transpose(1, 2).contiguous().view(dy.shape) if reference_layout else dy


def _assert_close(name, got, ref, d):
    """The tolerances of test_fused_attention_matches_oracle."""
    if name == "y":
        assert torch.allclose(got, ref, atol=2e-2, rtol=2e-2), name
    else:
        atol = max(4e-2 if d == 64 else 8e-2, 1.5e-2 * ref.abs().max().item())
        assert torch.allclose(got, ref, atol=atol, rtol=3e-2), (name, (got - ref).abs().max().item())
    err = ((got - ref).norm() / ref.norm()).item()
    assert err < 1e-2, (name, err)


def _check_heads(y, grads, q, k, v, dyh, mask, extra0, scale, reference_layout, heads):
    """dyh: the gradient of y per head [B, S, d]."""
    d = q.shape[-1]
    yh = _y_heads(y, reference_layout)
    qh, kh, vh = (_heads(t) for t in (q, k, v))
    gh = [_heads(t) for t in grads] if grads is not None else None
    for b in heads:
        want = _reference(qh[b], kh[b], vh[b], dyh[b], mask[b], extra0[b], scale)
        _assert_close("y", yh[b].double(), want[0], d)
        if gh is not None:
            for name, g, w in zip(("dq", "dk", "dv"), gh, want[1:]):
                _assert_close(name, g[b].double(), w, d)


def _attn_inputs(N, S, H, d, dtype, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    q, k, v, dy = (torch.randn(N, S, H, d, generator=g, device=DEV).to(dtype) for _ in range(4))
    w = torch.randn(d // 8, 16, 8, generator=g, device=DEV)
    return q, k, v, dy, w


ATTN_CASES = ([(S, d, torch.bfloat16, rl) for S in (16384, 32768) for d in (64, 80, 128) for rl in (False, True)]
              + [(16384, 64, torch.float16, True), (16384, 128, torch.float16, False), (65536, 64, torch.bfloat16, True)])


@gpu
@pytest.mark.parametrize("S,d,dtype,reference_layout", ATTN_CASES)
def test_attention_on_long_masks(S, d, dtype, reference_layout):
    """y, dq, dk, dv of the fused kernels on the streaming lookup's masks against the float64 reference, one sampled
    head of two (all heads at S 65536, which has one)."""
    from spt_proto_b200 import ext
    H = 1 if S == 65536 else 2
    q, k, v, dy, w = _attn_inputs(1, S, H, d, dtype, S + d)
    mask, extra0, _ = ext.lookup_mask(*ext.pq_encode_pair(q, k, w), 8, n_codewords=16)
    scale = d ** -0.5
    y, z = ext.sparse_attn_fwd(q, k, v, mask, extra0, scale, reference_layout=reference_layout)
    grads = ext.sparse_attn_bwd(q, k, v, y, _dy_memory(dy, reference_layout), mask, extra0, z, scale,
                                reference_layout=reference_layout)
    head = int(torch.randint(0, H, (1,), generator=torch.Generator().manual_seed(S + d)))
    _check_heads(y, grads, q, k, v, _heads(dy), mask, extra0, scale, reference_layout, [head])


# ---------------------------------------------------------------------------------------------------------------------
# layers
# ---------------------------------------------------------------------------------------------------------------------
def _layer(cls, d, dtype):
    from spt_proto_b200 import layers
    attn = cls(d_head=d, d_codeword=8, n_codewords=16, p_dropout=0.0).to(DEV)
    if dtype == torch.float16:
        attn = attn.half()
    attn.host_trigger = False
    return attn


@gpu
@pytest.mark.parametrize("kind", ["vanilla", "rotary"])
def test_layers_at_16384(kind):
    """The V2 layers at S 16384, d 128: fused, y against the float64 reference on the mask of the (rotated) operands,
    and (vanilla) gradients too; the recompute path's gradients equal ext.sparse_attn_bwd on the saved-mask inputs bit
    for bit; no mask-sized tensor is saved for the backward."""
    from spt_proto_b200 import ext, layers
    cls = layers.SparseVanillaAttentionV2 if kind == "vanilla" else layers.SparseRotaryAttentionV2
    N, S, H, d = 1, 16384, 2, 128
    attn = _layer(cls, d, torch.bfloat16)
    q, k, v, dy, _ = _attn_inputs(N, S, H, d, torch.bfloat16, 99 + len(kind))
    q, k, v = (t.requires_grad_() for t in (q, k, v))
    saved = []

    def pack(t):
        saved.append(t.numel() * t.element_size())
        return t

    with torch.autograd.graph.saved_tensors_hooks(pack, lambda t: t):
        y = attn(q, k, v)
    assert attn.last_path == "fused"
    mask_bytes = N * H * S * S // 8
    assert saved and max(saved) < mask_bytes // 4, (max(saved), mask_bytes)
    y.backward(dy)

    with torch.no_grad():
        qr, kr = (attn._rotate(t).to(t.dtype) for t in (q, k)) if kind == "rotary" else (q, k)
        qr, kr, vr = qr.contiguous(), kr.contiguous(), v.detach().contiguous()
        mask, extra0, _ = ext.lookup_mask(*ext.pq_encode_pair(qr, kr, attn.quantizer.weight), 8, n_codewords=16)
        y2, z2 = ext.sparse_attn_fwd(qr, kr, vr, mask, extra0, attn.scaling, reference_layout=True)
        assert torch.equal(y.detach(), y2)
        g2 = ext.sparse_attn_bwd(qr, kr, vr, y2, dy.contiguous(), mask, extra0, z2, attn.scaling, reference_layout=True)
    if kind == "vanilla":
        for a, b in zip((q.grad, k.grad, v.grad), g2):
            assert torch.equal(a, b)
        _check_heads(y.detach(), g2, q.detach(), k.detach(), v.detach(), _y_heads(dy, True), mask, extra0, attn.scaling,
                     True, [1])
    else:
        assert torch.equal(v.grad, g2[2])
        _check_heads(y.detach(), None, qr, kr, vr, _y_heads(dy, True), mask, extra0, attn.scaling, True, [0])


@gpu
def test_forward_packed_d128_long():
    """forward_packed at d 128 with max_seqlen 16384 runs fused_packed; each sequence whose length is a multiple of 128
    equals forward() on it alone bit for bit, y and gradients."""
    from spt_proto_b200 import layers
    attn = _layer(layers.SparseVanillaAttentionV2, 128, torch.bfloat16)
    H, T = 2, sum(PACKED)
    g = torch.Generator(device=DEV).manual_seed(4)
    q, k, v, dy = (torch.randn(T, H, 128, generator=g, device=DEV).bfloat16() for _ in range(4))
    q, k, v = (t.requires_grad_() for t in (q, k, v))
    cu_h = [0, 16384, 20480, 21536]
    y = attn.forward_packed(q, k, v, cu_h)
    assert attn.last_path == "fused_packed"
    y.backward(dy)
    for a, b in zip(cu_h[:-1], cu_h[1:]):
        if (b - a) % 128:
            continue
        qs, ks, vs = (t.detach()[a:b].unsqueeze(0).clone().requires_grad_() for t in (q, k, v))
        ys = attn(qs, ks, vs)
        assert attn.last_path == "fused"
        assert torch.equal(ys.detach()[0], y.detach()[a:b]), (a, b)
        # the layer's y memory per sequence is its own [H, d, S] block: feed the matching slice of dy's memory
        dys = dy[a:b].contiguous().unsqueeze(0)
        ys.backward(dys)
        for name, gs, gp in (("dq", qs.grad, q.grad), ("dk", ks.grad, k.grad), ("dv", vs.grad, v.grad)):
            assert torch.equal(gs[0], gp[a:b]), (a, b, name)


@gpu
def test_graph_capture_d128_16384():
    """SparseVanillaAttentionV2 (d 128, S 16384, the recompute path) captured forward + backward: two replays give y
    and the gradients of the eager step bit for bit."""
    from spt_proto_b200 import layers
    torch.manual_seed(21)
    N, S, H, E = 1, 16384, 4, 128
    attn = _layer(layers.SparseVanillaAttentionV2, E, torch.bfloat16)
    q, k, v = (torch.randn(N, S, H, E, device=DEV).bfloat16().requires_grad_() for _ in range(3))
    dy = torch.randn(N, S, H, E, device=DEV).bfloat16()

    def step():
        q.grad = k.grad = v.grad = None
        y = attn(q, k, v)
        y.backward(dy)
        return [y, q.grad, k.grad, v.grad]

    want = [t.detach().clone() for t in step()]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = step()
    assert attn.last_path == "fused"
    for _ in range(2):
        for t in outs:
            t.detach().zero_()
        graph.replay()
        torch.cuda.synchronize()
        for name, a, b in zip(("y", "dq", "dk", "dv"), outs, want):
            assert torch.equal(a.detach(), b), name


# ---------------------------------------------------------------------------------------------------------------------
# writes stay inside mask / extra0
# ---------------------------------------------------------------------------------------------------------------------
GUARD = 4096          # int32 words of sentinel on each side
SENTINEL = 0x5A5A5A5A


def _guarded(n):
    buf = torch.full((GUARD + n + GUARD,), SENTINEL, dtype=torch.int32, device=DEV)
    return buf, buf[GUARD:GUARD + n]


def _guards_intact(buf):
    return bool((buf[:GUARD] == SENTINEL).all()) and bool((buf[-GUARD:] == SENTINEL).all())


def _broken_promise_codes(shape, seed):
    """Codes < 16 with every 7th one replaced by a value in [16, 40): a promise of n_codewords = 16 that is broken."""
    q, k = _codes(shape, 16, seed)
    g = torch.Generator().manual_seed(seed + 1)
    for t in (q, k):
        hit = torch.rand(t.shape, generator=g) < 1 / 7
        t[hit] = torch.randint(16, 40, (int(hit.sum()),), generator=g, dtype=torch.int32)
    return q, k


def _no_match(q, k):
    """What a code >= 16 does without the fallback: it matches no key.  Query codes >= 16 -> -1, key codes -> -2."""
    q, k = q.numpy().astype(np.int64), k.numpy().astype(np.int64)
    return np.where(q >= 16, -1, q), np.where(k >= 16, -2, k)


@gpu
@pytest.mark.parametrize("broken", [False, True])
@pytest.mark.parametrize("m", [8, 16])
def test_stream_writes_stay_inside_fixed(m, broken):
    from spt_proto_b200 import ext
    from spt_proto_b200._lib import check, lib
    B, S, nnz = 2, 32768, 4096
    q, k = _broken_promise_codes((B, S, m), m) if broken else _codes((B, S, m), 16, m)
    qd, kd = q.to(DEV), k.to(DEV)
    mbuf, mask = _guarded(B * S * S // 32)
    ebuf, extra0 = _guarded(B * S)
    ws = ext._workspace(lib.spt_lookup_workspace_bytes(B, S, m, nnz), qd)
    outs = []
    for _ in range(2):
        check(lib.spt_lookup_mask_fwd_ex(qd.data_ptr(), kd.data_ptr(), None, mask.data_ptr(), extra0.data_ptr(),
                                         ws.data_ptr(), B, S, m, nnz, 1, 16, ext._stream(qd)))
        torch.cuda.synchronize()
        assert _guards_intact(mbuf) and _guards_intact(ebuf)
        outs.append((mask.clone(), extra0.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])    # deterministic
    mask, extra0 = mask.view(B, S, S // 32), extra0.view(B, S)
    rows = _sample_rows(S, m, groups=2, extra=4)
    idx = torch.tensor(rows, device=DEV)
    for b in range(B):
        qn, kn = _no_match(q[b], k[b])
        _check_rows(mask[b, idx], extra0[b, idx], qn, kn, rows, nnz, S // 32, (b, broken))


@gpu
@pytest.mark.parametrize("broken", [False, True])
def test_stream_writes_stay_inside_varlen(broken):
    from spt_proto_b200 import ext
    from spt_proto_b200._lib import check, lib
    m, H = 16, 2
    lengths = [32768, 1056, 4096]
    T = sum(lengths)
    cu_h = [0, 32768, 33824, 37920]
    q, k = _broken_promise_codes((T, H, m), 3) if broken else _codes((T, H, m), 16, 3)
    qd, kd = q.to(DEV), k.to(DEV)
    cu = torch.tensor(cu_h, dtype=torch.int32, device=DEV)
    max_s = max(lengths)
    Wm = 4 * max_s // 128
    work = ext.varlen_worklist(cu, T, max_s)
    mbuf, mask = _guarded(H * T * Wm)
    ebuf, extra0 = _guarded(H * T)
    ws = ext._workspace(lib.spt_lookup_mask_varlen_workspace_bytes(len(lengths), T, H, m), qd)
    check(lib.spt_lookup_mask_varlen_fwd_ex(qd.data_ptr(), kd.data_ptr(), work.data_ptr(), mask.data_ptr(),
                                            extra0.data_ptr(), ws.data_ptr(), len(lengths), T, max_s, H, m, 8, 16,
                                            ext._stream(qd)))
    torch.cuda.synchronize()
    assert _guards_intact(mbuf) and _guards_intact(ebuf)
    mask, extra0 = mask.view(H, T, Wm), extra0.view(H, T)
    for a, b in zip(cu_h[:-1], cu_h[1:]):
        S = b - a
        rows = [r for r in _sample_rows(-(-S // 128) * 128, S, groups=2, extra=4) if r < S]
        idx = torch.tensor([a + r for r in rows], device=DEV)
        for h in range(H):
            qn, kn = _no_match(q[a:b, h], k[a:b, h])
            _check_rows(mask[h, idx], extra0[h, idx], qn, kn, rows, S // 8, 4 * ((S + 127) // 128), (S, h, broken))
