"""The fused attention kernels past one scheduling round, at long sequences, on masks at the edges of what the lookup
emits, and under CUDA graph capture.

At head dim 64 the backward runs on persistent grids (`attn_tc128.cu`): G = min(items, SMs) CTAs walk the items
(key or query tile, head) round by round, round w taking items [w G, (w + 1) G), odd rounds in reversed CTA order.  A
CTA's second and later items reuse state of the earlier ones (owner double buffer and its parity, the accumulator
hand-off, the running stage counter, the prefetch of the next owner tiles), so the shapes here are derived from the
device's SM count to put CTAs on a second and third item.

The reference is a float64 dense computation from the kernels' own inputs (the lane-major mask words and extra0), in
query-row chunks: it fits S 8192 where the gathered fp32 oracle does not.  Its CPU test pins it to the oracle's
autograd formulation."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import spt_oracle as O

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLAMP = 10.0
gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# mask words <-> dense selections
# ---------------------------------------------------------------------------------------------------------------------
def _pack(sel):
    """Boolean selection [R, S] -> lane-major words [R, S / 32] int32: word 4 g + t, bit i <=> key 128 g + 4 i + t."""
    R, S = sel.shape
    bits = sel.view(R, S // 128, 32, 4).transpose(2, 3).long()          # [R, g, t, i]
    words = (bits << torch.arange(32)).sum(-1).view(R, S // 32)
    return torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32)


def _unpack(words):
    """Lane-major words [R, S / 32] -> selection bits [R, S] int64 (the inverse of _pack)."""
    R, W = words.shape
    bits = ((words.long() & 0xFFFFFFFF).view(R, W // 4, 4, 1) >> torch.arange(32)) & 1   # [R, g, t, i]
    return bits.transpose(2, 3).reshape(R, W * 32)


def _mask_from_indices(indices, S, chunk=1024):
    """Index lists [B, S, nnz] -> (words [B, S, S / 32], extra0 [B, S]): key 0's multiplicity beyond its bit is the zero
    padding.  Built in row chunks, so that S 8192 stays small."""
    B = indices.shape[0]
    words = torch.empty(B, S, S // 32, dtype=torch.int32)
    extra0 = torch.empty(B, S, dtype=torch.int32)
    for b in range(B):
        for r0 in range(0, S, chunk):
            idx = indices[b, r0:r0 + chunk].long()
            dense = torch.zeros(idx.shape[0], S, dtype=torch.int32).scatter_add_(1, idx, torch.ones_like(idx, dtype=torch.int32))
            assert (dense[:, 1:] <= 1).all()         # only key 0 is ever duplicated (zero padding)
            words[b, r0:r0 + chunk] = _pack(dense > 0)
            extra0[b, r0:r0 + chunk] = dense[:, 0] - (dense[:, 0] > 0).int()
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


def _assert_causal(words, chunk=1024):
    """The lookup's contract, which the kernels rely on (they carry no causal term): no bit above the diagonal."""
    B, S, _ = words.shape
    for b in range(B):
        for r0 in range(0, S, chunk):
            bits = _unpack(words[b, r0:r0 + chunk])
            rows = torch.arange(r0, r0 + bits.shape[0]).unsqueeze(1)
            assert not (bits.bool() & (torch.arange(S).unsqueeze(0) > rows)).any(), (b, r0)


# ---------------------------------------------------------------------------------------------------------------------
# float64 dense reference from (mask, extra0): the formulas in the header of attn_tc.cu
# ---------------------------------------------------------------------------------------------------------------------
def _reference(q, k, v, dy, words, extra0, scale, clamp=CLAMP, chunk=512):
    """One head.  q, k, v, dy [S, d]; words [S, S / 32] int32; extra0 [S].  In float64, rows in chunks:
        w[r][j] = bit + (j == 0) extra0[r],  e = w exp(clamp(scale q k^T, -c, c)) [j <= r],  Z = max(sum e, 1e-9),
        y = e V / Z,  dP = dO V^T,  dS = (e / Z)(dP - rowsum(dO y)) [|scale s| <= c],
        dQ = scale dS K,  dK = scale dS^T Q,  dV = (e / Z)^T dO.
    -> y, dq, dk, dv [S, d] float64."""
    q, k, v, dy = (t.double().cpu() for t in (q, k, v, dy))
    words, extra0 = words.cpu(), extra0.cpu()
    S, d = q.shape
    y, dq = torch.empty(S, d, dtype=torch.float64), torch.empty(S, d, dtype=torch.float64)
    dk, dv = torch.zeros(S, d, dtype=torch.float64), torch.zeros(S, d, dtype=torch.float64)
    for r0 in range(0, S, chunk):
        r1 = min(S, r0 + chunk)                      # keys beyond r1 - 1 are above the diagonal of every row here
        w = _unpack(words[r0:r1])[:, :r1].double()
        w[:, 0] += extra0[r0:r1].double()
        w *= torch.arange(r1).unsqueeze(0) <= torch.arange(r0, r1).unsqueeze(1)
        s = scale * (q[r0:r1] @ k[:r1].T)
        e = w * torch.exp(s.clamp(-clamp, clamp))
        p = e / e.sum(1, keepdim=True).clamp_min(1e-9)
        y[r0:r1] = p @ v[:r1]
        ds = p * (dy[r0:r1] @ v[:r1].T - (dy[r0:r1] * y[r0:r1]).sum(1, keepdim=True)) * (s.abs() <= clamp)
        dq[r0:r1] = scale * (ds @ k[:r1])
        dk[:r1] += scale * (ds.T @ q[r0:r1])
        dv[:r1] += p.T @ dy[r0:r1]
    return y, dq, dk, dv


@pytest.mark.parametrize("case", ["normal", "clamp", "overflow_c1", "overflow_c2"])
def test_reference_matches_oracle_autograd(case):
    """The chunked float64 reference equals O.sparse_attention_values + autograd (run in float64) on masks built from
    O.lookup_forward's index lists.  'clamp' multiplies the scale by 6, so that scores pass +-10; the overflow cases feed
    codes with c = 1, 2 distinct values, whose buckets overflow: extra0 > 0 then appears outside the first S / coeff
    rows."""
    B, S, d = 2, 384, 64
    coeff = 32 if case == "overflow_c2" else 8          # c = 2 leaves padding only where the list is short against S
    g = torch.Generator().manual_seed(77)
    q, k, v, dy = (torch.randn(B, S, d, generator=g, dtype=torch.float64) for _ in range(4))
    scale = d ** -0.5 * (6.0 if case == "clamp" else 1.0)
    if case.startswith("overflow"):
        c = int(case[-1])
        q_c, k_c = (torch.randint(0, c, (B, S, d // 8), generator=g, dtype=torch.int32) for _ in range(2))
    else:
        w = torch.randn(d // 8, 16, 8, generator=g)
        q_c, k_c = O.pq_encode(q.float(), w), O.pq_encode(k.float(), w)
    idx = O.lookup_forward(q_c, k_c, coeff)
    words, extra0 = _mask_from_indices(idx, S)
    if case.startswith("overflow"):
        assert (extra0[:, S // coeff:] > 0).any()
    if case == "clamp":
        assert (scale * (q @ k.transpose(1, 2))).abs().max() > 2 * CLAMP
    qf, kf, vf = (t.clone().requires_grad_() for t in (q, k, v))
    y_want, _ = O.sparse_attention_values(O.fixed_indptr(S, S // coeff), idx.flatten(1), qf, kf, vf, scale)
    y_want.backward(dy)
    for b in range(B):
        got = _reference(q[b], k[b], v[b], dy[b], words[b], extra0[b], scale, chunk=160)   # chunks cross the tiles
        for a, want in zip(got, (y_want[b].detach(), qf.grad[b], kf.grad[b], vf.grad[b])):
            assert ((a - want).norm() / want.norm()).item() < 1e-10
            assert torch.allclose(a, want, rtol=1e-10, atol=1e-10 * want.abs().max().item())


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count     # what num_sms() reads


def _split(B):
    """B heads as (N, H) with H > 1 where B has a small factor (the interleaved layout), else (B, 1)."""
    for H in (4, 3, 2):
        if B % H == 0:
            return B // H, H
    return B, 1


def _cta_of(item, G):
    """Mirror of sched_item: (CTA, round) that runs `item` on a grid of G CTAs."""
    w, pos = divmod(item, G)
    return (G - 1 - pos if w & 1 else pos), w


def _edge_heads(S, B, G, n_sample=4, seed=0):
    """Heads whose items CTA 0 and CTA G - 1 run in the first, second and last rounds of the dK/dV and dQ grids, plus a
    seeded sample of the others.  Items are (tile, head) with the head fastest, so one rule covers both kernels."""
    items = (S // 128) * B
    G = min(G, items)
    rounds = -(-items // G)
    heads = set()
    for w in sorted({0, 1, rounds - 1}):
        for cta in (0, G - 1):
            item = w * G + (G - 1 - cta if w & 1 else cta)
            if item < items:
                assert _cta_of(item, G) == (cta, w)
                heads.add(item % B)
    rest = [b for b in range(B) if b not in heads]
    g = torch.Generator().manual_seed(seed)
    heads.update(rest[i] for i in torch.randperm(len(rest), generator=g)[:n_sample].tolist())
    return sorted(heads)


def _case_shape(case, G):
    """(S, B) of the multi-round cases, derived from the SM count G (items = S / 128 x B)."""
    return {
        "items_G-1": (128, G - 1),                       # one item per CTA, one CTA idle
        "items_G": (128, G),                             # exactly one full round
        "items_G+1": (128, G + 1),                       # CTA G - 1 takes a second item, in the reversed round
        "items_2G+1": (128, 2 * G + 1),                  # a third, non-reversed round
        "s1024_3rounds": (1024, -(-2 * G // 8) + 1),     # items 2G < 8B: a CTA's items have different tile counts
        "s2048_5rounds": (2048, -(-4 * G // 16) + 1),    # items 4G < 16B
    }[case]


CASES = ["items_G-1", "items_G", "items_G+1", "items_2G+1", "s1024_3rounds", "s2048_5rounds"]


def _inputs(N, S, H, d, seed):
    g = torch.Generator().manual_seed(seed)
    q, k, v, dy = (torch.randn(N, S, H, d, generator=g).bfloat16() for _ in range(4))
    w = torch.randn(d // 8, 16, 8, generator=g)
    return q, k, v, dy, w


def _heads(t):
    """[N, S, H, d] -> [N * H, S, d] (head b = n H + h)."""
    N, S, H, d = t.shape
    return t.permute(0, 2, 1, 3).reshape(N * H, S, d)


def _dy_memory(dy, reference_layout):
    """grad_y as the backward reads it: with reference_layout its memory is dy^T [B, d, S] per head."""
    if not reference_layout:
        return dy
    return _heads(dy).transpose(1, 2).contiguous().view(dy.shape)


def _y_heads(y, reference_layout):
    N, S, H, d = y.shape
    return y.reshape(N * H, d, S).transpose(1, 2) if reference_layout else _heads(y)


def _run(q, k, v, dy_mem, mask, extra0, scale, reference_layout):
    from spt_proto_b200 import ext
    y, z = ext.sparse_attn_fwd(q, k, v, mask, extra0, scale, reference_layout=reference_layout)
    gq, gk, gv = ext.sparse_attn_bwd(q, k, v, y, dy_mem, mask, extra0, z, scale, reference_layout=reference_layout)
    return y, z, gq, gk, gv


def _assert_matches_reference(out, q, k, v, dy, mask, extra0, scale, reference_layout, heads):
    """y, dq, dk, dv of `heads` against the float64 reference with the tolerances of test_fused_attention_matches_oracle:
    allclose (y: 2e-2 / 2e-2; gradients: rtol 3e-2, atol 1.5 % of the largest entry, at least 4e-2 at d 64 and 8e-2
    above) and relative Frobenius error < 1e-2."""
    y, _, gq, gk, gv = out
    d = q.shape[-1]
    got_all = [_y_heads(y, reference_layout).cpu()] + [_heads(t).cpu() for t in (gq, gk, gv)]
    qh, kh, vh, dyh = (_heads(t) for t in (q, k, v, dy))
    mask, extra0 = mask.cpu(), extra0.cpu()
    for b in heads:
        want = _reference(qh[b], kh[b], vh[b], dyh[b], mask[b], extra0[b], scale)
        for name, got, ref in zip(("y", "dq", "dk", "dv"), (t[b].double() for t in got_all), want):
            if name == "y":
                assert torch.allclose(got, ref, atol=2e-2, rtol=2e-2), (b, name)
            else:
                atol = max(4e-2 if d == 64 else 8e-2, 1.5e-2 * ref.abs().max().item())
                assert torch.allclose(got, ref, atol=atol, rtol=3e-2), (b, name, (got - ref).abs().max().item())
            err = ((got - ref).norm() / ref.norm()).item()
            assert err < 1e-2, (b, name, err)


def _lookup_case(case, seed=1):
    """Inputs of a multi-round case in [N, S, H, 64] and the lookup's mask on them."""
    from spt_proto_b200 import ext
    S, B = _case_shape(case, _num_sms())
    N, H = _split(B)
    q, k, v, dy, w = _inputs(N, S, H, 64, seed + S + B)
    qd, kd = q.to(DEV), k.to(DEV)
    mask, extra0, _ = ext.lookup_mask(*ext.pq_encode_pair(qd, kd, w.to(DEV)), 8)
    return q, k, v, dy, mask, extra0


@gpu
@pytest.mark.parametrize("reference_layout", [False, True])
@pytest.mark.parametrize("case", CASES)
def test_multi_round_parity(case, reference_layout):
    """d 64, the default kernels: y, dq, dk, dv against the float64 reference.  Every head where S <= 1024; at S 2048 the
    heads of CTA 0 and CTA G - 1 in the first, second and last rounds plus a seeded sample."""
    q, k, v, dy, mask, extra0 = _lookup_case(case)
    S, B = q.shape[1], q.shape[0] * q.shape[2]
    scale = 64 ** -0.5
    out = _run(q.to(DEV), k.to(DEV), v.to(DEV), _dy_memory(dy, reference_layout).to(DEV), mask, extra0, scale,
               reference_layout)
    heads = range(B) if S <= 1024 else _edge_heads(S, B, _num_sms())
    _assert_matches_reference(out, q, k, v, dy, mask, extra0, scale, reference_layout, heads)


def _assert_batch_invariant(q, k, v, dy_mem, mask, extra0, scale, reference_layout):
    """Every head of the batched call equals the same head called alone (B = 1: one item per CTA), bit for bit.  An item's
    instructions and accumulation order do not depend on the CTA that runs it or on what that CTA ran before, and there
    are no atomics, so any state leaking from one item into the next shows here exactly."""
    N, S, H, d = q.shape
    B = N * H
    out = _run(q, k, v, dy_mem, mask, extra0, scale, reference_layout)
    y, z, gq, gk, gv = out
    for b in range(B):
        n, h = divmod(b, H)
        one = lambda t: t[n, :, h].contiguous().view(1, S, d)
        dy1 = dy_mem.reshape(B, d, S)[b].contiguous().view(1, S, d) if reference_layout else one(dy_mem)
        y1, z1, gq1, gk1, gv1 = _run(one(q), one(k), one(v), dy1, mask[b:b + 1], extra0[b:b + 1], scale, reference_layout)
        y_b = y.reshape(B, d, S)[b] if reference_layout else y[n, :, h]
        assert torch.equal(y1.reshape(y_b.shape), y_b), (b, "y")
        assert torch.equal(z1[0], z[b]), (b, "zsum")
        for name, a, t in (("dq", gq1, gq), ("dk", gk1, gk), ("dv", gv1, gv)):
            assert torch.equal(a[0], t[n, :, h]), (b, name)


@gpu
@pytest.mark.parametrize("reference_layout", [False, True])
@pytest.mark.parametrize("case", CASES + ["bench_shape"])
def test_batch_invariance(case, reference_layout):
    """y, zsum, dq, dk, dv of each head: batched call == the head alone, bit for bit.  bench_shape is bench.py's step
    (4 x 32 heads, S 2048: 2048 items)."""
    from spt_proto_b200 import ext
    if case == "bench_shape":
        q, k, v, dy, w = _inputs(4, 2048, 32, 64, 123)
        mask, extra0, _ = ext.lookup_mask(*ext.pq_encode_pair(q.to(DEV), k.to(DEV), w.to(DEV)), 8)
    else:
        q, k, v, dy, mask, extra0 = _lookup_case(case)
    _assert_batch_invariant(q.to(DEV), k.to(DEV), v.to(DEV), _dy_memory(dy, reference_layout).to(DEV), mask, extra0,
                            64 ** -0.5, reference_layout)


# ---------------------------------------------------------------------------------------------------------------------
# long sequences
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("S,d", [(4096, 64), (8192, 64), (4096, 128), (8192, 128), (4096, 80)])
def test_long_sequence_matches_reference(S, d):
    """S 4096 / 8192 at top-k S / 8 (1024 keys per row at S 8192): first the mask-only lookup against O.lookup_forward on
    the same codes, then y, dq, dk, dv against the float64 reference.  Two heads at S 4096 (interleaved), one at 8192."""
    from spt_proto_b200 import ext
    N, H, coeff = 1, (2 if S == 4096 else 1), 8
    q, k, v, dy, w = _inputs(N, S, H, d, S + d)
    q_c, k_c = ext.pq_encode_pair(q.to(DEV), k.to(DEV), w.to(DEV))
    mask, extra0, none = ext.lookup_mask(q_c, k_c, coeff)
    assert none is None
    want_idx = O.lookup_forward(_heads(q_c.cpu()), _heads(k_c.cpu()), coeff)
    _check_mask(mask, extra0, want_idx, S, coeff)
    del want_idx
    scale = d ** -0.5
    out = _run(q.to(DEV), k.to(DEV), v.to(DEV), dy.to(DEV), mask, extra0, scale, False)
    _assert_matches_reference(out, q, k, v, dy, mask, extra0, scale, False, range(N * H))


# ---------------------------------------------------------------------------------------------------------------------
# masks at the edges of what the lookup emits
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("kind", ["codes_c1", "codes_c2", "full_causal", "key0_only_rows", "unselected_group"])
def test_edge_masks_multi_round(kind):
    """At S 1024, with three rounds of the persistent grids:
    codes_c*: codes with 1 or 2 distinct values fed straight to the lookup; buckets overflow and leave zero padding in
        rows outside the first S / coeff.  With c = 1 (top-k S / 8) such rows lie in query tiles j > 0 of the key-0
        items, where the dK/dV kernel takes its `pad` variant; c = 2 leaves padding only at top-k S / 128;
    full_causal: every key at or below the diagonal;
    key0_only_rows: one row in 32 (four in every query tile) selects key 0 alone, with extra0 = S / coeff - 1.  Such a
        row's dS is zero in exact arithmetic; the kernels' bf16 dO' = dO / Z leaves a rounding residue of about
        2^-9 |dO'| |v_0| sqrt(d) there, and every such row adds its residue into row 0 of dK.  One row in three would
        make that sum alone larger than the shared atol at this size;
    unselected_group: no row selects keys 128 .. 255; their dK and dV are exactly zero."""
    from spt_proto_b200 import ext
    G = _num_sms()
    S, B = _case_shape("s1024_3rounds", G)
    N, H = _split(B)
    coeff = 128 if kind == "codes_c2" else 8
    q, k, v, dy, w = _inputs(N, S, H, 64, 500 + len(kind))
    qd, kd = q.to(DEV), k.to(DEV)
    if kind.startswith("codes"):
        g = torch.Generator().manual_seed(int(kind[-1]))
        q_c, k_c = (torch.randint(0, int(kind[-1]), (N, S, H, 8), generator=g, dtype=torch.int32).to(DEV) for _ in range(2))
    else:
        q_c, k_c = ext.pq_encode_pair(qd, kd, w.to(DEV))
    mask, extra0, _ = ext.lookup_mask(q_c, k_c, coeff)
    if kind.startswith("codes"):
        assert (extra0[:, S // coeff:] > 0).any()       # padding outside the rows shorter than the list
        if kind == "codes_c1":
            assert (extra0[:, 128:] > 0).any()
    elif kind == "full_causal":
        causal = torch.arange(S).unsqueeze(0) <= torch.arange(S).unsqueeze(1)
        mask = _pack(causal).unsqueeze(0).expand(B, -1, -1).contiguous().to(DEV)
        extra0 = torch.zeros(B, S, dtype=torch.int32, device=DEV)
    elif kind == "key0_only_rows":
        rows = torch.arange(5, S, 32, device=DEV)
        mask[:, rows] = 0
        mask[:, rows, 0] = 1
        extra0[:, rows] = S // coeff - 1
    else:
        mask[:, :, 4:8] = 0
    _assert_causal(mask.cpu())
    heads = set(_edge_heads(S, B, G, seed=7))
    heads.update((extra0[:, S // coeff:] > 0).any(1).nonzero().flatten().tolist()[:4])    # heads with late padding
    scale = 64 ** -0.5
    for reference_layout in (False, True):
        out = _run(qd, kd, v.to(DEV), _dy_memory(dy, reference_layout).to(DEV), mask, extra0, scale, reference_layout)
        _assert_matches_reference(out, q, k, v, dy, mask, extra0, scale, reference_layout, sorted(heads))
        if kind == "unselected_group":
            for t in out[3:]:
                assert torch.equal(t[:, 128:256], torch.zeros_like(t[:, 128:256]))


# ---------------------------------------------------------------------------------------------------------------------
# run-time switches (read once per process): child processes
# ---------------------------------------------------------------------------------------------------------------------
def _child_pytest(env_extra, expr):
    env = dict(os.environ, **env_extra)
    res = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", os.path.abspath(__file__), "-k", expr],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert " passed" in res.stdout and "failed" not in res.stdout


@gpu
@pytest.mark.parametrize("switch", ["SPT_ATTN_TILE=64"])
def test_switch_parity_and_batch_invariance(switch):
    """SPT_ATTN_TILE=64 (128 x 64-tile backward) is documented to give the same results: the multi-round parity and the
    bit-exact batch invariance hold under it."""
    name, value = switch.split("=")
    _child_pytest({name: value}, "test_multi_round_parity or test_batch_invariance")


# ---------------------------------------------------------------------------------------------------------------------
# CUDA graph capture of the d 64 layer
# ---------------------------------------------------------------------------------------------------------------------
def _graph_replay_equals_eager(first_backward_in_capture=False, dtype=torch.bfloat16, seed=17):
    """SparseVanillaAttentionV2 (d 64, fused, N 1, S 2048, G / 16 + 2 heads: two rounds) captured forward + backward
    with torch.cuda.graph; two replays give y and the three gradients of the eager step bit for bit.
    first_backward_in_capture: the capture holds the process's first backward, so the launcher cannot create its side
    stream (no stream or event creation during a capture) and runs the dK/dV and dQ kernels one after the other.
    dtype: of q, k, v; float16 also converts the layer with .half()."""
    from spt_proto_b200 import layers
    torch.manual_seed(seed)
    N, S, H, E = 1, 2048, _num_sms() // 16 + 2, 64
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0).to(DEV)
    if dtype == torch.float16:
        attn = attn.half()
    attn.host_trigger = False                          # no device -> host read of the PQ-loss trigger inside the capture
    q, k, v = (torch.randn(N, S, H, E, device=DEV).to(dtype).requires_grad_() for _ in range(3))
    dy = torch.randn(N, S, H, E, device=DEV).to(dtype)

    def step():
        q.grad = k.grad = v.grad = None
        y = attn(q, k, v)
        y.backward(dy)
        return [y, q.grad, k.grad, v.grad]

    def eager():
        return [t.detach().clone() for t in step()]

    want = None if first_backward_in_capture else eager()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                      # warm-up off the capture stream, as bench.py does for the FFN
        for _ in range(2):
            if first_backward_in_capture:
                with torch.no_grad():
                    attn(q, k, v)
            else:
                step()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = step()
    assert attn.last_path == "fused"
    if want is None:
        want = eager()
    for _ in range(2):
        for t in outs:
            t.detach().zero_()
        graph.replay()
        torch.cuda.synchronize()
        for name, a, b in zip(("y", "dq", "dk", "dv"), outs, want):
            assert torch.equal(a.detach(), b), name


@gpu
def test_graph_capture_layer_d64():
    _graph_replay_equals_eager()


@gpu
def test_graph_capture_first_backward_in_capture():
    """In a fresh process whose first backward is captured (the serial fall-back of the launcher's side stream)."""
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_attn_persistent_gpu as t; "
            "t._graph_replay_equals_eager(first_backward_in_capture=True)" % (ROOT, os.path.dirname(os.path.abspath(__file__))))
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]


# ---------------------------------------------------------------------------------------------------------------------
# writes stay inside the outputs
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("reference_layout", [False, True])
@pytest.mark.parametrize("d", [64, 128])
def test_writes_stay_inside_outputs(d, reference_layout):
    """As test_fused_d80_writes_stay_inside_outputs, at N 2, S 1024 and G / 16 + 2 heads (two rounds of the d 64
    persistent grids): y, grad_q, grad_k, grad_v at the front of sentinel-filled buffers, pre-filled with NaN.  Afterwards
    every output element is finite and every sentinel unchanged."""
    from spt_proto_b200 import ext
    from spt_proto_b200._lib import SPT_ATTN_Y_TRANSPOSED, SPT_BF16, check, lib
    g = torch.Generator().manual_seed(33 + d)
    N, S, H = 2, 1024, _num_sms() // 16 + 2
    B = N * H
    q, k, v, dy = (torch.randn(N, S, H, d, generator=g).bfloat16().to(DEV) for _ in range(4))
    w = torch.randn(d // 8, 16, 8, generator=g).to(DEV)
    mask, extra0, _ = ext.lookup_mask(*ext.pq_encode_pair(q, k, w), 8)
    n, tail = q.numel(), 128 * S + 4096
    sentinel = 1536.0                # exactly representable in bf16
    bufs = [torch.full((n + tail,), sentinel, dtype=torch.bfloat16, device=DEV) for _ in range(4)]
    for b in bufs:
        b[:n] = float("nan")
    y, gq, gk, gv = bufs
    zsum = torch.empty(B, S, dtype=torch.float32, device=DEV)
    flags = SPT_ATTN_Y_TRANSPOSED if reference_layout else 0
    st = torch.cuda.current_stream().cuda_stream
    scale = d ** -0.5
    check(lib.spt_sparse_attn_fwd_ex(q.data_ptr(), k.data_ptr(), v.data_ptr(), mask.data_ptr(), extra0.data_ptr(),
                                     y.data_ptr(), zsum.data_ptr(), B, S, d, H, scale, CLAMP, SPT_BF16, flags, st))
    ws = torch.empty(lib.spt_sparse_attn_bwd_workspace_bytes(B, S), dtype=torch.uint8, device=DEV)
    check(lib.spt_sparse_attn_bwd_ex(q.data_ptr(), k.data_ptr(), v.data_ptr(), y.data_ptr(), dy.data_ptr(),
                                     mask.data_ptr(), extra0.data_ptr(), zsum.data_ptr(), gq.data_ptr(), gk.data_ptr(),
                                     gv.data_ptr(), ws.data_ptr(), B, S, d, H, scale, CLAMP, SPT_BF16, flags, st))
    torch.cuda.synchronize()
    for name, b in zip(("y", "grad_q", "grad_k", "grad_v"), bufs):
        assert torch.isfinite(b[:n].float()).all(), name
        assert (b[n:].float() == sentinel).all(), name
    y2, z2 = ext.sparse_attn_fwd(q, k, v, mask, extra0, scale, reference_layout=reference_layout)
    assert torch.equal(y[:n].view_as(q), y2) and torch.equal(zsum, z2)
    for got, want in zip((gq, gk, gv), ext.sparse_attn_bwd(q, k, v, y2, dy, mask, extra0, z2, scale,
                                                           reference_layout=reference_layout)):
        assert torch.equal(got[:n].view_as(q), want)
