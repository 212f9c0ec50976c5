"""fp16 through every layer: the PQ kernels, the fused attention kernels (d 64, 80, 128; both output layouts; head-major
and interleaved inputs), the V2 layers in `.half()`, the run-time switches and the rejections.

The fp16 kernels scale every score row by a power of two 2^-o_r (DESIGN.md section 4.1).  The scale cancels exactly in
y and in the gradients, so they are compared with the same float64 reference as the bf16 kernels
(tests/test_attn_persistent_gpu.py), computed on the fp16 inputs.  The range-edge cases compare row by row: a few bad rows
would disappear in a Frobenius norm."""
import os
import re
import subprocess
import sys

import pytest
import torch

from oracle import spt_oracle as O
from test_attn_persistent_gpu import (_assert_batch_invariant, _case_shape, _dy_memory, _edge_heads,
                                      _graph_replay_equals_eager, _heads, _mask_from_indices, _num_sms, _pack, _reference,
                                      _run, _split, _unpack, _y_heads)

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
CLAMP = 10.0
gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the header and the Python binding agree on the element-type codes
# ---------------------------------------------------------------------------------------------------------------------
def test_header_dtype_codes_match_binding():
    text = open(os.path.join(ROOT, "include", "spt_b200.h")).read()
    enum = re.search(r"typedef enum \{([^}]*)\} spt_dtype;", text).group(1)
    codes = {name: int(val) for name, val in re.findall(r"(SPT_\w+)\s*=\s*(\d+)", enum)}
    src = open(os.path.join(ROOT, "spt_proto_b200", "_lib.py")).read()
    for name in ("SPT_F32", "SPT_BF16", "SPT_F16"):
        assert int(re.search(rf"^{name} = (\d+)", src, re.M).group(1)) == codes[name], name
    assert codes["SPT_F16"] == 2


# ---------------------------------------------------------------------------------------------------------------------
# PQ kernels
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dc", [4, 8, 16])
def test_pq_encode_fp16_codes_bit_exact(dc):
    """fp16 -> fp32 is exact: the codes of z equal the oracle's codes of z.float(), single and pair."""
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(dc)
    m = 64 // dc
    z0, z1 = (torch.randn(3, 517, m * dc, generator=g).half() for _ in range(2))
    w = torch.randn(m, 16, dc, generator=g)
    want0, want1 = O.pq_encode(z0.float(), w), O.pq_encode(z1.float(), w)
    assert torch.equal(ext.pq_encode(z0.to(DEV), w.to(DEV)).cpu(), want0)
    c0, c1 = ext.pq_encode_pair(z0.to(DEV), z1.to(DEV), w.to(DEV))
    assert torch.equal(c0.cpu(), want0) and torch.equal(c1.cpu(), want1)


@gpu
@pytest.mark.parametrize("shape,m", [((4, 256, 64), 8), ((2, 300, 80), 10)])
def test_pq_train_fp16_matches_torch_formulation(shape, m):
    """As test_pq_train_fused_matches_torch_formulation, with fp16 z: loss, hard centroids, grad z (fp16), grad codebook."""
    from spt_proto_b200 import layers
    g = torch.Generator().manual_seed(sum(shape) + m)
    z = torch.randn(*shape, generator=g).half()
    ref = layers.PQV1(d_codeword=8, n_codewords=16, n_subspaces=m)
    with torch.no_grad():
        ref.weight.copy_(torch.randn(m, 16, 8, generator=g))
    zc = z.float().clone().requires_grad_()
    zq_ref, loss_ref = ref("train", z=zc)
    (3.0 * loss_ref + (zq_ref * 0.01).sum()).backward()
    mod = layers.PQV2(d_codeword=8, n_codewords=16, n_subspaces=m).to(DEV)
    with torch.no_grad():
        mod.weight.copy_(ref.weight)
    zd = z.to(DEV).requires_grad_()
    zq, loss = mod("train", z=zd)
    (3.0 * loss + (zq * 0.01).sum()).backward()
    assert zd.grad.dtype == torch.float16
    assert zq.shape == zq_ref.shape and torch.allclose(zq.cpu(), zq_ref.detach(), atol=1e-6)
    assert abs(loss.item() - loss_ref.item()) < 1e-4 * max(1.0, abs(loss_ref.item()))
    rel = lambda a, b: ((a.float().cpu() - b).norm() / b.norm()).item()
    assert rel(mod.weight.grad, ref.weight.grad) < 1e-4
    assert rel(zd.grad, zc.grad) < 6e-3


# ---------------------------------------------------------------------------------------------------------------------
# fused attention: parity with the float64 reference
# ---------------------------------------------------------------------------------------------------------------------
def _inputs16(N, S, H, d, seed):
    """fp16-representable float inputs (so fp16 takes them exactly) and PQ codebook."""
    g = torch.Generator().manual_seed(seed)
    q, k, v, dy = (torch.randn(N, S, H, d, generator=g).half().float() for _ in range(4))
    w = torch.randn(d // 8, 16, 8, generator=g)
    return q, k, v, dy, w


def _lookup(q, k, w, coeff=8):
    from spt_proto_b200 import ext
    mask, extra0, _ = ext.lookup_mask(*ext.pq_encode_pair(q.half().to(DEV), k.half().to(DEV), w.to(DEV)), coeff)
    return mask, extra0


def _run_dtype(dtype, q, k, v, dy, mask, extra0, scale, reference_layout, head_major=False, clamp=CLAMP):
    """Forward + backward of the fused kernels on the float inputs cast to `dtype` -> (y, zsum, gq, gk, gv), the
    tensors in the [N, S, H, d] layout (y in the reference layout's memory when reference_layout)."""
    from spt_proto_b200 import ext
    N, S, H, d = q.shape
    cast = lambda t: t.to(dtype).to(DEV)
    qd, kd, vd, dyd = cast(q), cast(k), cast(v), cast(_dy_memory(dy, reference_layout))
    if head_major:                              # [B, S, d] operands (H = 1 in the kernels)
        assert H == 1
        qd, kd, vd, dyd = (t.view(N, S, d) for t in (qd, kd, vd, dyd))
    y, z = ext.sparse_attn_fwd(qd, kd, vd, mask, extra0, scale, clamp, reference_layout=reference_layout)
    gq, gk, gv = ext.sparse_attn_bwd(qd, kd, vd, y, dyd, mask, extra0, z, scale, clamp, reference_layout=reference_layout)
    assert y.dtype == gq.dtype == gk.dtype == gv.dtype == dtype
    return [t.view(N, S, H, d) if t.dim() == 3 and t is not z else t for t in (y, z, gq, gk, gv)]


def _errors(out, q, k, v, dy, mask, extra0, scale, reference_layout, heads, clamp=CLAMP):
    """Relative Frobenius errors of y, dq, dk, dv over `heads` against the float64 reference."""
    y, _, gq, gk, gv = out
    got_all = [_y_heads(y, reference_layout).cpu()] + [_heads(t).cpu() for t in (gq, gk, gv)]
    qh, kh, vh, dyh = (_heads(t) for t in (q, k, v, dy))
    mask, extra0 = mask.cpu(), extra0.cpu()
    num, den = [0.0] * 4, [0.0] * 4
    for b in heads:
        want = _reference(qh[b], kh[b], vh[b], dyh[b], mask[b], extra0[b], scale, clamp)
        for i, (got, ref) in enumerate(zip((t[b].double() for t in got_all), want)):
            assert torch.isfinite(got).all(), (b, i)
            num[i] += (got - ref).norm().item() ** 2
            den[i] += ref.norm().item() ** 2
    return [(n / dd) ** 0.5 for n, dd in zip(num, den)]


def _assert_fp16_parity(q, k, v, dy, mask, extra0, scale, reference_layout, heads, head_major=False):
    """fp16 within 1e-2 relative Frobenius of the reference, and no worse than bf16 on the same inputs."""
    e16 = _errors(_run_dtype(torch.float16, q, k, v, dy, mask, extra0, scale, reference_layout, head_major),
                  q, k, v, dy, mask, extra0, scale, reference_layout, heads)
    e_bf = _errors(_run_dtype(torch.bfloat16, q, k, v, dy, mask, extra0, scale, reference_layout, head_major),
                   q, k, v, dy, mask, extra0, scale, reference_layout, heads)
    print("fp16 errors (y, dq, dk, dv):", ["%.2e" % e for e in e16], " bf16:", ["%.2e" % e for e in e_bf])
    for name, a, b in zip(("y", "dq", "dk", "dv"), e16, e_bf):
        assert a < 1e-2, (name, a)
        assert a <= b, (name, a, b)


@gpu
@pytest.mark.parametrize("layout", ["interleaved", "interleaved_reference_layout", "head_major"])
@pytest.mark.parametrize("S", [256, 2048])
@pytest.mark.parametrize("d", [64, 80, 128])
def test_fp16_parity(d, S, layout):
    """d 64, 80, 128 at S 256 and 2048: interleaved [N, S, H, d] inputs in both output layouts, and head-major [B, S, d]."""
    head_major = layout == "head_major"
    N, H = (2, 1) if head_major else (1, 2)
    q, k, v, dy, w = _inputs16(N, S, H, d, 1000 * d + S)
    mask, extra0 = _lookup(q, k, w)
    _assert_fp16_parity(q, k, v, dy, mask, extra0, d ** -0.5, layout.endswith("reference_layout"), range(N * H),
                        head_major)


@gpu
@pytest.mark.parametrize("reference_layout", [False, True])
@pytest.mark.parametrize("case", ["items_G+1", "s1024_3rounds"])
def test_fp16_parity_persistent_rounds(case, reference_layout):
    """The d 64 persistent backward past one round: S 128 x (G + 1) heads and S 1024 x (2G / 8 + 1) heads."""
    G = _num_sms()
    S, B = _case_shape(case, G)
    N, H = _split(B)
    q, k, v, dy, w = _inputs16(N, S, H, 64, S + B)
    mask, extra0 = _lookup(q, k, w)
    heads = range(B) if S == 128 else _edge_heads(S, B, G)
    _assert_fp16_parity(q, k, v, dy, mask, extra0, 64 ** -0.5, reference_layout, heads)


@gpu
@pytest.mark.parametrize("S", [4096, 8192])
def test_fp16_parity_long_sequence(S):
    q, k, v, dy, w = _inputs16(1, S, 1, 64, S)
    mask, extra0 = _lookup(q, k, w)
    _assert_fp16_parity(q, k, v, dy, mask, extra0, 64 ** -0.5, False, [0])


# ---------------------------------------------------------------------------------------------------------------------
# range edges, row by row
# ---------------------------------------------------------------------------------------------------------------------
def _assert_rows(out, q, k, v, dy, mask, extra0, scale, reference_layout, heads, rtol=3e-2):
    """Every output element finite; per row r of y, dq (queries) and dk, dv (keys):
    |got_r - ref_r| <= rtol |ref_r| + 2e-3 max_r |ref_r| (rows whose exact value is 0, such as those that select key 0
    alone, keep a rounding residue of dO').  Rows and keys with a selected score within 1e-4 of the clamp
    are skipped: there the fp32 score of the kernel and the float64 one of the reference may fall on different sides of
    the zero-gradient indicator."""
    y, _, gq, gk, gv = out
    got_all = [_y_heads(y, reference_layout).cpu()] + [_heads(t).cpu() for t in (gq, gk, gv)]
    for t in got_all:
        assert torch.isfinite(t.float()).all()
    qh, kh, vh, dyh = (_heads(t) for t in (q, k, v, dy))
    mask, extra0 = mask.cpu(), extra0.cpu()
    for b in heads:
        want = _reference(qh[b], kh[b], vh[b], dyh[b], mask[b], extra0[b], scale)
        S = qh.shape[1]
        sel = (_unpack(mask[b]) > 0) | (torch.arange(S) == 0).unsqueeze(0) & (extra0[b] > 0).unsqueeze(1)
        sel &= torch.arange(S).unsqueeze(0) <= torch.arange(S).unsqueeze(1)
        edge = sel & (((scale * qh[b].double() @ kh[b].double().T).abs() - CLAMP).abs() < 1e-4)
        skip = {"y": edge.any(1), "dq": edge.any(1), "dk": edge.any(0), "dv": edge.any(0)}
        for name, got, ref in zip(("y", "dq", "dk", "dv"), (t[b].double() for t in got_all), want):
            err, norm = (got - ref).norm(dim=1), ref.norm(dim=1)
            bad = (err > rtol * norm + 2e-3 * norm.max()) & ~skip[name]
            assert not bad.any(), (b, name, bad.nonzero().flatten()[:8].tolist(), (err / norm.clamp_min(1e-30)).max().item())


def _low_scores(N, S, H, d, seed):
    """q, k with q.k within 0.5 of -clamp for every pair (scale 1): q_r = -9.75 u, k_j = u + n_j with n_j orthogonal to u
    (so that dQ does not cancel to rounding noise)."""
    g = torch.Generator().manual_seed(seed)
    u = torch.randn(d, generator=g)
    u /= u.norm()
    n = 0.5 * torch.randn(N, S, H, d, generator=g)
    n -= (n @ u).unsqueeze(-1) * u
    k = (u + n).half().float()
    q = (-9.75 * u).expand(N, S, H, d).half().float().contiguous()
    s = q[0, 0, 0] @ k.reshape(-1, d).T
    assert ((s + CLAMP).abs() <= 0.5).all() and (s > -CLAMP).all()
    return q, k


@gpu
@pytest.mark.parametrize("kind", ["scale_x6", "codes_c1", "codes_c2", "plus_clamp_max_extra0", "low_rows",
                                  "low_rows_padded", "dy_x256"])
@pytest.mark.parametrize("d", [64, 128])
def test_fp16_range_edges(kind, d):
    """scale_x6: most scores clamp, padded early rows (the lookup's r < nnz).  codes_c1 / codes_c2: overflowing codes
    put padding in late rows.  plus_clamp_max_extra0: rows with q_r = k_0 (score at +clamp) that select key 0 alone with
    extra0 = nnz - 1.  low_rows(_padded): every score within 0.5 of -clamp, without / with zero padding.  dy_x256: dO
    scaled by 2^8, as under loss scaling.  Both output layouts; every output finite; row-by-row against the reference."""
    N, S, H = 1, 1024, 2
    coeff = 128 if kind == "codes_c2" else 8       # two distinct codes leave late-row padding only at top-k S / 128
    nnz = S // coeff
    q, k, v, dy, w = _inputs16(N, S, H, d, 77 + len(kind) + d)
    scale = d ** -0.5
    if kind.startswith("codes"):
        from spt_proto_b200 import ext
        g = torch.Generator().manual_seed(int(kind[-1]))
        q_c, k_c = (torch.randint(0, int(kind[-1]), (N, S, H, 8), generator=g, dtype=torch.int32).to(DEV) for _ in range(2))
        mask, extra0, _ = ext.lookup_mask(q_c, k_c, coeff)
        assert (extra0[:, nnz:] > 0).any()
    elif kind.startswith("low_rows"):
        q, k = _low_scores(N, S, H, d, 5)
        scale = 1.0
        g = torch.Generator().manual_seed(6)
        sel = (torch.rand(N * H, S, S, generator=g) < 1.0 / coeff) & (torch.arange(S) <= torch.arange(S).unsqueeze(1))
        sel[:, :, 0] = True
        mask = torch.stack([_pack(s) for s in sel]).to(DEV)
        extra0 = torch.zeros(N * H, S, dtype=torch.int32)
        if kind == "low_rows_padded":
            extra0 = torch.randint(0, nnz, (N * H, S), generator=g, dtype=torch.int32)
        extra0 = extra0.to(DEV)
    else:
        if kind == "scale_x6":
            scale *= 6
        mask, extra0 = _lookup(q, k, w)
        if kind == "scale_x6":
            assert (extra0[:, :nnz] > 0).any()
        if kind == "plus_clamp_max_extra0":
            rows = torch.arange(3, S, 16)
            q[:, rows] = k[:, :1].expand(N, len(rows), H, d)         # scale q_r . k_0 = sqrt(d) |k_0|^2 / d >> 10
            mask[:, rows.to(DEV)] = 0
            mask[:, rows.to(DEV), 0] = 1
            extra0[:, rows.to(DEV)] = nnz - 1
        if kind == "dy_x256":
            dy = dy * 256
    for reference_layout in (False, True):
        out = _run_dtype(torch.float16, q, k, v, dy, mask, extra0, scale, reference_layout)
        _assert_rows(out, q, k, v, dy, mask, extra0, scale, reference_layout, range(N * H))


# ---------------------------------------------------------------------------------------------------------------------
# bit-exact behaviour
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("d", [64, 80, 128])
def test_fp16_two_runs_equal(d):
    q, k, v, dy, w = _inputs16(2, 1024, 3, d, d)
    mask, extra0 = _lookup(q, k, w)
    for reference_layout in (False, True):
        a = _run_dtype(torch.float16, q, k, v, dy, mask, extra0, d ** -0.5, reference_layout)
        b = _run_dtype(torch.float16, q, k, v, dy, mask, extra0, d ** -0.5, reference_layout)
        for x, y in zip(a, b):
            assert torch.equal(x, y)


@gpu
@pytest.mark.parametrize("reference_layout", [False, True])
@pytest.mark.parametrize("case", ["s1024_3rounds", "d80", "d128"])
def test_fp16_batch_invariance(case, reference_layout):
    """Each head of a batched fp16 call equals that head called alone, bit for bit (y, zsum, dq, dk, dv)."""
    if case == "s1024_3rounds":
        S, B = _case_shape(case, _num_sms())
        N, H = _split(B)
        d = 64
    else:
        N, S, H, d = 2, 512, 3, int(case[1:])
    q, k, v, dy, w = _inputs16(N, S, H, d, 9 + d)
    mask, extra0 = _lookup(q, k, w)
    _assert_batch_invariant(q.half().to(DEV), k.half().to(DEV), v.half().to(DEV),
                            _dy_memory(dy, reference_layout).half().to(DEV), mask, extra0, d ** -0.5, reference_layout)


@gpu
def test_fp16_switch_tile64_parity():
    """SPT_ATTN_TILE=64 (the 128 x 64 backward at d 64), in a child process: the parity tests at d 64, including the
    shapes of the persistent-grid tests."""
    env = dict(os.environ, SPT_ATTN_TILE="64")
    res = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", os.path.abspath(__file__), "-k",
                          "(test_fp16_parity and 64) or test_fp16_parity_persistent_rounds"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert " passed" in res.stdout and "failed" not in res.stdout


@gpu
def test_fp16_graph_capture_layer():
    """The fp16 SparseVanillaAttentionV2 (d 64, fused, two rounds) captured forward + backward with torch.cuda.graph:
    two replays give y and the three gradients of the eager step bit for bit."""
    _graph_replay_equals_eager(dtype=torch.float16, seed=19)


@gpu
def test_fp16_graph_capture_first_backward_in_capture():
    """As test_fp16_graph_capture_layer in a fresh process whose first backward is captured: the replays run the dK/dV
    and dQ kernels one after the other (the launcher's fall-back without a side stream) and equal the eager step, which
    forks dQ onto the side stream, bit for bit."""
    code = ("import sys, torch; sys.path[:0] = [%r, %r]; import test_attn_persistent_gpu as t; "
            "t._graph_replay_equals_eager(first_backward_in_capture=True, dtype=torch.float16, seed=19)" % (ROOT, HERE))
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]


@gpu
@pytest.mark.parametrize("reference_layout", [False, True])
@pytest.mark.parametrize("d", [64, 80, 128])
def test_fp16_writes_stay_inside_outputs(d, reference_layout):
    """y, grad_q, grad_k, grad_v at the front of sentinel-filled fp16 buffers pre-filled with NaN (N 2, S 1024, G / 16 + 2
    heads): afterwards every output element is finite and every sentinel unchanged."""
    from spt_proto_b200 import ext
    from spt_proto_b200._lib import SPT_ATTN_Y_TRANSPOSED, SPT_F16, check, lib
    N, S, H = 2, 1024, _num_sms() // 16 + 2
    B = N * H
    q, k, v, dy, w = _inputs16(N, S, H, d, 33 + d)
    q, k, v, dy = (t.half().to(DEV) for t in (q, k, v, dy))
    mask, extra0, _ = ext.lookup_mask(*ext.pq_encode_pair(q, k, w.to(DEV)), 8)
    n, tail = q.numel(), 128 * S + 4096
    sentinel = 1536.0                # exactly representable in fp16
    bufs = [torch.full((n + tail,), sentinel, dtype=torch.float16, device=DEV) for _ in range(4)]
    for b in bufs:
        b[:n] = float("nan")
    y, gq, gk, gv = bufs
    zsum = torch.empty(B, S, dtype=torch.float32, device=DEV)
    flags = SPT_ATTN_Y_TRANSPOSED if reference_layout else 0
    st = torch.cuda.current_stream().cuda_stream
    scale = d ** -0.5
    check(lib.spt_sparse_attn_fwd_ex(q.data_ptr(), k.data_ptr(), v.data_ptr(), mask.data_ptr(), extra0.data_ptr(),
                                     y.data_ptr(), zsum.data_ptr(), B, S, d, H, scale, CLAMP, SPT_F16, flags, st))
    ws = torch.empty(lib.spt_sparse_attn_bwd_workspace_bytes(B, S), dtype=torch.uint8, device=DEV)
    check(lib.spt_sparse_attn_bwd_ex(q.data_ptr(), k.data_ptr(), v.data_ptr(), y.data_ptr(), dy.data_ptr(),
                                     mask.data_ptr(), extra0.data_ptr(), zsum.data_ptr(), gq.data_ptr(), gk.data_ptr(),
                                     gv.data_ptr(), ws.data_ptr(), B, S, d, H, scale, CLAMP, SPT_F16, flags, st))
    torch.cuda.synchronize()
    for name, b in zip(("y", "grad_q", "grad_k", "grad_v"), bufs):
        assert torch.isfinite(b[:n].float()).all(), name
        assert (b[n:].float() == sentinel).all(), name
    y2, z2 = ext.sparse_attn_fwd(q, k, v, mask, extra0, scale, reference_layout=reference_layout)
    assert torch.equal(y2.reshape(-1), y[:n]) and torch.equal(z2, zsum)


@gpu
@pytest.mark.parametrize("kind", ["lookup", "plus_clamp_max_extra0", "low_rows"])
def test_fp16_zsum_matches_bf16_definition(kind):
    """fp16 zsum = sum_j w exp(clamp(scale s)) in fp32 without the row scale: within fp16 rounding of the float64 sum."""
    N, S, H, d = 1, 1024, 2, 64
    q, k, v, dy, w = _inputs16(N, S, H, d, 4)
    scale = d ** -0.5
    mask, extra0 = _lookup(q, k, w)
    if kind == "plus_clamp_max_extra0":
        rows = torch.arange(3, S, 16)
        q[:, rows] = k[:, :1].expand(N, len(rows), H, d)
        mask[:, rows.to(DEV)] = 0
        mask[:, rows.to(DEV), 0] = 1
        extra0[:, rows.to(DEV)] = S // 8 - 1
    elif kind == "low_rows":
        q, k = _low_scores(N, S, H, d, 8)
        scale = 1.0
    _, z, *_ = _run_dtype(torch.float16, q, k, v, dy, mask, extra0, scale, False)
    qh, kh = _heads(q).double(), _heads(k).double()
    for b in range(N * H):
        wts = _unpack(mask[b].cpu()).double()
        wts[:, 0] += extra0[b].cpu().double()
        wts *= torch.arange(S).unsqueeze(0) <= torch.arange(S).unsqueeze(1)
        zref = (wts * torch.exp((scale * qh[b] @ kh[b].T).clamp(-CLAMP, CLAMP))).sum(1).clamp_min(1e-9)
        assert torch.allclose(z[b].cpu().double(), zref, rtol=2e-3, atol=0), b


# ---------------------------------------------------------------------------------------------------------------------
# layers in .half()
# ---------------------------------------------------------------------------------------------------------------------
def _layer_run(attn, q, k, v, dy):
    q.grad = k.grad = v.grad = None
    y = attn(q, k, v)
    y.backward(dy)
    assert y.dtype == q.grad.dtype == torch.float16
    return [t.detach().float().clone() for t in (y, q.grad, k.grad, v.grad)]


def _rope_cpu(x, cos, sin):
    lo, hi = x.chunk(2, dim=-1)
    return x * cos.view(1, -1, 1, x.size(-1)) + torch.cat((-hi, lo), dim=-1) * sin.view(1, -1, 1, x.size(-1))


@gpu
@pytest.mark.parametrize("reference_layout", [False, True])
@pytest.mark.parametrize("rotary", [False, True])
def test_fp16_layer_fused_matches_oracle(rotary, reference_layout):
    """SparseVanillaAttentionV2 / SparseRotaryAttentionV2 in .half() take the fused path and match the oracle layer, in
    both output layouts.  The rotary layer's tables are fp16 after .half(), so it rotates in fp16 arithmetic: the oracle
    takes that rotation's values (the operands the kernels and the PQ encoder see) with the fp32 rotation's gradient."""
    from spt_proto_b200 import layers
    torch.manual_seed(21)
    N, S, H, E = 2, 256, 4, 64
    cls = layers.SparseRotaryAttentionV2 if rotary else layers.SparseVanillaAttentionV2
    attn = cls(d_head=E, p_dropout=0.0, d_codeword=8, n_codewords=16,
               reference_output_layout=reference_layout).to(DEV).half()
    q, k, v, dy = (torch.randn(N, S, H, E).half() for _ in range(4))
    qd, kd, vd = (t.to(DEV).requires_grad_() for t in (q, k, v))
    y, gq, gk, gv = _layer_run(attn, qd, kd, vd, dy.to(DEV))
    assert attn.last_path == "fused"
    qf, kf, vf = (t.float().requires_grad_() for t in (q, k, v))
    qr, kr = qf, kf
    if rotary:
        emb = attn.embedding
        cos, sin = emb.cos_cached[:S].float().cpu(), emb.sin_cached[:S].float().cpu()
        qr, kr = _rope_cpu(qf, cos, sin), _rope_cpu(kf, cos, sin)
        with torch.no_grad():
            q16, k16 = (attn._rotate(t.to(DEV)).float().cpu() for t in (q, k))
        qr = qr + (q16 - qr.detach())                           # the layer's fp16 rotation, straight-through gradient
        kr = kr + (k16 - kr.detach())
    y_ref = O.sparse_mha_layer(qr, kr, vf, attn.quantizer.weight.detach().float().cpu(), 8,
                               reference_output_layout=reference_layout)
    y_ref.backward(dy.float())
    rel = lambda a, b: ((a.cpu() - b).norm() / b.norm()).item()
    assert rel(y, y_ref.detach()) < 1e-2
    assert rel(gv, vf.grad) < 1.5e-2
    assert rel(gq, qf.grad) < 2e-2
    assert rel(gk, kf.grad) < 2e-2


@gpu
@pytest.mark.parametrize("case", ["s1088", "use_fused_false"])
def test_fp16_layer_stage_path_matches_oracle(case):
    """Outside the fused envelope (S 1088 is not a multiple of 128) or with use_fused = False, the fp16 layer runs the
    stage chain in fp32 and returns fp16; it matches the oracle layer."""
    from spt_proto_b200 import layers
    torch.manual_seed(22)
    N, S, H, E = 1, (1088 if case == "s1088" else 256), 2, 64
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0,
                                           reference_output_layout=False).to(DEV).half()
    attn.use_fused = case != "use_fused_false"
    q, k, v, dy = (torch.randn(N, S, H, E).half() for _ in range(4))
    qd, kd, vd = (t.to(DEV).requires_grad_() for t in (q, k, v))
    y, gq, gk, gv = _layer_run(attn, qd, kd, vd, dy.to(DEV))
    assert attn.last_path == "stage"
    qf, kf, vf = (t.float().requires_grad_() for t in (q, k, v))
    y_ref = O.sparse_mha_layer(qf, kf, vf, attn.quantizer.weight.detach().float().cpu(), 8)
    y_ref.backward(dy.float())
    rel = lambda a, b: ((a.cpu() - b).norm() / b.norm()).item()
    assert rel(y, y_ref.detach()) < 2e-3
    for got, want in ((gq, qf.grad), (gk, kf.grad), (gv, vf.grad)):
        assert rel(got, want) < 5e-3


@gpu
def test_fp16_layer_armed_pq_loss_matches_fp32_formulation():
    """The armed PQ loss of an fp16 layer (fused PQ train kernels on fp16 q, k) equals the fp32 formulation on the same
    values, and its gradient reaches the codebook."""
    from spt_proto_b200 import layers
    torch.manual_seed(23)
    N, S, H, E = 1, 256, 2, 64
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0).to(DEV).half()
    q, k, v = (torch.randn(N, S, H, E).half() for _ in range(3))
    attn.host_trigger = True
    attn(q.to(DEV), k.to(DEV), v.to(DEV))
    assert attn.last_path == "fused"
    w32 = attn.quantizer.weight.detach().float().cpu()
    want = O.pq_train_loss(q.float(), w32) + O.pq_train_loss(k.float(), w32)
    assert abs(attn.loss.item() - want.item()) < 1e-4 * max(1.0, abs(want.item()))
    attn.loss.backward()
    assert attn.quantizer.weight.grad is not None and torch.isfinite(attn.quantizer.weight.grad.float()).all()


# ---------------------------------------------------------------------------------------------------------------------
# rejections
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_fp16_rejections():
    from spt_proto_b200 import ext
    q, k, v, dy, w = _inputs16(1, 256, 1, 64, 3)
    mask, extra0 = _lookup(q, k, w)
    h = lambda t: t.half().to(DEV)
    with pytest.raises(RuntimeError, match="k must be type of torch.float16"):
        ext.sparse_attn_fwd(h(q), k.bfloat16().to(DEV), h(v), mask, extra0, 0.125)
    y, z = ext.sparse_attn_fwd(h(q), h(k), h(v), mask, extra0, 0.125)
    with pytest.raises(RuntimeError, match="grad_y must be type of torch.float16"):
        ext.sparse_attn_bwd(h(q), h(k), h(v), y, dy.bfloat16().to(DEV), mask, extra0, z, 0.125)
    for clamp in (10.5, 20.0):
        with pytest.raises(RuntimeError, match="fp16 needs 0 <= clamp <= 10"):
            ext.sparse_attn_fwd(h(q), h(k), h(v), mask, extra0, 0.125, clamp)
        with pytest.raises(RuntimeError, match="fp16 needs 0 <= clamp <= 10"):
            ext.sparse_attn_bwd(h(q), h(k), h(v), y, h(dy), mask, extra0, z, 0.125, clamp)
    # bf16 keeps accepting any clamp
    ext.sparse_attn_fwd(q.bfloat16().to(DEV), k.bfloat16().to(DEV), v.bfloat16().to(DEV), mask, extra0, 0.125, 20.0)
