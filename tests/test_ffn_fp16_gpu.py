"""fp16 routed FFN on the GPU: the grouped GEMM with fp16 operands against float64 products of the same fp16 values,
fp16 overflow, the elementwise kernels against torch, the four layers in .half() against a float64 oracle on their
own values (and against the error of the same module in bf16), the headline shapes, the absence of any bf16 copy or
saved bf16 tensor, determinism, graph capture, and an OPT-1.3B-shape block upgraded and run in fp16."""
import copy
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SENT = 1234.0          # sentinel of the guard band around every GEMM output (exact in fp16 and fp32)


def _groups(sizes):
    """padded (x128) bucket layout for the given real group sizes"""
    ptr, tiles = [0], []
    for g, n in enumerate(sizes):
        pad = (n + 127) // 128 * 128
        ptr.append(ptr[-1] + pad)
        tiles += [g] * (pad // 128)
    return ptr, tiles


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm()).item()


def _guarded(rows, cols, dtype):
    """NaN-filled [rows, cols] output view inside a buffer with a sentinel band of 1 row and 8 columns on every side
    (leading dimension cols + 16: 16-byte aligned rows in fp16 and fp32)."""
    full = torch.full((rows + 2, cols + 16), SENT, dtype=dtype, device=DEV)
    view = full[1:1 + rows, 8:8 + cols]
    view.fill_(float("nan"))
    return full, view


def _check_guard(full, rows, cols):
    f = full.float().cpu()
    band = torch.ones_like(f, dtype=torch.bool)
    band[1:1 + rows, 8:8 + cols] = False
    assert (f[band] == SENT).all(), "a write left the output"


def _bound(out_dtype):
    return 1e-4 if out_dtype == torch.float32 else 1e-3


def _assert_fp16_accuracy(got, want, want_bf, out_dtype):
    """got within the bound of the float64 product of the fp16 values; the same product on bf16-rounded operands
    (want_bf) must miss that bound, so the check would catch a bf16 rounding anywhere in the GEMM."""
    bound = _bound(out_dtype)
    assert _rel(got, want) < bound, _rel(got, want)
    assert _rel(want_bf, want) > bound, _rel(want_bf, want)


# ---------------------------------------------------------------------------------------------- grouped GEMM, fp16
@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("b_mn", [False, True])
@pytest.mark.parametrize("sizes,N,K", [([300, 0, 77, 513], 256, 192), ([200, 129], 2752, 128)])
def test_fp16_gemm_mode0(sizes, N, K, b_mn, out_dtype):
    """fc1 form: bias + ReLU + row scale, K- and MN-major B, ragged N (2752 = 10.75 x 256); tail tiles (-1) come out
    as zeros in a NaN-filled buffer."""
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(N + K + sum(sizes))
    G = len(sizes)
    ptr, tiles = _groups(sizes)
    R = ptr[-1]
    A = torch.zeros(R, K)
    for gi, n in enumerate(sizes):
        A[ptr[gi]: ptr[gi] + n] = torch.randn(n, K, generator=g)
    W = torch.randn(G * N, K, generator=g)
    A, W = A.half(), W.half()
    bias = torch.randn(G * N, generator=g)
    scale = torch.rand(R, generator=g) + 0.5

    def product(a, w):
        out = torch.zeros(R, N, dtype=torch.float64)
        for gi in range(G):
            rows = slice(ptr[gi], ptr[gi + 1])
            out[rows] = torch.relu(a[rows].double() @ w[gi * N:(gi + 1) * N].double().t()
                                   + bias[gi * N:(gi + 1) * N].double()) * scale[rows, None].double()
        return out

    want, want_bf = product(A, W), product(A.bfloat16(), W.bfloat16())
    full, out = _guarded(R + 256, N, out_dtype)
    Bm = W.t().contiguous() if b_mn else W
    ext.grouped_gemm(0, A.to(DEV), False, Bm.to(DEV), b_mn, tile_group=torch.tensor(tiles + [-1, -1], dtype=torch.int32,
                     device=DEV), N=N, K=K, b_mn_off=N, out=out, bias=bias.to(DEV), bias_stride=N,
                     row_scale=torch.cat([scale, torch.ones(256)]).to(DEV), act=1)
    got = out.float().cpu()
    assert (got[R:] == 0).all()
    _assert_fp16_accuracy(got[:R], want, want_bf, out_dtype)
    _check_guard(full, R + 256, N)


@pytest.mark.parametrize("sizes,bs,d,out_dtype", [([200, 129, 384], 128, 256, torch.float16),
                                                  ([130, 260], 2752, 256, torch.float32),
                                                  ([130, 260], 2752, 384, torch.float16)])
def test_fp16_gemm_mode0_fc2_layout(sizes, bs, d, out_dtype):
    """fc2: B_g = W2[:, g*bs:(g+1)*bs], K-major with a K offset per group and leading dim F; K = 2752 is ragged in
    256-wide B panels."""
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(bs + d)
    G = len(sizes)
    ptr, tiles = _groups(sizes)
    R = ptr[-1]
    H = (torch.randn(R, bs, generator=g) * 0.1).half()
    W2 = torch.randn(d, G * bs, generator=g).half()

    def product(h, w):
        out = torch.zeros(R, d, dtype=torch.float64)
        for gi in range(G):
            rows = slice(ptr[gi], ptr[gi + 1])
            out[rows] = h[rows].double() @ w[:, gi * bs:(gi + 1) * bs].double().t()
        return out

    full, out = _guarded(R, d, out_dtype)
    ext.grouped_gemm(0, H.to(DEV), False, W2.to(DEV), False, tile_group=torch.tensor(tiles, dtype=torch.int32,
                     device=DEV), N=d, K=bs, b_k_off=bs, out=out)
    _assert_fp16_accuracy(out.float().cpu(), product(H, W2), product(H.bfloat16(), W2.bfloat16()), out_dtype)
    _check_guard(full, R, d)


@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float16])
@pytest.mark.parametrize("sizes,M,N", [([384, 0, 128, 640], 256, 192), ([256, 320], 2752, 128)])
def test_fp16_gemm_mode1_weight_grad(sizes, M, N, out_dtype):
    """dW_g [M, N] = dU_g^T X_g over the group's rows, both operands MN-major, blocks stacked along the rows
    (c_row_off) and side by side along the columns (c_col_off); M = 2752 leaves a half 128-row tile."""
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(M + N)
    G = len(sizes)
    ptr = [0]
    for n in sizes:
        ptr.append(ptr[-1] + n)
    R = ptr[-1]
    dU = (torch.randn(R, M, generator=g) * 0.1).half()
    X = torch.randn(R, N, generator=g).half()
    gp = torch.tensor(ptr, dtype=torch.int32, device=DEV)

    def product(a, b):
        return torch.stack([a[ptr[i]:ptr[i + 1]].double().t() @ b[ptr[i]:ptr[i + 1]].double() for i in range(G)])

    want, want_bf = product(dU, X), product(dU.bfloat16(), X.bfloat16())
    nz = [i for i in range(G) if sizes[i]]          # an empty group's block is exactly zero: compare the others
    full, out = _guarded(G * M, N, out_dtype)
    ext.grouped_gemm(1, dU.to(DEV), True, X.to(DEV), True, group_ptr=gp, M=M, N=N, c_row_off=M, out=out)
    got = out.float().cpu().reshape(G, M, N)
    _assert_fp16_accuracy(got[nz], want[nz], want_bf[nz], out_dtype)
    assert all((got[i] == 0).all() for i in range(G) if not sizes[i])
    _check_guard(full, G * M, N)
    full2, out2 = _guarded(M, G * N, out_dtype)
    ext.grouped_gemm(1, dU.to(DEV), True, X.to(DEV), True, group_ptr=gp, M=M, N=N, c_col_off=N, out=out2)
    got2 = out2.float().cpu().reshape(M, G, N).transpose(0, 1)
    _assert_fp16_accuracy(got2[nz], want[nz], want_bf[nz], out_dtype)
    _check_guard(full2, M, G * N)


@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float16])
def test_fp16_gemm_gate_epilogue(out_dtype):
    """dH = dY . W2_g (MN-major B with an N offset) zeroed where the fp16 gate H <= 0 (ReLU backward in the epilogue),
    at a ragged block of 2752 columns."""
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(77)
    sizes, bs, d = [300, 100], 2752, 256
    G = len(sizes)
    ptr, tiles = _groups(sizes)
    R = ptr[-1]
    dY = (torch.randn(R, d, generator=g) * 0.1).half()
    W2 = torch.randn(d, G * bs, generator=g).half()
    Hg = torch.randn(R, bs, generator=g).half()
    Hg[::5, ::3] = 0                                  # exact zeros are masked too (gate <= 0)
    want = torch.zeros(R, bs, dtype=torch.float64)
    want_bf = torch.zeros(R, bs, dtype=torch.float64)
    for gi in range(G):
        rows = slice(ptr[gi], ptr[gi + 1])
        want[rows] = dY[rows].double() @ W2[:, gi * bs:(gi + 1) * bs].double()
        want_bf[rows] = dY[rows].bfloat16().double() @ W2[:, gi * bs:(gi + 1) * bs].bfloat16().double()
    keep = (Hg > 0).double()
    want, want_bf = want * keep, want_bf * keep
    full, out = _guarded(R, bs, out_dtype)
    ext.grouped_gemm(0, dY.to(DEV), False, W2.to(DEV), True, tile_group=torch.tensor(tiles, dtype=torch.int32, device=DEV),
                     N=bs, K=d, b_mn_off=bs, out=out, gate=Hg.to(DEV))
    got = out.float().cpu()
    assert (got[keep == 0] == 0).all()
    _assert_fp16_accuracy(got, want, want_bf, out_dtype)
    _check_guard(full, R, bs)


def test_fp16_gemm_single_cta_kernel():
    """The same GEMM cases on the single-CTA kernel (SPT_GEMM_CTA_PAIR=0 is read once per process: a child)."""
    env = dict(os.environ, SPT_GEMM_CTA_PAIR="0")
    res = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", os.path.abspath(__file__), "-k",
                          "fp16_gemm and not single_cta"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert " passed" in res.stdout and "failed" not in res.stdout


def test_fp16_gemm_overflow_is_inf_like_torch():
    """An output whose fp32 value exceeds the fp16 range stores +-inf (no saturation), as torch.matmul does on the
    same fp16 operands; its finite neighbours are correct."""
    from spt_proto_b200 import ext
    g = torch.Generator().manual_seed(3)
    N, K = 256, 128
    A = torch.randn(128, K, generator=g).half()
    W = torch.randn(N, K, generator=g).half()
    A[0], W[0] = 64.0, 64.0          # 64 * 64 * 128 = 524288 > 65504
    A[1] = -64.0                     # row 1, column 0: -524288
    out = torch.empty(128, N, dtype=torch.float16, device=DEV)
    ext.grouped_gemm(0, A.to(DEV), False, W.to(DEV), False, tile_group=torch.zeros(1, dtype=torch.int32, device=DEV),
                     N=N, K=K, out=out)
    ref = torch.matmul(A.to(DEV), W.to(DEV).t())
    got = out.cpu()
    assert got[0, 0].item() == float("inf") and got[1, 0].item() == float("-inf")
    assert ref[0, 0].item() == float("inf") and ref[1, 0].item() == float("-inf")
    fin = torch.ones_like(got, dtype=torch.bool)
    fin[0, 0] = fin[1, 0] = False
    assert torch.isfinite(got[fin]).all()
    want = A.double() @ W.double().t()
    assert _rel(got.double()[fin], want[fin]) < 1e-3


def test_fp16_binding_rejections():
    from spt_proto_b200 import ext
    A = torch.zeros(128, 64, dtype=torch.float16, device=DEV)
    tg = torch.zeros(1, dtype=torch.int32, device=DEV)
    with pytest.raises(RuntimeError, match="A and B must have the same dtype"):
        ext.grouped_gemm(0, A, False, A.bfloat16(), False, tile_group=tg, N=128, K=64, out=torch.empty(128, 128, device=DEV))
    with pytest.raises(RuntimeError, match="gate must have the operands' dtype"):
        ext.grouped_gemm(0, A, False, A, False, tile_group=tg, N=128, K=64, out=torch.empty(128, 128, device=DEV),
                         gate=torch.zeros(128, 128, dtype=torch.bfloat16, device=DEV))
    with pytest.raises(RuntimeError, match="out must be torch.float32 or the operand type"):
        ext.grouped_gemm(0, A, False, A, False, tile_group=tg, N=128, K=64,
                         out=torch.empty(128, 128, dtype=torch.bfloat16, device=DEV))
    with pytest.raises(RuntimeError, match="bf16 and fp16 do not mix"):
        ext.ffn_combine(torch.zeros(128, 64, dtype=torch.bfloat16, device=DEV),
                        torch.zeros(4, 2, dtype=torch.int32, device=DEV), None, torch.float16)


# ------------------------------------------------------------------------------------------ elementwise kernels, fp16
def _one_rounding(got, ref, dtype, atol=1e-5):
    """|got - ref| within one rounding to `dtype` of the exact value (plus fp32 arithmetic slack)."""
    rt = 2.0 ** -11 if dtype == torch.float16 else 2e-6
    err = (got.double().cpu() - ref.double().cpu()).abs()
    lim = rt * ref.double().cpu().abs() * 1.01 + atol
    assert (err <= lim).all(), (err - lim).max().item()


def test_fp16_gather_rows_and_combine():
    from spt_proto_b200 import ext
    torch.manual_seed(4)
    T, nb, k, C = 700, 8, 4, 520
    prob = torch.rand(T, nb, device=DEV)
    b = ext.route_bucket(prob, k)
    x = torch.randn(T, C, device=DEV).half()
    xp = ext.gather_rows(x, b.row_token)
    assert xp.dtype == torch.float16
    tok = b.row_token.long()
    want = torch.where((tok >= 0)[:, None], x[tok.clamp(min=0)], torch.zeros((), dtype=x.dtype, device=DEV))
    assert torch.equal(xp, want)
    bias = torch.randn(C, device=DEV)
    rows = b.token_rows.long()
    for p_dt, y_dt in ((torch.float16, torch.float16), (torch.float16, torch.float32), (torch.float32, torch.float16)):
        part = (torch.randn(b.R, C, device=DEV) * 4).to(p_dt)
        y = ext.ffn_combine(part, b.token_rows, bias, y_dt)
        assert y.dtype == y_dt
        ref = bias.double() + part.double()[rows].sum(1)
        _one_rounding(y, ref, y_dt, atol=1e-4)


def test_fp16_group_colsum():
    from spt_proto_b200 import ext
    torch.manual_seed(5)
    ptr = torch.tensor([0, 384, 384, 1152, 1280], dtype=torch.int32, device=DEV)
    for C in (520, 2752, 7):
        x = torch.randn(1280, C, device=DEV).half()
        got = ext.group_colsum(x, ptr)
        ref = torch.stack([x[a:b].double().sum(0) for a, b in zip(ptr[:-1].tolist(), ptr[1:].tolist())])
        torch.testing.assert_close(got.double(), ref, atol=1e-3, rtol=1e-5)


@pytest.mark.parametrize("a_dt,b_dt,o_dt", [(torch.float16, torch.float16, torch.float16),
                                            (torch.float32, torch.float32, torch.float16),
                                            (torch.float32, torch.float16, torch.float32),
                                            (torch.float16, torch.float32, torch.float16)])
def test_fp16_scale_add(a_dt, b_dt, o_dt):
    from spt_proto_b200.kernels import ffn as F
    g = torch.Generator(device="cpu").manual_seed(5)
    R, C = 384, 1032
    coeff = torch.rand(R, generator=g).to(DEV).requires_grad_()
    a = torch.randn(R, C, generator=g).to(DEV).to(a_dt).requires_grad_()
    b = torch.randn(R, C, generator=g).to(DEV).to(b_dt).requires_grad_()
    out = F.scale_add(coeff, a, b, o_dt)
    assert out.dtype == o_dt
    cf = coeff.detach().double()[:, None]
    _one_rounding(out, cf * a.detach().double() + b.detach().double(), o_dt)
    go = torch.randn(R, C, generator=g).to(DEV).to(o_dt)
    out.backward(go)
    assert a.grad.dtype == a_dt and b.grad.dtype == b_dt
    _one_rounding(a.grad, cf * go.double(), a_dt)
    assert torch.equal(b.grad, go.to(b_dt))
    torch.testing.assert_close(coeff.grad.double(), (go.double() * a.detach().double()).sum(1), atol=1e-3, rtol=1e-4)


def test_fp16_silu_mul():
    from spt_proto_b200.kernels import ffn as F
    torch.manual_seed(5)
    g = (torch.randn(300, 512, device=DEV) * 2).half().requires_grad_()
    s = torch.randn(300, 512, device=DEV).half().requires_grad_()
    dh = torch.randn(300, 512, device=DEV).half()
    h = F.silu_mul(g, s)
    h.backward(dh)
    assert h.dtype == g.grad.dtype == s.grad.dtype == torch.float16
    gd, sd = g.detach().double().requires_grad_(), s.detach().double().requires_grad_()
    hd = torch.nn.functional.silu(gd) * sd
    hd.backward(dh.double())
    _one_rounding(h, hd.detach(), torch.float16)
    _one_rounding(g.grad, gd.grad, torch.float16)
    _one_rounding(s.grad, sd.grad, torch.float16)


def test_fp16_lora_glu():
    from spt_proto_b200.kernels import ffn as F
    g = torch.Generator(device="cpu").manual_seed(6)
    R, C = 256, 520
    ts = [torch.randn(R, C, generator=g).to(DEV) for _ in range(4)]
    coeff = torch.rand(R, generator=g).to(DEV)
    leaf = [t.clone().requires_grad_() for t in ts]
    cf = coeff.clone().requires_grad_()
    h = F.lora_glu(cf, *leaf, torch.float16)
    assert h.dtype == torch.float16
    ref_in = [t.double().requires_grad_() for t in ts]
    cr = coeff.double().requires_grad_()
    href = torch.nn.functional.silu(cr[:, None] * ref_in[0] + ref_in[1]) * (cr[:, None] * ref_in[2] + ref_in[3])
    _one_rounding(h, href.detach(), torch.float16)
    go = torch.randn(R, C, generator=g).to(DEV).half()
    h.backward(go)
    href.backward(go.double())
    for t, r in zip(leaf, ref_in):
        torch.testing.assert_close(t.grad.double(), r.grad, atol=1e-5, rtol=1e-4)
    torch.testing.assert_close(cf.grad.double(), cr.grad, atol=1e-3, rtol=1e-4)


# ------------------------------------------------------------------------------------------------ layers in .half()
def _oracle(kind, x, P, bs, k, prob):
    """float64 masked-dense restatement of the four layers (oracle/spt_oracle.py routed_ffn ... lora_routed_llama_ffn)
    routed on `prob`, the layer's own router output: an fp16 sigmoid ties values an fp32 one keeps apart.  prob's
    values replace the oracle's straight-through, its gradient flows through the oracle's own sigmoid."""
    from oracle import spt_oracle as O
    x2 = x.reshape(-1, x.size(-1))
    p_own = torch.sigmoid(x2 @ P["router.0.weight"].t() + P["router.0.bias"])
    prob = prob.to(x2) + (p_own - p_own.detach())
    mask = O.route_topk_mask(prob.detach(), k)
    act = {"relu": torch.relu, "gelu": torch.nn.functional.gelu, "silu": torch.nn.functional.silu}[kind[1]]
    if kind[0] == "routed":
        h = act(x2 @ P["fc1.weight"].t() + P["fc1.bias"]) * mask.repeat_interleave(bs, dim=-1).to(x2)
        y = h @ P["fc2.weight"].t() + P["fc2.bias"]
    elif kind[0] == "routed_llama":
        h = act(x2 @ P["gate.weight"].t()) * (x2 @ P["side.weight"].t()) * mask.repeat_interleave(bs, dim=-1).to(x2)
        y = h @ P["down.weight"].t()
    else:
        y = torch.zeros_like(x2)
        for i in range(mask.size(1)):
            sl = slice(i * bs, (i + 1) * bs)
            coeff, m_i = 2.0 * prob[:, i: i + 1], mask[:, i: i + 1].to(x2)
            lora = lambda name, t, rows=sl: (t @ P[name + ".lora.left.weight"]) @ P[name + ".lora.right.weight"][rows].t()
            if kind[0] == "lora":
                h = act(coeff * (x2 @ P["fc1.weight"][sl].t() + P["fc1.bias"][sl]) + lora("fc1", x2))
                y = y + m_i * (coeff * (h @ P["fc2.weight"][:, sl].t())
                               + (h @ P["fc2.lora.left.weight"][sl]) @ P["fc2.lora.right.weight"].t())
            else:
                h = act(coeff * (x2 @ P["gate.weight"][sl].t()) + lora("gate", x2)) * \
                    (coeff * (x2 @ P["side.weight"][sl].t()) + lora("side", x2))
                y = y + m_i * (coeff * (h @ P["down.weight"][:, sl].t())
                               + (h @ P["down.lora.left.weight"][sl]) @ P["down.lora.right.weight"].t())
        if kind[0] == "lora":
            y = y + P["fc2.bias"]
    return y.reshape(x.shape)


_ACTS = {"relu": torch.nn.ReLU, "gelu": torch.nn.GELU, "silu": torch.nn.SiLU}


def _make(kind, d, Fdim, bs, r=16, seed=0):
    """fp32 module with the layer's trainable set; LoRA right factors non-zero so that every gradient is exercised."""
    from spt_proto_b200 import layers
    torch.manual_seed(seed)
    act = _ACTS[kind[1]]()
    if kind[0] == "routed":
        m = layers.RoutedFFN(d_model=d, d_feedforward=Fdim, block_size=bs, activation=act)
    elif kind[0] == "routed_llama":
        m = layers.RoutedLLaMaFFN(d_model=d, d_feedforward=Fdim, block_size=bs, activation=act)
    else:
        cls = layers.LoRARoutedFFN if kind[0] == "lora" else layers.LoRARoutedLLaMaFFN
        m = cls(d_lora=r, block_size=bs, d_model=d, d_feedforward=Fdim, activation=act)
        with torch.no_grad():
            for n, p in m.named_parameters():
                if "lora.right" in n:
                    torch.nn.init.normal_(p, std=0.05)
    return m.to(DEV)


def _run_vs_oracle(m, x, dy, kind, oracle_dev=DEV):
    """-> ({name: relative error}, module) for y, x's gradient and every trainable gradient of m."""
    xg = x.detach().clone().requires_grad_()
    y = m(xg)
    y.backward(dy)
    prob = m.router(xg.detach().reshape(-1, x.size(-1))).detach()
    P = {n: p.detach().to(oracle_dev, torch.float64).requires_grad_(p.requires_grad) for n, p in m.state_dict(keep_vars=True).items()}
    xo = x.detach().to(oracle_dev, torch.float64).requires_grad_()
    yo = _oracle(kind, xo, P, m.block_size, m.k_active, prob.to(oracle_dev))
    yo.backward(dy.to(oracle_dev, torch.float64))
    err = {"y": _rel(y.detach(), yo.detach()), "x": _rel(xg.grad, xo.grad)}
    for n, p in m.named_parameters():
        if not p.requires_grad:
            continue
        if p.grad is None:                    # the router of the plain forms: no gradient on either side
            assert P[n].grad is None, n
            continue
        assert p.grad.dtype == p.dtype, (n, p.grad.dtype)
        err[n] = _rel(p.grad, P[n].grad)
    return err, y


# (kind, shape (d, F, bs, T), bf16 bounds of tests/test_ffn_gpu.py for y, dx, parameter gradients)
_LAYERS = [
    (("routed", "relu"), (128, 1024, 128, 512), (1e-2, 1e-2, 1e-2)),
    (("routed", "gelu"), (128, 1024, 128, 512), (1e-2, 1e-2, 1e-2)),
    (("routed_llama", "silu"), (256, 2048, 256, 1024), (1.5e-2, 1.5e-2, 1.5e-2)),
    (("lora", "relu"), (256, 1024, 256, 1024), (1.5e-2, 2e-2, 3e-2)),
    (("lora_llama", "silu"), (256, 1024, 256, 768), (1.5e-2, 2e-2, 3e-2)),
]


@pytest.mark.parametrize("kind,shape,bounds", _LAYERS, ids=["-".join(c[0]) for c in _LAYERS])
def test_fp16_layer_matches_oracle(kind, shape, bounds):
    """The layer in .half() against the float64 oracle on the same fp16 values: within a quarter of the bf16 bounds,
    gradients in fp16, and at least 4x more accurate than the same module in .bfloat16() against its own oracle
    (fp16 keeps 3 more mantissa bits; a leftover bf16 cast would erase the difference)."""
    d, Fdim, bs, T = shape
    m32 = _make(kind, d, Fdim, bs, seed=T + d)
    x = torch.randn(T, d, device=DEV)
    dy = torch.randn(T, d, device=DEV)
    errs = {}
    for dt in (torch.float16, torch.bfloat16):
        errs[dt], y = _run_vs_oracle(copy.deepcopy(m32).to(dt), x.to(dt), dy.to(dt), kind)
        assert y.dtype == dt
    e16, ebf = errs[torch.float16], errs[torch.bfloat16]
    assert e16["y"] < bounds[0] / 4 and e16["x"] < bounds[1] / 4, e16
    for n, e in e16.items():
        if n not in ("y", "x"):
            assert e < bounds[2] / 4, (n, e16)
    lora = kind[0].startswith("lora")
    assert ("router.0.weight" in e16) == lora, e16      # the router is trained only in the LoRA forms
    assert e16["y"] * 4 <= ebf["y"] and e16["x"] * 4 <= ebf["x"], (e16, ebf)
    assert max(v for n, v in e16.items()) * 4 <= max(v for n, v in ebf.items()), (e16, ebf)


def _exact_router(ffn, gain=4.0):
    """Router whose logits are single products (weight row i = gain * e_i), as in tests/test_ffn_gpu.py."""
    with torch.no_grad():
        w = ffn.router[0].weight
        w.zero_()
        for i in range(w.size(0)):
            w[i, i] = gain
        ffn.router[0].bias.zero_()


@pytest.mark.parametrize("kind,shape,bounds,gain", [
    (("routed", "relu"), (2048, 8192, 1024, 2048), (1e-2, 1e-2, 1e-2), 4.0),
    (("lora_llama", "silu"), (4096, 11008, 2752, 1024), (1.5e-2, 2e-2, 3e-2), 1.0)], ids=["routed-opt1.3b", "lora-llama7b"])
def test_fp16_headline_shapes(kind, shape, bounds, gain):
    """RoutedFFN at the bench.py FFN shape and LoRARoutedLLaMaFFN at configs[3]'s FFN (ragged 2752 blocks), in fp16."""
    d, Fdim, bs, T = shape
    m = _make(kind, d, Fdim, bs, seed=bs)
    _exact_router(m, gain)
    m = m.half()
    x = torch.randn(T, d, device=DEV).half()
    # dy at the scale of a mean loss's gradient: with a unit dy, the LoRA right-factor gradients at d 4096 pass the fp16
    # range (65504), which fp16 training keeps clear of with loss scaling
    dy = (torch.randn(T, d, device=DEV) * 2.0 ** -6).half()
    err, _ = _run_vs_oracle(m, x, dy, kind)
    assert err["y"] < bounds[0] / 4 and err["x"] < bounds[1] / 4, err
    for n, e in err.items():
        if n not in ("y", "x"):
            assert e < bounds[2] / 4, (n, err)


@pytest.mark.parametrize("kind", [("routed", "relu"), ("routed", "gelu"), ("routed_llama", "silu"), ("lora", "relu"),
                                  ("lora_llama", "silu")], ids=lambda k: "-".join(k))
def test_fp16_layer_makes_no_bf16(kind):
    """After forward + backward of a .half() layer the weight-copy cache holds nothing for its parameters, and every
    floating tensor autograd saved is fp16 or fp32."""
    from spt_proto_b200.kernels import ffn as F
    m = _make(kind, 256, 1024, 256).half()
    x = torch.randn(512, 256, device=DEV).half().requires_grad_()
    saved = []

    def pack(t):
        saved.append(t.dtype)
        return t

    with torch.autograd.graph.saved_tensors_hooks(pack, lambda t: t):
        y = m(x)
    y.backward(torch.randn_like(y))
    assert not any(p in F._W16 for p in m.parameters())
    floats = {dt for dt in saved if dt.is_floating_point}
    assert floats and floats <= {torch.float16, torch.float32}, floats


def _lora_step(m, x, dy):
    params = [p for p in m.parameters() if p.requires_grad]
    for p in params:
        p.grad = None
    x.grad = None
    y = m(x)
    y.backward(dy)
    # y is returned detached: a step's autograd graph must not outlive it, or its AccumulateGrad nodes (bound to the
    # stream of that step) would be reused by the next step, and a captured step would then touch the default stream
    return [y.detach(), x.grad] + [p.grad for p in params]


def test_fp16_lora_deterministic_and_graph_capture():
    """Two eager runs of the fp16 LoRARoutedFFN are bit-identical, and its forward + backward captured with
    torch.cuda.graph and replayed twice equals the eager step bit for bit."""
    m = _make(("lora", "relu"), 256, 1024, 256, seed=21).half()
    x = torch.randn(1024, 256, device=DEV).half().requires_grad_()
    dy = torch.randn(1024, 256, device=DEV).half()
    want = [t.detach().clone() for t in _lora_step(m, x, dy)]
    for i, (a, b) in enumerate(zip(_lora_step(m, x, dy), want)):
        assert torch.equal(a, b), i
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            _lora_step(m, x, dy)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = _lora_step(m, x, dy)
    for _ in range(2):
        for t in outs:
            t.detach().zero_()
        graph.replay()
        torch.cuda.synchronize()
        for i, (a, b) in enumerate(zip(outs, want)):
            assert torch.equal(a.detach(), b), i


def test_fp16_opt_block_user_story():
    """An OPT-1.3B-shape block (d 2048, 32 heads, F 8192, ReLU) built dense, upgraded through the four passes, then
    .half(): the attention runs fused, the FFN makes no weight copy, every trainable gradient is fp16 and finite.
    (No value comparison with an fp32 block: the PQ selection of fp16 q / k may differ from fp32 by design.)"""
    from spt_proto_b200 import layers, utils
    from spt_proto_b200.kernels import ffn as F
    torch.manual_seed(13)
    d, H, Fdim = 2048, 32, 8192
    blk = layers.TransformerBlock(d_model=d, n_heads=H, layernorm_fn=torch.nn.LayerNorm(d),
                                  attention_fn=layers.VanillaAttention(d_head=d // H, p_dropout=0.0),
                                  feedforward_fn=layers.Feedforward(d_model=d, d_feedforward=Fdim, p_dropout=0.0,
                                                                    activation=torch.nn.ReLU()),
                                  attention_bias=True, pre_norm=True)
    for stage in ("lora", "ffn", "mha_v1", "mha_v2"):
        blk = utils.ModuleUpgrader(utils.SparseLoRAHandler(d_lora=16, stage=stage, verbose=False)).visit(blk)
    assert isinstance(blk.ffd, layers.LoRARoutedFFN)
    blk = blk.to(DEV).half()
    with torch.no_grad():
        for n, p in blk.named_parameters():
            if "lora.right" in n:
                torch.nn.init.normal_(p, std=0.02)
    x = torch.randn(1, 2048, d, device=DEV).half().requires_grad_()
    y = blk(x)
    y.float().pow(2).mean().backward()
    assert blk.mha.attn_fn.last_path == "fused"
    assert y.dtype == torch.float16 and torch.isfinite(y).all()
    assert not any(p in F._W16 for p in blk.parameters())
    trainable = {n: p for n, p in blk.named_parameters() if p.requires_grad}
    # every trainable parameter gets a gradient, except the PQ codebook, which learns from the layer's separate PQ loss
    assert all(p.grad is not None for n, p in trainable.items() if not n.startswith("mha.attn_fn.quantizer")), \
        [n for n, p in trainable.items() if p.grad is None]
    assert "ffd.router.0.weight" in trainable and "ffd.fc1.lora.left.weight" in trainable
    for n, p in trainable.items():
        if p.grad is not None:
            assert p.grad.dtype == torch.float16, n
            assert torch.isfinite(p.grad).all(), n
