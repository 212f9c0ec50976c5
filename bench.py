#!/usr/bin/env python
"""bench.py — headline benchmark of the SPT hot path on B200.

Metric (BASELINE.json): sparse-MHA fwd+bwd tokens/s at the OPT-1.3B shape
(configs[1]: 32 heads, d_head 64, seq 2048, bf16, PQ 8 subspaces x 16 codewords, top-k S/8 = 256).
A "step" is one forward+backward pass of SparseVanillaAttentionV2 over one batch of `--seqs`
synthetic sequences per GPU (weak scaling: every rank owns its own sequences; the path has no
collective).  One JSON line is printed by rank 0 — see the keys below.

    python bench.py --gpus 1 --steps 10 --warmup 3
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference          # the CPU port of the reference path (oracle/)
    python bench.py --dump-outputs DIR        # also write the last timed step's y, dq, dk, dv to DIR/<name>.npy

value    : tokens/s, inputs resident in HBM, CUDA-event timed, max over ranks
e2e      : tokens/s through the public layer API with HOST (pinned) buffers: H2D of q,k,v,dO and
           D2H of y,dq,dk,dv inside the timed region; `e2e.host_link` = the pinned-copy bandwidth every
           GPU gets when all N ranks copy at once (measured in the same run) and the e2e ceiling it implies
roofline : dominant kernel group of the step (attention backward), ALGORITHMIC bytes of SURVEY.md
           section 8(d)'s fused-path formula / its CUDA-event time, vs the measured HBM peak in
           MEASURED_PEAKS.json (the bound 8(d) names for the MHA path); the executed dense-tile flops
           fraction, the selected-pair flops fraction and the ncu tensor-pipe reading sit beside it
stages   : the same for every stage kernel (extra key, explains `value`)
mha_plus_ffn : BASELINE.json's metric as worded — one sparse-MHA step + one routed-FFN step (configs[2],
           block 1024) on the same 8192 tokens per GPU, timed together
finetune_step : BASELINE configs[3] (LLaMA-7B-shape 4-layer SPT step, NCCL gradient all-reduce overlapped
           with backward) at this N;  sweep : configs[4] (S 512-8192 x top-k 16-256) at this N
cpu_baseline : the oracle port (torch CPU) on a bounded sample of the same workload, 1 warm-up + median of 5
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

_REAL_STDOUT = sys.stdout

HEADS, D_HEAD, SEQ, M_SUB, N_CODE, D_CODE, COEFF = 32, 64, 2048, 8, 16, 8, 8
METRIC = "sparse_mha_fwd_bwd_tokens_per_s"
UNIT = "tokens/s"
WORKLOAD = "OPT-1.3B-shape sparse MHA fwd+bwd (32 heads, d_head 64, seq 2048, bf16, PQ 8x16, top-k 256)"


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))), "measured"
    return 6650.0, 1590.0, "fallback"


def _traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) and tensor-pipe activity of the top
    kernels at the bench shape, read from the newest committed `ncu --set full` summary (profiles/rN_traffic.json)."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as f:
                return json.load(f)
    return {}


# ---------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md: sample nvidia-smi DURING the timed region)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference path on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_reference_step(heads: int, seed: int = 1234):
    """One fwd+bwd of the reference path (oracle port, torch CPU) on 1 sequence x `heads` heads."""
    from oracle import spt_oracle as O

    g = torch.Generator().manual_seed(seed)
    mk = lambda: torch.randn(1, SEQ, heads, D_HEAD, generator=g).bfloat16().float().requires_grad_()
    q, k, v = mk(), mk(), mk()
    w = torch.randn(M_SUB, N_CODE, D_CODE, generator=g)
    t0 = time.perf_counter()
    y = O.sparse_mha_layer(q, k, v, w, COEFF)
    y.backward(torch.ones_like(y))
    return time.perf_counter() - t0


def base_config(n_seq: int, world: int, fused: bool = True) -> dict:
    """`config` of the line — the same dict on both arms (the reference arm runs a bounded sample of it)."""
    return {"workload": WORKLOAD, "seqs_per_gpu": n_seq, "global_tokens_per_step": n_seq * SEQ * world,
            "l2": "inputs+intermediates per step exceed L2 (>1 GB vs 126 MB); no explicit flush",
            "path": ("fused: pq_encode(q,k) -> lookup(bitmask) -> masked-dense-tile attention fwd/bwd "
                     "(tcgen05 + TMEM + TMA, bf16)" if fused else
                     "stage kernels (pq_encode, lookup, tile index, sddmm / spmm / transposed spmm on dense tiles, softmax)"),
            "pq_train": "off (fwd+bwd of the layer as configs[1] words it; the one-shot PQ loss the reference's "
                        "training loop arms per step is part of the finetune_step section)",
            "output_layout": "reference (the shipped layer's [N*H, E, S] memory viewed as [N, S, H, E])",
            "parallelism": f"dp{world} (batch x head sharded, no collective)"}


def run_reference(args):
    """Reference arm: the reference's path on the host cores.  The reference's own implementation is CUDA-only
    (its CPU form is exactly the oracle port, oracle/spt_oracle.py), so this times the port with every host
    thread, `--steps` timed steps after `--warmup` warm-ups, each step a bounded sample (1 sequence x
    `--ref-heads` of the 32 heads) of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    heads = args.ref_heads
    steps, warmup = args.steps, args.warmup
    for _ in range(warmup):
        cpu_reference_step(heads)
    times = [cpu_reference_step(heads) for _ in range(steps)]
    t = statistics.median(times)
    tokens = SEQ * heads / HEADS            # a step of h of the 32 heads is h/32 of a sequence
    value = tokens / t
    sample = (f"1 sequence x {heads} of {HEADS} heads per step (S={SEQ}, d={D_HEAD}), fp32, oracle port (torch CPU), "
              f"median of {len(times)} steps after {warmup} warm-ups")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": base_config(args.seqs, max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


# ---------------------------------------------------------------------------------------------------
# stage micro-timings -> roofline
# ---------------------------------------------------------------------------------------------------
def _time_cuda(fn, iters=5, warm=2, prequeue=True):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # a short device-side spin queued ahead of the start event lets the host enqueue fn's launches while the
        # GPU is still busy, so a multi-kernel stage is timed without host launch gaps (8 ranks share the host cores)
        if prequeue:
            torch.cuda._sleep(400_000)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return statistics.median(ts)


def _time_back_to_back(fn, iters=10, warm=3):
    """Average device time of `iters` calls launched back to back behind a short device-side spin (no sync between
    them): the steady state of a loop whose host side runs ahead of the GPU."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(2_000_000)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e-3 / iters


FUSED_PATH = ["pq_encode", "lookup_mask", "attn_fwd", "attn_bwd"]
# what bounds each kernel according to its ncu capture (profiles/README.md, DESIGN.md section 4): the HBM fraction
# reported beside it is NOT the target for the issue-bound ones
STAGE_BOUND = {
    "attn_fwd": "exp unit (one ex2 per score element: 512 clk per 128x64 tile, loop at 702) + per-CTA prologue / epilogue; tensor pipe 24 % active",
    "attn_bwd": "element math (XU, ALU and issue all near saturation in the math phase) + MMA<->math-warp handshake latency of the single chain per CTA; tensor pipe 31 % active (128x128 tiles, N=128 score MMAs)",
    "pq_encode": "fp32-add issue (L1 distances, packed FADD2); DRAM = algorithmic bytes",
    "lookup_mask": "integer issue (bit-sliced adder tree + selection)",
    "lookup": "integer issue + index write",
    "sddmm": "instruction issue per gathered pair (not L2)",
    "spmm": "instruction issue per gathered pair (not L2)",
    "spmm_t": "instruction issue per gathered pair (not L2)",
    "softmax_fwd": "hbm",
    "softmax_bwd": "hbm",
    "csr2csc": "shared-memory bit-matrix build + scan per 64-row tile (one CTA of 1024 threads per SM); index read + write",
    "csr_tiles": "two passes over the indices (count, place) with shared-memory histograms over the column tiles",
    "sddmm_tiles": "LSU data pipe: one index word read + one 4-byte store per entry, score tile through shared memory",
    "spmm_tiles": "LSU data pipe: one value gather per entry + tile scatter / fragment loads",
    "spmm_t_tiles": "LSU data pipe: one value gather per entry + tile scatter / fragment loads; latency of the first column tile's long buckets",
}
STAGE_PATH = ["pq_encode", "lookup", "sddmm_tiles", "softmax_fwd", "spmm_tiles", "softmax_bwd", "csr_tiles", "spmm_t_tiles"]


def stage_roofline(n_seq: int, dev, hbm_gbs: float, tensor_tflops: float):
    """Times every stage kernel of the step on the bench shapes (inputs >> L2: B = n_seq*32 heads) and
    reports algorithmic bytes (SURVEY.md section 8d formulas; e = 2 for bf16) / time."""
    from spt_proto_b200 import ext

    B, S, d, k, m, e = n_seq * HEADS, SEQ, D_HEAD, SEQ // COEFF, M_SUB, 2
    g = torch.Generator(device="cpu").manual_seed(7)
    q = torch.randn(B, S, d, generator=g).to(dev, torch.bfloat16)
    kk = torch.randn(B, S, d, generator=g).to(dev, torch.bfloat16)
    v = torch.randn(B, S, d, generator=g).to(dev, torch.bfloat16)
    w = torch.randn(m, N_CODE, D_CODE, generator=g).to(dev)
    qc, kc = ext.pq_encode(q, w), ext.pq_encode(kk, w)
    cfg = torch.empty([COEFF], device="meta")
    idx = ext.lookup_forward_cuda(cfg, qc, kc).flatten(1)
    indptr = torch.arange(0, k * S + 1, k, dtype=torch.int32, device=dev)
    vals = ext.sddmm_forward_cuda(False, True, indptr, idx, q, kk)
    sc = torch.clamp(vals * d ** -0.5, -10, 10)
    p = ext.softmax_forward_cuda(indptr, idx, sc)
    csc = ext.csr2csc(indptr, idx)
    tiles = ext.csr_tiles(indptr, idx)
    dy = torch.randn(B, S, d, generator=g).to(dev, torch.bfloat16)
    Sd, Sk = S * d * e, S * k * 4
    stages = {
        # name: (callable, algorithmic bytes per head)
        "pq_encode": (lambda: ext.pq_encode_pair(q, kk, w), 2 * (Sd + S * m * 4)),     # q and k in one launch
        "lookup": (lambda: ext.lookup_forward_cuda(cfg, qc, kc), 2 * S * m * 4 + Sk),
        "sddmm": (lambda: ext.sddmm_forward_cuda(False, True, indptr, idx, q, kk), 2 * Sd + 2 * Sk),
        "softmax_fwd": (lambda: ext.softmax_forward_cuda(indptr, idx, sc), 3 * Sk),
        "spmm": (lambda: ext.spmm_forward_cuda(False, False, indptr, idx, p, v), 2 * Sk + 2 * Sd),
        "softmax_bwd": (lambda: ext.softmax_backward_cuda(indptr, idx, p, sc), 4 * Sk),
        "csr2csc": (lambda: ext.csr2csc(indptr, idx), 4 * Sk + S * 4),
        "spmm_t": (lambda: ext.spmm_csc(csc, p, dy), 3 * Sk + 2 * Sd),
        # what the bf16 stage path runs instead of the two rows above: the tile index (indices read, one word per entry
        # written) and the transposed product on it (entry word + value per entry, x read, y written)
        "csr_tiles": (lambda: ext.csr_tiles(indptr, idx), 2 * Sk + S * 4),
        "spmm_t_tiles": (lambda: ext.spmm_tiles(tiles, p, dy), 2 * Sk + 2 * Sd),
        "spmm_tiles": (lambda: ext.spmm_tiles(tiles, p, v, trans=False), 2 * Sk + 2 * Sd),
        "sddmm_tiles": (lambda: ext.sddmm_tiles(tiles, q, kk, d ** -0.5, 10.0), 2 * Sd + 2 * Sk),
    }
    mask, extra0, _ = ext.lookup_mask(qc, kc, COEFF)
    y_f, z_f = ext.sparse_attn_fwd(q, kk, v, mask, extra0, d ** -0.5)
    stages["lookup_mask"] = (lambda: ext.lookup_mask(qc, kc, COEFF), 2 * S * m * 4 + S * S // 8 + S * 4)
    out = {}
    T = S // 64
    tile_flops = (T * (T + 1) // 2) * 2 * 64 * 64 * 64          # one causal dense GEMM over a head
    sparse_flops = 2 * S * k * d                                 # one selected-pair product over a head
    # SURVEY.md 8(d), fused-path formula (per head): fwd reads q,k,v,idx and writes o,P; bwd reads idx,P,q,k,v,dO
    # and writes dq,dk,dv.  (The kernels move LESS than this: the selection travels as a bitmask, P is recomputed.)
    fused_bytes = {"attn_fwd": 4 * Sd + 2 * Sk, "attn_bwd": 2 * Sk + 7 * Sd}
    for name, fn, n_gemm in (("attn_fwd", lambda: ext.sparse_attn_fwd(q, kk, v, mask, extra0, d ** -0.5), 2),
                             ("attn_bwd", lambda: ext.sparse_attn_bwd(q, kk, v, y_f, dy, mask, extra0, z_f, d ** -0.5), 7)):
        t = _time_cuda(fn)
        tf = n_gemm * tile_flops * B / t / 1e12
        n_sparse = 2 if name == "attn_fwd" else 6
        gbs = fused_bytes[name] * B / t / 1e9
        out[name] = {"ms": t * 1e3, "algorithmic_GB": fused_bytes[name] * B / 1e9, "achieved_GBps": gbs,
                     "frac_hbm": gbs / hbm_gbs,
                     "executed_dense_GFLOP": n_gemm * tile_flops * B / 1e9, "executed_dense_TFLOPs": tf,
                     "executed_frac_tensor": tf / tensor_tflops,
                     "algorithmic_sparse_TFLOPs": n_sparse * sparse_flops * B / t / 1e12,
                     "selected_pair_frac_tensor": n_sparse * sparse_flops * B / t / 1e12 / tensor_tflops,
                     "bound": STAGE_BOUND[name]}
    for name, (fn, bytes_per_head) in stages.items():
        t = _time_cuda(fn)
        gbs = bytes_per_head * B / t / 1e9
        out[name] = {"ms": t * 1e3, "algorithmic_GB": bytes_per_head * B / 1e9, "achieved_GBps": gbs,
                     "frac_hbm": gbs / hbm_gbs, "bound": STAGE_BOUND.get(name, "hbm")}
    return out


def ffn_bench(dev, tensor_tflops: float):
    """BASELINE configs[2]: OPT-1.3B-shape routed FFN (d 2048, ffn 8192, half the blocks active) fwd+bwd
    with weight gradients, T = 8192 tokens, bf16, grouped GEMM on tcgen05.  Reported beside the headline."""
    from spt_proto_b200 import layers
    out = {}
    for bs in (1024, 2048):
        torch.manual_seed(4321)
        d, F, T = 2048, 8192, 8192
        ffn = layers.RoutedFFN(d_model=d, d_feedforward=F, block_size=bs, activation=torch.nn.ReLU()).to(dev).bfloat16()
        x = torch.randn(16, T // 16, d, device=dev).bfloat16().requires_grad_()
        dy = torch.randn(16, T // 16, d, device=dev).bfloat16()

        def step():
            x.grad = None
            for p in ffn.parameters():
                p.grad = None
            ffn(x).backward(dy)

        # eager, two readings: `isolated` = one step launched into an idle GPU and waited for (host launch time of
        # ~25 launches + autograd shows in full), `steady` = ten steps launched back to back the way a training loop
        # runs them (the host stays ahead of the device; what is left are the device-side gaps between ~25 kernels).
        t_isolated = _time_cuda(step, iters=5, warm=3, prequeue=False)
        t_eager = _time_back_to_back(step, iters=10, warm=3)
        # Routing and bucketing are device-side (no host sync), so the whole forward + backward is capturable:
        # replay one CUDA graph.
        t, graphed = t_eager, False
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step()
            t, graphed = _time_cuda(graph.replay, iters=5, warm=3), True
        except Exception as exc:   # keep the eager number, say why
            print(f"[bench] routed FFN graph capture failed: {exc!r}", file=sys.stderr)
            torch.cuda.synchronize()
        flops = 12 * T * 0.5 * F * d          # fwd 4 T rho F d, bwd dX 4 ..., bwd dW 4 ... (SURVEY.md 8d)
        out[f"block_{bs}"] = {"ms": t * 1e3, "ms_eager": t_eager * 1e3, "ms_eager_isolated": t_isolated * 1e3,
                              "cuda_graph": graphed, "tokens_per_s": T / t,
                              "algorithmic_TFLOPs": flops / t / 1e12,
                              "frac_tensor": flops / t / 1e12 / tensor_tflops, "T": T, "d": d, "ffn": F,
                              "n_blocks": F // bs, "active": (F // bs) // 2}
    return out


# ---------------------------------------------------------------------------------------------------
# extra sections (all ranks take part; every time is the max over ranks)
# ---------------------------------------------------------------------------------------------------
def _max_over_ranks(values, dev, world):
    if world == 1:
        return list(values)
    import torch.distributed as dist
    t = torch.tensor(list(values), device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def mha_plus_ffn_bench(mha_step, n_seq, dev, world, barrier, steps):
    """BASELINE.json's metric as worded: sparse MHA fwd+bwd + routed FFN fwd+bwd (configs[2]: d 2048, ffn 8192,
    block 1024, half the blocks active, weight gradients included) on the SAME n_seq*2048 tokens per GPU, one after
    the other in one timed loop.  The FFN step is a replayed CUDA graph when capture succeeds (its ~45 launches are
    otherwise Python-bound)."""
    from spt_proto_b200 import layers
    torch.manual_seed(4321)
    d, F, bs, T = 2048, 8192, 1024, n_seq * SEQ
    ffn = layers.RoutedFFN(d_model=d, d_feedforward=F, block_size=bs, activation=torch.nn.ReLU()).to(dev).bfloat16()
    x = torch.randn(n_seq, SEQ, d, device=dev).bfloat16().requires_grad_()
    dyf = torch.randn(n_seq, SEQ, d, device=dev).bfloat16()

    def ffn_step():
        x.grad = None
        for p in ffn.parameters():
            p.grad = None
        ffn(x).backward(dyf)

    for _ in range(3):
        ffn_step()
    run_ffn, graphed = ffn_step, False
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            ffn_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            ffn_step()
        run_ffn, graphed = graph.replay, True
    except Exception as exc:
        print(f"[bench] routed FFN graph capture failed: {exc!r}", file=sys.stderr)
        torch.cuda.synchronize()
    for _ in range(2):
        mha_step()
        run_ffn()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        mha_step()
        run_ffn()
    ev[1].record()
    barrier()
    (t,) = _max_over_ranks([ev[0].elapsed_time(ev[1]) * 1e-3 / steps], dev, world)
    flops = 12 * T * 0.5 * F * d
    return {"value": T * world / t, "unit": UNIT, "ms_per_step": t * 1e3, "steps": steps, "tokens_per_gpu_per_step": T,
            "ffn": {"d_model": d, "d_ff": F, "block": bs, "active_blocks": (F // bs) // 2, "cuda_graph": graphed,
                    "algorithmic_GFLOP_per_step": flops / 1e9},
            "note": "one MHA step (configs[1]) + one routed-FFN step (configs[2]) on the same tokens, back to back"}


def sweep_bench(dev, rank, world, barrier, iters=3):
    """BASELINE configs[4]: S 512-8192 x top-k 16-256, fwd+bwd tokens/s (32 heads x d 64, bf16, 8192 tokens/GPU/step)."""
    from spt_proto_b200 import layers
    attn = layers.SparseVanillaAttentionV2(d_head=D_HEAD, d_codeword=D_CODE, n_codewords=N_CODE, p_dropout=0.0).to(dev)
    attn.host_trigger = False
    torch.manual_seed(99 + rank)
    rows = []
    for S in (512, 1024, 2048, 4096, 8192):
        n_seq = max(1, 8192 // S)
        q, k, v = (torch.randn(n_seq, S, HEADS, D_HEAD, device=dev).bfloat16().requires_grad_() for _ in range(3))
        dy = torch.randn(n_seq, S, HEADS, D_HEAD, device=dev).bfloat16()
        for topk in (16, 32, 64, 128, 256):
            attn.sparse_coeff = S // topk

            def step():
                q.grad = k.grad = v.grad = None
                attn(q, k, v).backward(dy)

            for _ in range(2):
                step()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                step()
            b.record()
            torch.cuda.synchronize()
            (t,) = _max_over_ranks([a.elapsed_time(b) * 1e-3 / iters], dev, world)
            rows.append({"S": S, "top_k": topk, "ms_per_step": round(t * 1e3, 4), "tokens_per_s": n_seq * S * world / t,
                         "path": attn.last_path})
        del q, k, v, dy
    return rows


DUMP_BYTES = 32 << 20       # float32 bytes over all dumped arrays; at the bench shape every output is sampled


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes every array as out_dir/<name>.npy in float32.  One larger than its share of DUMP_BYTES is reduced to
    the elements at a fixed sample of flat positions (seeded, ascending, the same on every run), so the files of two
    builds can be compared element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n_max = DUMP_BYTES // 4 // len(arrays)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > n_max:
            pos = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:n_max].sort().values
            t = t.reshape(-1)[pos.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------
# main arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    from spt_proto_b200 import ext, host_io, layers

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — spt_proto_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = host_io.bind_to_gpu_numa(local)      # before any pinned allocation (first touch decides the node)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    hbm_gbs, tensor_tflops, peak_kind = _peaks()

    n_seq = args.seqs
    torch.manual_seed(1234 + rank)
    attn = layers.SparseVanillaAttentionV2(d_head=D_HEAD, d_codeword=D_CODE, n_codewords=N_CODE, p_dropout=0.0).to(dev)
    attn.sparse_coeff = COEFF
    attn.use_fused = not args.stage_path
    attn.host_trigger = False    # fwd+bwd of the layer (configs[1]): PQ loss not armed, decided on the host (no D2H sync)
    shape = (n_seq, SEQ, HEADS, D_HEAD)
    q = torch.randn(shape, device=dev).bfloat16().requires_grad_()
    k = torch.randn(shape, device=dev).bfloat16().requires_grad_()
    v = torch.randn(shape, device=dev).bfloat16().requires_grad_()
    dy = torch.randn(shape, device=dev).bfloat16()

    def step():
        q.grad = k.grad = v.grad = None
        y = attn(q, k, v)
        y.backward(dy)
        return y

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled (nvidia-smi, 100 ms period) from the warm-up to the end of the e2e loop: the timed
    # region itself lasts only K x ~1 ms, less than one sampling period for small K
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # the stage path needs 6 untimed steps: its CSR->CSC cache (4 patterns) and the caching allocator only reach their
    # steady state after the fifth step (steps 4 and 5 take 31 / 17 ms of host time against 8.8 ms afterwards)
    n_warm = max(args.warmup, 6 if not attn.use_fused else 3)
    for _ in range(n_warm):
        step()
    barrier()
    launches0 = ext.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # the steps are launched eagerly (autograd, ~10 launches per step): a short device-side spin queued AHEAD of the start
    # event lets the host get one step ahead, so the timed region sees the steady state of the launch queue from its first
    # step on (without it the first step of K contains the host's start-up latency: 0.5 - 1 % of a 10-step region)
    torch.cuda._sleep(1_000_000)
    a.record()
    for _ in range(args.steps):
        y = step()
    b.record()
    barrier()
    elapsed = a.elapsed_time(b) * 1e-3
    launches = ext.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"y": y, "dq": q.grad, "dk": k.grad, "dv": v.grad})

    # ---- e2e: host (pinned) buffers in, host buffers out, through the public layer API ---------------
    # chunk-major pinned buffers: the four operands of a sequence are contiguous, one copy per chunk and direction
    s_in = host_io.alloc_host(n_seq, shape[1:], torch.bfloat16, chunk=1)
    s_out = host_io.alloc_host(n_seq, shape[1:], torch.bfloat16, chunk=1)
    for j, t in enumerate((q, k, v, dy)):
        host_io.fill_operand(s_in, j, t.detach().cpu())
    pipe = host_io.HostPipeline(attn, dev, chunk=1)     # per-sequence chunks: H2D / kernels / D2H overlap

    def step_e2e():
        pipe.run_stacked(s_in, s_out)

    for _ in range(4):     # the first passes over the pinned buffers on a fresh box run at 80 % of the steady link rate
        step_e2e()
    pipe.finish()
    barrier()
    e2e_steps = max(4, args.steps)
    a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a2.record()
    for _ in range(e2e_steps):
        step_e2e()      # consecutive steps stream through the pipeline (no stall between them) ...
    pipe.finish()       # ... and the timed region ends only when the last result has landed in host memory
    b2.record()
    barrier()
    elapsed_e2e = a2.elapsed_time(b2) * 1e-3
    clocks = sampler.stop() if rank == 0 else None
    elapsed, elapsed_e2e = _max_over_ranks([elapsed, elapsed_e2e], dev, world)

    # what the host fabric gives every GPU when all N ranks copy at once (both directions): the e2e ceiling at this N
    link = host_io.measure_host_link(dev, barrier=barrier)
    link_min = [-x for x in _max_over_ranks([-link["h2d_GBps_duplex"], -link["d2h_GBps_duplex"]], dev, world)]

    tokens_per_step = n_seq * SEQ * world
    value = tokens_per_step * args.steps / elapsed
    e2e_value = tokens_per_step * e2e_steps / elapsed_e2e
    tensor_bytes = n_seq * SEQ * HEADS * D_HEAD * 2
    link_ceiling = tokens_per_step / max(4 * tensor_bytes / (link_min[0] * 1e9), 4 * tensor_bytes / (link_min[1] * 1e9))

    combined = mha_plus_ffn_bench(step, n_seq, dev, world, barrier, max(3, args.steps // 2)) if attn.use_fused else None
    finetune = None
    if not args.no_finetune and attn.use_fused:
        try:
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            import finetune_step
            finetune = finetune_step.run(dev, rank, world, steps=3, warmup=2, seq=2048, batch=1, graph=True)
        except Exception as exc:      # keep the headline; say what failed
            finetune = {"error": repr(exc)}
            print(f"[bench] finetune_step section failed: {exc!r}", file=sys.stderr)
        torch.cuda.empty_cache()
    sweep = sweep_bench(dev, rank, world, barrier) if (not args.no_sweep and attn.use_fused) else None

    if rank == 0:
        stages = stage_roofline(n_seq, dev, hbm_gbs, tensor_tflops)
        on_path = FUSED_PATH if attn.use_fused else STAGE_PATH
        dom = max(on_path, key=lambda s: stages[s]["ms"])
        st = stages[dom]
        roof = {"bound": "hbm", "kernel": dom, "achieved": st["achieved_GBps"], "peak": hbm_gbs, "unit": "GB/s",
                "frac": st["frac_hbm"], "traffic": None, "peak_source": peak_kind,
                "algorithmic_bytes_per_launch": st["algorithmic_GB"] * 1e9,
                "formula": "SURVEY.md 8(d) fused-path bytes per head x heads / CUDA-event time of the kernel group / "
                           "measured HBM peak (the bound 8(d) names for the MHA path)"}
        if "executed_frac_tensor" in st:
            roof["formula"] += ("; attn_bwd per head = idx S*k*4 + P S*k*4 + (q,k,v,dO read + dq,dk,dv written) 7*S*d*2; "
                                "attn_fwd = q,k,v,o 4*S*d*2 + idx,P 2*S*k*4")
            roof["executed_frac"] = st["executed_frac_tensor"]          # executed dense-causal-tile flops / bf16 peak
            roof["selected_pair_tensor_frac"] = st["selected_pair_frac_tensor"]
            roof["note"] = ("the kernels compute masked dense causal tiles (7 GEMMs in the backward), 1/4 of whose entries "
                            "are selected pairs; executed_frac counts all of them, selected_pair_tensor_frac only the "
                            "2*S*k*d products the stage API defines")
        traffic = _traffic().get(dom)
        if traffic is not None:
            roof["traffic"] = traffic["dram_bytes_per_launch"]
            roof["traffic_source"] = traffic["source"]
            if "tensor_pipe_active_pct" in traffic:
                roof["ncu_tensor_pipe_active_pct"] = traffic["tensor_pipe_active_pct"]
        step_bytes = sum(stages[s]["algorithmic_GB"] for s in on_path) * 1e9
        step_roof = {"algorithmic_bytes_per_step": step_bytes, "achieved_GBps": step_bytes / (elapsed / args.steps) / 1e9,
                     "frac_hbm": step_bytes / (elapsed / args.steps) / 1e9 / hbm_gbs,
                     "note": "whole step vs the fused-path formula of SURVEY.md 8(d) (~13.5 MiB per head)"}
        cpu = None
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            cpu_reference_step(args.ref_heads)                                   # 1 warm-up
            t_cpu = statistics.median(cpu_reference_step(args.ref_heads) for _ in range(5))
            cpu = {"value": SEQ * args.ref_heads / HEADS / t_cpu, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"1 sequence x {args.ref_heads} of {HEADS} heads, fwd+bwd, fp32, oracle port (torch CPU), "
                             "1 warm-up + median of 5"}
        gpu_ref = gpu_reference_baseline(dev) if args.stage_path else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": elapsed / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": base_config(n_seq, world, attn.use_fused),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 4 * tensor_bytes,
                    "d2h_bytes_per_step": 4 * tensor_bytes, "steps": e2e_steps,
                    "copies_per_step": {"h2d": n_seq, "d2h": n_seq},
                    "host_link": {"min_over_ranks_h2d_GBps": link_min[0], "min_over_ranks_d2h_GBps": link_min[1],
                                  "rank0": link, "numa": numa,
                                  "ceiling_tokens_per_s": link_ceiling, "frac_of_ceiling": e2e_value / link_ceiling,
                                  "note": "pinned-copy bandwidth per GPU with all ranks copying both ways at once, "
                                          "measured in this run; ceiling = tokens per step / time to move the step's bytes"}},
            "gpu_launches": launches,
            "timing": ("CUDA events around exactly K eagerly launched steps, barrier + synchronize on both sides, max over "
                       "ranks; a 0.5 ms device-side spin is queued ahead of the start event so that the host is one step "
                       "ahead when the region starts (steady-state launch queue)"),
            "roofline": roof,
            "step_roofline": step_roof,
            "mha_plus_ffn": combined,
            "mha_plus_ffn_tokens_per_s": None if combined is None else combined["value"],
            "finetune_step": finetune,
            "sweep": sweep,
            "stages": stages,
            "routed_ffn": ffn_bench(dev, tensor_tflops),
            "cpu_baseline": cpu,
        }
        if gpu_ref is not None:
            line["gpu_reference_baseline"] = gpu_ref
        print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


def gpu_reference_baseline(dev):
    """Same-box GPU baseline (BASELINE.md section 4): the UNMODIFIED reference extension (oracle/_ref/ext_ref.so:
    its SIMT cdist / lookup / softmax kernels + cuSPARSE SDDMM / SpMM) timed stage by stage at the largest shape it
    supports — fp32, S 1024, top-k 128 — beside this repo's stage kernels on the same tensors.  Reported only."""
    import importlib.util
    path = os.path.join(ROOT, "oracle", "_ref", "ext_ref.so")
    if not os.path.exists(path):
        return {"unavailable": "oracle/_ref/ext_ref.so not built"}
    try:
        spec = importlib.util.spec_from_file_location("ext_ref", path)
        ref = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(ref)
    except Exception as exc:
        return {"unavailable": repr(exc)}
    from spt_proto_b200 import ext
    B, S, d, m, coeff = 128, 1024, D_HEAD, M_SUB, COEFF
    k = S // coeff
    g = torch.Generator(device="cpu").manual_seed(11)
    q, kk, v, dyy = (torch.randn(B, S, d, generator=g).to(dev) for _ in range(4))
    w = torch.randn(m, N_CODE, D_CODE, generator=g).to(dev)
    zq = q.view(B * S, m, D_CODE).transpose(0, 1).contiguous()
    zk = kk.view(B * S, m, D_CODE).transpose(0, 1).contiguous()
    qc = ext.cdist_forward_cuda(zq, w)[1].t().contiguous().view(B, S, m)
    kc = ext.cdist_forward_cuda(zk, w)[1].t().contiguous().view(B, S, m)
    cfg = torch.empty([coeff], device="meta")
    cfg_ref = torch.empty([coeff])
    idx = ext.lookup_forward_cuda(cfg, qc, kc).flatten(1)
    indptr = torch.arange(0, k * S + 1, k, dtype=torch.int32, device=dev)
    f, t_ = torch.scalar_tensor(False), torch.scalar_tensor(True)
    vals = ext.sddmm_forward_cuda(f, t_, indptr, idx, q, kk)
    sc = torch.clamp(vals * d ** -0.5, -10, 10)
    p = ext.softmax_forward_cuda(indptr, idx, sc)
    pairs = [
        ("cdist", lambda: ext.cdist_forward_cuda(zq, w), lambda: ref.cdist_forward_cuda(zq, w)),
        ("lookup", lambda: ext.lookup_forward_cuda(cfg, qc, kc), lambda: ref.lookup_forward_cuda(cfg_ref, qc, kc)),
        ("sddmm", lambda: ext.sddmm_forward_cuda(f, t_, indptr, idx, q, kk),
         lambda: ref.sddmm_forward_cuda(f, t_, indptr, idx, q, kk)),
        ("softmax_fwd", lambda: ext.softmax_forward_cuda(indptr, idx, sc), lambda: ref.softmax_forward_cuda(indptr, idx, sc)),
        ("softmax_bwd", lambda: ext.softmax_backward_cuda(indptr, idx, p, sc),
         lambda: ref.softmax_backward_cuda(indptr, idx, p, sc)),
        ("spmm", lambda: ext.spmm_forward_cuda(f, f, indptr, idx, p, v), lambda: ref.spmm_forward_cuda(f, f, indptr, idx, p, v)),
        ("spmm_t (dK/dV form)", lambda: ext.spmm_forward_cuda(t_, f, indptr, idx, p, dyy),
         lambda: ref.spmm_forward_cuda(t_, f, indptr, idx, p, dyy)),
    ]
    out = {"shape": f"fp32, B {B} heads, S {S}, d {d}, top-k {k} (the largest the reference kernels are instantiated for)",
           "stages": {}}
    for name, ours, theirs in pairs:
        row = {}
        try:
            row["ours_ms"] = _time_cuda(ours) * 1e3
        except Exception as exc:
            row["ours_error"] = repr(exc)
        try:
            row["reference_ms"] = _time_cuda(theirs) * 1e3
        except Exception as exc:
            row["reference_error"] = repr(exc)
        if "ours_ms" in row and "reference_ms" in row:
            row["speedup"] = row["reference_ms"] / row["ours_ms"]
        out["stages"][name] = row
    return out


def main():
    # the contract is ONE JSON line on stdout: libraries (NCCL prints its version banner there) get
    # stderr, the line goes to the saved descriptor
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seqs", type=int, default=4, help="sequences per GPU per step")
    ap.add_argument("--ref-heads", type=int, default=8, help="heads in the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--stage-path", action="store_true", help="run the reference-style stage kernels, not the fused path")
    ap.add_argument("--no-finetune", action="store_true", help="skip the configs[3] fine-tuning-step section")
    ap.add_argument("--no-sweep", action="store_true", help="skip the configs[4] sweep section")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write y, dq, dk, dv of the last timed step (rank 0) as DIR/<name>.npy, float32, a fixed "
                         "seeded sample of each (32 MiB in all); GPU path only, refused with --impl reference")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
