#!/usr/bin/env python
"""One attention layer step (forward + backward of SparseVanillaAttentionV2, reference output layout, bf16, H 32,
sparse_coeff 8 so top-k = S_i / 8) on variable-length samples, at head dims 64, 80 and 128:

    (a) packed:     forward_packed on a seeded mix of lengths (multiples of 32 in [256, 2048], about 8192 tokens)
    (b) padded:     the same samples zero-padded to one S (the longest, rounded up to 128) through forward()
    (c) per_sample: forward() on every sample alone
    (d) equal:      forward_packed on four sequences of 2048 against (d_fixed) forward() at N 4, S 2048

    python scripts/attn_varlen.py --out DIR [--warmup 5] [--steps 20]

Arms alternate step by step; each is the median of --steps CUDA-event-timed steps after --warmup untimed ones.  Writes
one JSON line to DIR/attn_varlen.json (and prints it), with the GPU's name and power limit read in the same process."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from scripts.attn_head80 import _gpu_info  # noqa: E402

H, COEFF, TOKENS = 32, 8, 8192


def _lengths(seed=0):
    g = torch.Generator().manual_seed(seed)
    out = []
    while sum(out) < TOKENS - 256:
        out.append(min(int(torch.randint(8, 65, (1,), generator=g)) * 32, TOKENS - sum(out)))
    return out


def _arms(E: int):
    from spt_proto_b200 import layers
    torch.manual_seed(E)
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0).cuda()
    attn.sparse_coeff = COEFF
    lengths = _lengths()
    T = sum(lengths)
    cu = [0]
    for n in lengths:
        cu.append(cu[-1] + n)
    cu_d = torch.tensor(cu, dtype=torch.int32, device="cuda")
    S_pad = (max(lengths) + 127) // 128 * 128
    bf = dict(device="cuda", dtype=torch.bfloat16)
    q, k, v = (torch.randn(T, H, E, **bf).requires_grad_() for _ in range(3))
    dy = torch.randn(T, H, E, **bf)
    qp, kp, vp = (torch.zeros(len(lengths), S_pad, H, E, **bf) for _ in range(3))
    dyp = torch.zeros(len(lengths), S_pad, H, E, **bf)
    for i, (a, b) in enumerate(zip(cu[:-1], cu[1:])):
        for dst, src in ((qp, q), (kp, k), (vp, v), (dyp, dy)):
            dst[i, :b - a] = src.detach()[a:b]
    qp, kp, vp = (t.requires_grad_() for t in (qp, kp, vp))
    samples = [tuple(t[a:b].detach().unsqueeze(0).requires_grad_() for t in (q, k, v)) + (dy[a:b].unsqueeze(0),)
               for a, b in zip(cu[:-1], cu[1:])]
    q4, k4, v4 = (torch.randn(4, 2048, H, E, **bf).requires_grad_() for _ in range(3))
    dy4 = torch.randn(4, 2048, H, E, **bf)
    cu4 = torch.tensor([0, 2048, 4096, 6144, 8192], dtype=torch.int32, device="cuda")
    q4p, k4p, v4p = (t.detach().view(8192, H, E).requires_grad_() for t in (q4, k4, v4))
    dy4p = dy4.view(8192, H, E)

    def run(fn, *ts):
        for t in ts:
            t.grad = None
        attn.host_trigger = False
        fn()

    arms = {
        "packed": lambda: run(lambda: attn.forward_packed(q, k, v, cu_d, max(lengths)).backward(dy), q, k, v),
        "padded": lambda: run(lambda: attn(qp, kp, vp).backward(dyp), qp, kp, vp),
        "per_sample": lambda: [run(lambda s=s: attn(*s[:3]).backward(s[3]), *s[:3]) for s in samples],
        "equal_packed": lambda: run(lambda: attn.forward_packed(q4p, k4p, v4p, cu4, 2048).backward(dy4p), q4p, k4p, v4p),
        "equal_fixed": lambda: run(lambda: attn(q4, k4, v4).backward(dy4), q4, k4, v4),
    }
    return arms, {"n_samples": len(lengths), "tokens": T, "padded_S": S_pad,
                  "causal_tile_work_padded_over_packed": len(lengths) * S_pad ** 2 / sum(n * n for n in lengths)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for attn_varlen.json")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if args.warmup < 5 or args.steps < 20:
        ap.error("need --warmup >= 5 and --steps >= 20")
    if not torch.cuda.is_available():
        sys.exit("attn_varlen.py measures on the GPU; no CUDA device found")
    res = {"metric": "attn_layer_step_ms", "shape": {"H": H, "sparse_coeff": COEFF, "dtype": "bf16",
                                                    "output_layout": "reference"}, **_gpu_info(), "d_head": {}}
    for E in (64, 80, 128):
        arms, info = _arms(E)
        for _ in range(args.warmup):
            for fn in arms.values():
                fn()
        torch.cuda.synchronize()
        times = {name: [] for name in arms}
        for _ in range(args.steps):
            for name, fn in arms.items():          # arms alternate step by step
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                fn()
                t1.record()
                t1.synchronize()
                times[name].append(t0.elapsed_time(t1))
        med = {name: statistics.median(t) for name, t in times.items()}
        res["d_head"][str(E)] = {**info, "median_ms": med,
                                 "padded_over_packed": med["padded"] / med["packed"],
                                 "per_sample_over_packed": med["per_sample"] / med["packed"],
                                 "equal_packed_over_fixed": med["equal_packed"] / med["equal_fixed"]}
        del arms
        torch.cuda.empty_cache()
    line = json.dumps(res)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "attn_varlen.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
