#!/usr/bin/env python
"""Grouped-query attention on the fused path: one SparseVanillaAttentionV2 layer step (forward + backward, reference
output layout, sparse_coeff 8), three variants per shape, timed alternately step by step in one process:
  gqa     k, v with Hkv heads, passed as they are (native grouped-query path);
  repeat  the same k, v repeated to H heads with torch.repeat_interleave inside the timed step (the workaround: its
          autograd backward sums the repeated gradients);
  mha     multi-head attention with Hkv = H (k, v with H heads of their own).

    python scripts/attn_gqa.py --out DIR [--warmup 3] [--steps 20]

Shapes: the LLaMA-3-8B attention (H 32, Hkv 8, d 128) at S 2048 (N 4) and S 8192 (N 1), and an MQA point (H 32, Hkv 1,
d 64, S 2048, N 4); bf16.  Each number is the median of --steps CUDA-event-timed steps after --warmup untimed ones;
max_memory_allocated is the peak of one step of the variant alone (reset before it), with the inputs allocated.  Writes
one JSON line per case to DIR/attn_gqa.jsonl (and prints it); the first line holds the GPU's name and power limit, read
in the same process."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from attn_long import _gpu_info  # noqa: E402

SHAPES = [  # (N, S, H, Hkv, d)
    (4, 2048, 32, 8, 128),
    (1, 8192, 32, 8, 128),
    (4, 2048, 32, 1, 64),
]


def _variants(N, S, H, Hkv, E):
    from spt_proto_b200 import layers
    torch.manual_seed(S + Hkv + E)
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0).cuda()
    attn.host_trigger = False
    G = H // Hkv
    mk = lambda h: torch.randn(N, S, h, E, device="cuda", dtype=torch.bfloat16).requires_grad_()
    q, k, v, k_mha, v_mha = mk(H), mk(Hkv), mk(Hkv), mk(H), mk(H)
    dy = torch.randn(N, S, H, E, device="cuda", dtype=torch.bfloat16)

    def run(kk, vv, repeat):
        def step():
            for t in (q, kk, vv):
                t.grad = None
            k_in, v_in = (kk.repeat_interleave(G, 2), vv.repeat_interleave(G, 2)) if repeat else (kk, vv)
            attn(q, k_in, v_in).backward(dy)
            assert attn.last_path == "fused", attn.last_path
        return step

    return {"gqa": run(k, v, False), "repeat": run(k, v, True), "mha": run(k_mha, v_mha, False)}


def _case(N, S, H, Hkv, E, warmup: int, steps: int):
    fns = _variants(N, S, H, Hkv, E)
    peak = {}
    for name, fn in fns.items():
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        peak[name] = torch.cuda.max_memory_allocated()
    times = {name: [] for name in fns}
    for _ in range(steps):
        for name, fn in fns.items():            # alternating: one step of each variant per round
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b))
    out = {"N": N, "S": S, "H": H, "Hkv": Hkv, "d": E, "dtype": "bfloat16"}
    for name in fns:
        out[f"{name}_ms"] = round(statistics.median(times[name]), 3)
        out[f"{name}_max_mem_mib"] = round(peak[name] / 2 ** 20, 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    lines = [dict(_gpu_info(), sparse_coeff=8, layout="reference", warmup=args.warmup, steps=args.steps)]
    print(json.dumps(lines[0]), flush=True)
    for shape in SHAPES:
        lines.append(_case(*shape, args.warmup, args.steps))
        print(json.dumps(lines[-1]), flush=True)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "attn_gqa.jsonl"), "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
