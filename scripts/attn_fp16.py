#!/usr/bin/env python
"""One attention layer step (forward + backward of SparseVanillaAttentionV2, reference output layout, fused path) in
fp16 against the same step in bf16, at head dims 64, 80 and 128.

    python scripts/attn_fp16.py --out DIR [--warmup 5] [--steps 20]

Shape: N 4, S 2048, H 32, sparse_coeff 8 (top-k 256), random q, k, v and dO.  For each head dim the two dtypes are timed
alternately, step by step (bf16, fp16, bf16, ...), so that both see the same clocks; each arm reports the median of
--steps CUDA-event-timed steps after --warmup untimed ones.  Writes one JSON line to DIR/attn_fp16.json (and prints
it), with the GPU's name and power limit read in the same process."""
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

N, S, H, COEFF = 4, 2048, 32, 8


def _make_step(E: int, dtype):
    from spt_proto_b200 import layers
    torch.manual_seed(E)
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0).cuda().to(dtype)
    attn.sparse_coeff = COEFF
    attn.host_trigger = False          # no PQ training loss and no per-call device->host read of `trigger`
    q, k, v = (torch.randn(N, S, H, E, device="cuda", dtype=dtype).requires_grad_() for _ in range(3))
    dy = torch.randn(N, S, H, E, device="cuda", dtype=dtype)

    def step():
        q.grad = k.grad = v.grad = None
        attn(q, k, v).backward(dy)

    return attn, step


def _time_pair(E: int, warmup: int, steps: int):
    arms = {name: _make_step(E, dt) for name, dt in (("bf16", torch.bfloat16), ("fp16", torch.float16))}
    for _ in range(warmup):
        for _, step in arms.values():
            step()
    torch.cuda.synchronize()
    times = {name: [] for name in arms}
    for _ in range(steps):
        for name, (_, step) in arms.items():
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            step()
            t1.record()
            t1.synchronize()
            times[name].append(t0.elapsed_time(t1))
    out = {name: {"path": arms[name][0].last_path, "median_ms": statistics.median(t), "min_ms": min(t), "max_ms": max(t),
                  "steps": steps} for name, t in times.items()}
    out["fp16_over_bf16"] = out["fp16"]["median_ms"] / out["bf16"]["median_ms"]
    del arms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for attn_fp16.json")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if args.warmup < 5 or args.steps < 20:
        ap.error("need --warmup >= 5 and --steps >= 20")
    if not torch.cuda.is_available():
        sys.exit("attn_fp16.py measures on the GPU; no CUDA device found")
    arms = {f"d{E}": _time_pair(E, args.warmup, args.steps) for E in (64, 80, 128)}
    for a in arms.values():
        assert a["bf16"]["path"] == a["fp16"]["path"] == "fused"
    res = {"metric": "attn_layer_step_ms", "shape": {"N": N, "S": S, "H": H, "sparse_coeff": COEFF, "top_k": S // COEFF,
                                                    "output_layout": "reference"},
           **_gpu_info(), "arms": arms}
    line = json.dumps(res)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "attn_fp16.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
