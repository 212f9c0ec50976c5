#!/usr/bin/env python
"""Long sequences on the fused path: one attention layer step (forward + backward of SparseVanillaAttentionV2, reference
output layout, sparse_coeff 8) and the mask-only lookup alone, at S 8192, 16384, 32768 and 65536 for head dims 64, 80
and 128 (PQ subspaces m 8, 10, 16), in bf16 and fp16.

    python scripts/attn_long.py --out DIR [--warmup 2] [--steps 5]

N 1; the head count H = min(32, 2^32 / S^2) keeps the forward's bitmask (H S^2 / 8 bytes) at 512 MiB or less: H 32 at
S 8192, 16 at 16384, 4 at 32768, 1 at 65536.  Above S 8192 the layer recomputes the mask in the backward (DESIGN.md
section 4.1).  Every number is the median of --steps CUDA-event-timed calls after --warmup untimed ones; the lookup
timing includes the key-bitmap pre-pass.  The lookup kernels each case runs are read with torch.profiler in a separate
call.  Writes one JSON line per case to DIR/attn_long.jsonl (and prints it); the first line holds the GPU's name and
power limit, read in the same process."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

COEFF = 8


def _gpu_info():
    info = {"gpu": torch.cuda.get_device_name(), "power_limit_w": None, "sm_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}",
                              "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        pl, mhz = (x.strip() for x in out.split(","))
        info["power_limit_w"], info["sm_max_mhz"] = float(pl), float(mhz)
    except (OSError, subprocess.SubprocessError, ValueError, IndexError):
        pass
    return info


def _median_ms(fn, warmup: int, steps: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def _lookup_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({e.name.split("(")[0].replace("void spt::", "") for e in prof.events()
                   if "lookup_" in e.name and "kernel" in e.name})


def _case(S: int, E: int, dtype, warmup: int, steps: int):
    from spt_proto_b200 import ext, layers
    H = min(32, 2 ** 32 // (S * S))
    torch.manual_seed(S + E)
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0).cuda()
    if dtype == torch.float16:
        attn = attn.half()
    attn.host_trigger = False
    q, k, v = (torch.randn(1, S, H, E, device="cuda", dtype=dtype).requires_grad_() for _ in range(3))
    dy = torch.randn(1, S, H, E, device="cuda", dtype=dtype)

    def step():
        q.grad = k.grad = v.grad = None
        attn(q, k, v).backward(dy)

    step_ms = _median_ms(step, warmup, steps)
    assert attn.last_path == "fused", attn.last_path
    with torch.no_grad():
        q_c, k_c = ext.pq_encode_pair(q.detach(), k.detach(), attn.quantizer.weight)
    lookup = lambda: ext.lookup_mask(q_c, k_c, COEFF, n_codewords=16)
    lookup_ms = _median_ms(lookup, warmup, steps)
    return {"S": S, "d": E, "m": E // 8, "H": H, "dtype": str(dtype).replace("torch.", ""),
            "step_ms": round(step_ms, 3), "lookup_ms": round(lookup_ms, 4),
            "lookup_us_per_head_per_1k_tokens": round(1e3 * lookup_ms / H / (S / 1024), 3),
            "recompute": S > attn.recompute_mask_above, "lookup_kernels": _lookup_kernels(lookup)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    lines = [dict(_gpu_info(), N=1, sparse_coeff=COEFF, layout="reference", warmup=args.warmup, steps=args.steps)]
    print(json.dumps(lines[0]), flush=True)
    for dtype in (torch.bfloat16, torch.float16):
        for E in (64, 80, 128):
            for S in (8192, 16384, 32768, 65536):
                lines.append(_case(S, E, dtype, args.warmup, args.steps))
                print(json.dumps(lines[-1]), flush=True)
                torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "attn_long.jsonl"), "w") as f:
            f.write("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
