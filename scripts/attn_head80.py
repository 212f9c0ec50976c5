#!/usr/bin/env python
"""One OPT-2.7B attention layer step (forward + backward of SparseVanillaAttentionV2, reference output layout) at head
dim 80: the fused tensor-core path against the stage chain (use_fused = False), with the fused d 64 and d 128 steps at
the same N, S, H for context.

    python scripts/attn_head80.py --out DIR [--warmup 5] [--steps 20]

Shape: N 4, S 2048, H 32, sparse_coeff 8 (top-k 256), bf16, random dO; q, k, v and dO of the d 80 case are 168 MB,
more than the L2.  Each arm is timed as the median of --steps CUDA-event-timed steps after --warmup untimed ones.
Writes one JSON line to DIR/attn_head80.json (and prints it), with the GPU's name and power limit read in the same
process."""
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

N, S, H, COEFF = 4, 2048, 32, 8


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


def _time_arm(E: int, fused: bool, warmup: int, steps: int):
    from spt_proto_b200 import layers
    torch.manual_seed(E)
    attn = layers.SparseVanillaAttentionV2(d_head=E, d_codeword=8, n_codewords=16, p_dropout=0.0).cuda()
    attn.sparse_coeff = COEFF
    attn.use_fused = fused
    attn.host_trigger = False          # no PQ training loss and no per-call device->host read of `trigger`
    q, k, v = (torch.randn(N, S, H, E, device="cuda", dtype=torch.bfloat16).requires_grad_() for _ in range(3))
    dy = torch.randn(N, S, H, E, device="cuda", dtype=torch.bfloat16)

    def step():
        q.grad = k.grad = v.grad = None
        attn(q, k, v).backward(dy)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    path = attn.last_path
    times = []
    for _ in range(steps):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        step()
        t1.record()
        t1.synchronize()
        times.append(t0.elapsed_time(t1))
    del attn, q, k, v, dy
    torch.cuda.empty_cache()
    return {"d_head": E, "path": path, "median_ms": statistics.median(times), "min_ms": min(times),
            "max_ms": max(times), "steps": steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for attn_head80.json")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if args.warmup < 5 or args.steps < 20:
        ap.error("need --warmup >= 5 and --steps >= 20")
    if not torch.cuda.is_available():
        sys.exit("attn_head80.py measures on the GPU; no CUDA device found")
    arms = {
        "fused_d80": _time_arm(80, True, args.warmup, args.steps),
        "stage_d80": _time_arm(80, False, args.warmup, args.steps),
        "fused_d64": _time_arm(64, True, args.warmup, args.steps),
        "fused_d128": _time_arm(128, True, args.warmup, args.steps),
    }
    assert arms["fused_d80"]["path"] == "fused" and arms["stage_d80"]["path"] == "stage"
    res = {"metric": "attn_layer_step_ms", "shape": {"N": N, "S": S, "H": H, "sparse_coeff": COEFF, "top_k": S // COEFF,
                                                    "dtype": "bf16", "output_layout": "reference"},
           **_gpu_info(), "arms": arms,
           "stage_over_fused_d80": arms["stage_d80"]["median_ms"] / arms["fused_d80"]["median_ms"]}
    line = json.dumps(res)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "attn_head80.json"), "w") as f:
        f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
