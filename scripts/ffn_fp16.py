#!/usr/bin/env python
"""One routed-FFN layer step (forward + backward) in fp16 against the same step in bf16, at two shapes:

    RoutedFFN            T 8192, d 2048, F 8192, block 1024, ReLU            (bench.py's FFN, configs[2])
    LoRARoutedLLaMaFFN   T 2048, d 4096, F 11008, block 2752, rank 16, SiLU  (configs[3]'s FFN)

    python scripts/ffn_fp16.py [--out DIR] [--warmup 5] [--steps 20]

Both arms of a shape are the same fp32-initialised module converted with .half() / .bfloat16().  They are timed
alternately, step by step (bf16, fp16, bf16, ...), so that both see the same clocks; each arm reports the median of
--steps CUDA-event-timed steps after --warmup untimed ones.  Per arm it also reports the memory the arm holds
(torch.cuda.memory_allocated() growth from building it to the end of a step with every gradient set to None:
parameters, inputs and any cached weight copy; a throwaway arm runs first so that one-time library workspaces are not
charged to either) and the number of weight-copy cache entries for its parameters.
Prints one JSON line (and writes it to DIR/ffn_fp16.json with --out), with the GPU's name and power limit read in the same
process."""
from __future__ import annotations

import argparse
import copy
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
from torch import nn  # noqa: E402

from scripts.attn_head80 import _gpu_info  # noqa: E402

SHAPES = {
    "routed_ffn": dict(T=8192, d=2048, F=8192, block=1024, act="relu"),
    "lora_routed_llama_ffn": dict(T=2048, d=4096, F=11008, block=2752, rank=16, act="silu"),
}


def _module(name: str, s: dict) -> nn.Module:
    from spt_proto_b200 import layers
    torch.manual_seed(0)
    if name == "routed_ffn":
        return layers.RoutedFFN(d_model=s["d"], d_feedforward=s["F"], block_size=s["block"], activation=nn.ReLU())
    m = layers.LoRARoutedLLaMaFFN(d_lora=s["rank"], block_size=s["block"], d_model=s["d"], d_feedforward=s["F"],
                                  activation=nn.SiLU())
    with torch.no_grad():
        for n, p in m.named_parameters():
            if "lora.right" in n:
                nn.init.normal_(p, std=0.02)    # non-zero LoRA so that every gradient is exercised
    return m


def _arm(m32: nn.Module, s: dict, dtype):
    from spt_proto_b200.kernels import ffn as F
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    m = copy.deepcopy(m32).to("cuda", dtype)
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(s["T"], s["d"], device="cuda", generator=g).to(dtype).requires_grad_()
    dy = torch.randn(s["T"], s["d"], device="cuda", generator=g).to(dtype)
    params = list(m.parameters())

    def step():
        for p in params:
            p.grad = None
        x.grad = None
        m(x).backward(dy)

    step()
    for p in params:
        p.grad = None
    x.grad = None
    torch.cuda.synchronize()
    info = {"held_bytes": torch.cuda.memory_allocated() - base,
            "weight_copies": sum(1 for p in params if p in F._W16)}
    return step, info


def _time_pair(name: str, warmup: int, steps: int):
    s = SHAPES[name]
    m32 = _module(name, s)
    _arm(m32, s, torch.bfloat16)      # process-wide one-time allocations (library workspaces) are not an arm's memory
    arms = {label: _arm(m32, s, dt) for label, dt in (("bf16", torch.bfloat16), ("fp16", torch.float16))}
    del m32
    for _ in range(warmup):
        for step, _ in arms.values():
            step()
    torch.cuda.synchronize()
    times = {label: [] for label in arms}
    for _ in range(steps):
        for label, (step, _) in arms.items():
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            step()
            t1.record()
            t1.synchronize()
            times[label].append(t0.elapsed_time(t1))
    out = {label: {"median_ms": statistics.median(t), "min_ms": min(t), "max_ms": max(t), "steps": steps, **arms[label][1]}
           for label, t in times.items()}
    out["fp16_over_bf16"] = out["fp16"]["median_ms"] / out["bf16"]["median_ms"]
    out["shape"] = s
    del arms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="directory for ffn_fp16.json")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if args.warmup < 5 or args.steps < 20:
        ap.error("need --warmup >= 5 and --steps >= 20")
    if not torch.cuda.is_available():
        sys.exit("ffn_fp16.py measures on the GPU; no CUDA device found")
    res = {"metric": "ffn_layer_step_ms", **_gpu_info(), "arms": {n: _time_pair(n, args.warmup, args.steps) for n in SHAPES}}
    line = json.dumps(res)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "ffn_fp16.json"), "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
