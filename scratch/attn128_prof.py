"""Times of the fused attention at the bench shape + in-kernel phase timers of the 128 x 128-tile kernels
(library built with -DSPT_ATTN_PROF for the timers).  SPT_ATTN_TILE=64 runs the 128 x 64 kernels instead."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from spt_proto_b200 import ext
from spt_proto_b200._lib import lib
dev = "cuda"
B, S, d = int(os.environ.get("B", 128)), int(os.environ.get("S", 2048)), int(os.environ.get("D", 64))
g = torch.Generator().manual_seed(1)
q, k, v, dy = (torch.randn(B, S, d, generator=g).to(dev, torch.bfloat16) for _ in range(4))
w = torch.randn(d // 8, 16, 8, generator=g).to(dev)
mask, extra0, _ = ext.lookup_mask(ext.pq_encode(q, w), ext.pq_encode(k, w), 8)
def ev(fn, n=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n): fn()
    b.record(); b.synchronize()
    return a.elapsed_time(b) / n
y, z = ext.sparse_attn_fwd(q, k, v, mask, extra0, d ** -0.5)
print("tile", os.environ.get("SPT_ATTN_TILE", "128"), "fwd ms %.4f" % ev(lambda: ext.sparse_attn_fwd(q, k, v, mask, extra0, d ** -0.5)),
      "bwd ms %.4f" % ev(lambda: ext.sparse_attn_bwd(q, k, v, y, dy, mask, extra0, z, d ** -0.5)))
buf = (ctypes.c_ulonglong * 48)()
lib.spt_debug_attn_prof(buf, 3)
torch.cuda.synchronize()
ext.sparse_attn_fwd(q, k, v, mask, extra0, d ** -0.5)
ext.sparse_attn_bwd(q, k, v, y, dy, mask, extra0, z, d ** -0.5)
torch.cuda.synchronize()
if lib.spt_debug_attn_prof(buf, 2):
    mlab = ["wait_scores", "tmem_ld", "math", "st+arrive", "iters", "epilogue", "total"]
    ilab = ["issue_scores", "wait_math", "issue_acc", "total", "iters", "wait_k_full", "wait_s_read", "other"]
    for kidx, name in ((1, "bwd_q128"), (2, "bwd_kv128")):
        r = [buf[kidx * 16 + i] for i in range(16)]
        if r[4] == 0: continue
        it_m, it_i = max(r[4], 1), max(r[12], 1)
        print(name, "math thread, clk per tile:", {mlab[i]: round(r[i] / it_m, 1) for i in (0, 1, 2, 3, 5, 6)}, "tiles", r[4])
        print(name, "issuer, clk per tile:", {ilab[i]: round(r[8 + i] / it_i, 1) for i in (0, 1, 2, 3, 5, 6, 7)}, "tiles", r[12])
