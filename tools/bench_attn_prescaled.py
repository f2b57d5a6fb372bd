"""Micro-benchmark of the small-head attention kernels with Q prescaled (scale = -1: what the UNet plan runs).
usage: python tools/bench_attn_prescaled.py [B,h,N,hd ...]"""
import sys, os, math
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from weatherconverter_b200 import ops
dev = torch.device("cuda")
shapes = [(32, 4, 8192, 16), (32, 4, 8192, 32)]
if len(sys.argv) > 1:
    shapes = [tuple(int(v) for v in a.split(",")) for a in sys.argv[1:]]
for (B, h, N, hd) in shapes:
    q = (torch.randn(B, h, N, hd, device=dev) * (math.log2(math.e) / math.sqrt(hd))).bfloat16()
    k = torch.randn(B, h, N, hd, device=dev).bfloat16()
    vt = torch.randn(B, h, hd, N, device=dev).bfloat16()
    for _ in range(2): ops.attention(q, k, vt, scale=-1.0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): ops.attention(q, k, vt, scale=-1.0)
    e1.record(); torch.cuda.synchronize()
    print(f"B{B} h{h} N{N} hd{hd}: {e0.elapsed_time(e1)/5:.3f} ms", flush=True)
