"""Timing probe (not a pytest file): fvs_attention on the bench shape (32 frames x 577 tokens x 16 heads, f16) and on 16
frames, and fvs_attention80 on the Qwen2-VL grids; CUDA events around 50 back-to-back launches after a warm-up, two
repetitions per shape.  Prints one line per shape; with a path argument also writes them there as JSON:
    python tests/gpu_attn_probe.py [out.json]"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flash_vstream_b200 import ops  # noqa: E402


def time_it(fn, n=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3   # us


out = {}
SHAPES = ((64, torch.float16, 32, 577), (64, torch.float16, 16, 577), (80, torch.bfloat16, 8, 576), (80, torch.bfloat16, 8, 144))
for hd, dtype, frames, tokens in SHAPES:
    heads = 16
    qkv = torch.randn(frames * tokens, 3 * heads * hd, device="cuda").to(dtype)
    fn = (lambda: ops.attention(qkv, frames, tokens, heads)) if hd == 64 else (lambda: ops.attention80(qkv, frames, tokens, heads))
    us = [round(time_it(fn), 2) for _ in range(2)]
    flops = 4.0 * frames * heads * tokens * tokens * hd
    row = {"us": us, "tflops": round(flops / min(us) / 1e6, 1)}
    out[f"hd{hd}_f{frames}_t{tokens}"] = row
    print(f"hd{hd} frames={frames} tokens={tokens}: {row}", flush=True)
if len(sys.argv) > 1:
    json.dump(out, open(sys.argv[1], "w"), indent=1)
