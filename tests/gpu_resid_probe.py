"""Timing probe (not a pytest file) for the fp32-residual GEMM epilogue of one build of libfvs_b200.so (FVS_LIB_PATH):
out-proj and fc2 of a ViT-L/14 layer at the bench micro-batch (M = 32 x 577), x_f32 += A W^T + b in place with the L2
evicted between launches (as inside the encoder), next to the plain 16-bit epilogue on the same shapes; then the four
16-bit GEMMs of a layer back to back.  profiles/r2_resid_*.log were made with it (the ring builds that produced the
clock64 timelines there are gone from the tree; DESIGN.md §3.1 keeps what they showed)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flash_vstream_b200 import _lib as L  # noqa: E402


def time_it(fn, n=30):
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


tag = os.path.basename(os.environ.get("FVS_LIB_PATH", "base"))
lib = L.load()
M = 32 * 577
res = []
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
for N, K in ((1024, 1024), (1024, 4096)):
    A = torch.randn(M, K, device="cuda").half()
    W = (torch.randn(N, K, device="cuda") * 0.03).half()
    b = torch.randn(N, device="cuda").half()
    x = torch.zeros(M, N, device="cuda", dtype=torch.float32)
    o16 = torch.zeros(M, N, device="cuda").half()
    a4 = (L.ptr(A), L.ptr(W), L.ptr(b), L.ptr(x), L.ptr(x), M, N, K, K, N, L.EPI_BIAS_RESIDUAL_F32, 0, L.F16, L.cur_stream())
    a0 = (L.ptr(A), L.ptr(W), L.ptr(b), None, L.ptr(o16), M, N, K, K, N, L.EPI_BIAS, 0, L.F16, L.cur_stream())

    def cold(args):      # the residual stream is never L2-resident inside the encoder: evict between launches
        def fn():
            flush.zero_()
            L.check(lib.fvs_linear(*args))
        return fn

    def only_flush():
        flush.zero_()

    base = min(time_it(only_flush), time_it(only_flush))
    us4 = min(time_it(cold(a4)), time_it(cold(a4))) - base
    us0 = min(time_it(cold(a0)), time_it(cold(a0))) - base
    res.append(f"{N}x{K}: resid_f32 {us4:.1f}us ({2.0 * M * N * K / us4 / 1e6:.0f}TF)  bias16 {us0:.1f}us")
# the 16-bit epilogues of a layer, back to back (the four GEMM shapes of a ViT-L/14 layer at M = 32 x 577)
for N, K, epi in ((3072, 1024, 0), (1024, 1024, 0), (4096, 1024, 1), (1024, 4096, 0)):
    A = torch.randn(M, K, device="cuda").half()
    W = (torch.randn(N, K, device="cuda") * 0.03).half()
    b = torch.randn(N, device="cuda").half()
    out = torch.zeros(M, N, device="cuda").half()
    args = (L.ptr(A), L.ptr(W), L.ptr(b), L.ptr(out), L.ptr(out), M, N, K, K, N, epi, 577, L.F16, L.cur_stream())
    us = min(time_it(lambda: lib.fvs_linear(*args), 30), time_it(lambda: lib.fvs_linear(*args), 30))
    res.append(f"gemm{N}x{K} {us:.1f}us {2.0 * M * N * K / us / 1e6:.0f}TF")
print(tag, "|", " | ".join(res), flush=True)
