"""GPU: fvs_attention (head_dim 64) and fvs_attention80 (head_dim 80) against fp32 torch attention.  Shapes cover the
ViT-L/14-336 and Qwen2-VL grids, a single KV tile, a narrow last KV tile (stale score columns masked out), odd and even
KV-tile counts (the two TMEM score buffers alternate), one token, and both 16-bit dtypes with both head dims."""
import pytest
import torch

pytestmark = pytest.mark.gpu

REL_TOL = 2e-3   # 16-bit P and output rounding; the encoder-level 1e-3 bound is asserted in test_gpu_parity.py


def rel(a, b):
    return ((a - b).norm() / b.norm()).item()


def reference(nat, frames, tokens, heads, hd):
    q, k, v = (t.transpose(1, 2) for t in nat.float().view(frames, tokens, 3, heads, hd).unbind(2))
    return (torch.softmax(q @ k.transpose(-1, -2) * hd ** -0.5, -1) @ v).transpose(1, 2).reshape(frames * tokens, heads * hd)


def run(ops, nat, frames, tokens, heads, hd):
    if hd == 64:
        out = ops.attention(nat, frames, tokens, heads)
    else:
        out = ops.merge_heads_80(ops.attention80(ops.split_heads_80(nat, heads, 3), frames, tokens, heads), heads)
    torch.cuda.synchronize()
    return out


CASES = [  # (head_dim, dtype, frames, tokens, heads)
    (64, torch.float16, 3, 577, 16),      # ViT-L/14-336 grid: 10 KV tiles (even), the last one 16 wide with 1 valid key
    (64, torch.float16, 20, 577, 16),     # same grid, 1600 CTAs: several waves over the SMs
    (64, torch.bfloat16, 9, 577, 16),     # bf16
    (64, torch.float16, 40, 144, 16),     # 3 KV tiles (odd), the last one 16 wide
    (64, torch.float16, 48, 64, 16),      # single KV tile, full width
    (64, torch.float16, 33, 100, 16),     # 2 KV tiles, the second 48 wide: one column group partly valid
    (64, torch.float16, 5, 1, 16),        # one token: a single 16-wide tile, one column group without a valid key
    (80, torch.bfloat16, 4, 576, 16),     # Qwen2-VL full-resolution grid: 9 full KV tiles (odd)
    (80, torch.bfloat16, 12, 576, 16),    # same grid, more frames
    (80, torch.bfloat16, 30, 144, 16),    # half-resolution grid, 3 KV tiles, the last one 16 wide
    (80, torch.float16, 50, 36, 16),      # head_dim 80 in f16: single KV tile, 48 wide
]


@pytest.mark.parametrize("hd,dtype,frames,tokens,heads", CASES)
def test_attention_matches_reference(hd, dtype, frames, tokens, heads):
    from flash_vstream_b200 import ops
    g = torch.Generator().manual_seed(frames * 1000 + tokens)
    nat = torch.randn(frames * tokens, 3 * heads * hd, generator=g).to(dtype).cuda()
    ref = reference(nat, frames, tokens, heads, hd)
    out = run(ops, nat, frames, tokens, heads, hd)
    tol = REL_TOL if dtype == torch.float16 else 8e-3
    assert rel(out.float(), ref) < tol


def test_attention_large_scores_rescale_path():
    """scores that keep growing along the key axis force the lazy O|L rescale"""
    from flash_vstream_b200 import ops
    frames, tokens, heads, hd = 10, 577, 16, 64
    g = torch.Generator().manual_seed(11)
    nat = torch.randn(frames * tokens, 3 * heads * hd, generator=g)
    ramp = torch.linspace(0.2, 3.0, tokens).repeat(frames)[:, None]
    nat[:, heads * hd:2 * heads * hd] *= ramp       # keys grow with the token index -> row maxima keep rising
    nat = nat.half().cuda()
    ref = reference(nat, frames, tokens, heads, hd)
    out = run(ops, nat, frames, tokens, heads, hd)
    assert rel(out.float(), ref) < 3e-3
