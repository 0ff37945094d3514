"""TEST INFRASTRUCTURE — restatement of multi-scale deformable attention (sampling + weighted sum).

``msda_core`` restates the CUDA kernel's per-tap arithmetic (testr/adet/layers/csrc/DeformAttn/
ms_deform_im2col_cuda.cuh:237-299, bilinear taps :33-84) with explicit gathers, independently of
``F.grid_sample``; tests pin it against the reference's own ``ms_deform_attn_core_pytorch``
(testr/adet/layers/ms_deform_attn.py:39-59), which is the only checker the reference ships for this op.
``msda_module`` restates MSDeformAttn.forward (ms_deform_attn.py:116-153).
"""
from __future__ import annotations

from typing import Dict, Sequence

import torch
import torch.nn.functional as F


def msda_core(value: torch.Tensor, shapes: Sequence[Sequence[int]], loc: torch.Tensor, w: torch.Tensor) -> torch.Tensor:
    """value [B,S,M,D]; shapes [(H_l, W_l)]; loc [B,Lq,M,L,P,2] (x,y in [0,1]); w [B,Lq,M,L,P] -> [B,Lq,M*D]."""
    B, S, M, D = value.shape
    _, Lq, _, L, P, _ = loc.shape
    out = value.new_zeros(B, Lq, M, D)
    start = 0
    bidx = torch.arange(B, device=value.device).view(B, 1, 1, 1).expand(B, Lq, M, P)
    midx = torch.arange(M, device=value.device).view(1, 1, M, 1).expand(B, Lq, M, P)
    for l, (H, W) in enumerate(shapes):
        H, W = int(H), int(W)
        v = value[:, start:start + H * W]                                  # [B, HW, M, D]
        x = loc[:, :, :, l, :, 0] * W - 0.5                                # cuh:285-286
        y = loc[:, :, :, l, :, 1] * H - 0.5
        inside = (y > -1) & (x > -1) & (y < H) & (x < W)                   # cuh:288
        x0, y0 = torch.floor(x), torch.floor(y)
        lx, ly = x - x0, y - y0
        x0, y0 = x0.long(), y0.long()
        acc = value.new_zeros(B, Lq, M, P, D)
        for dy, dx, wt in ((0, 0, (1 - ly) * (1 - lx)), (0, 1, (1 - ly) * lx), (1, 0, ly * (1 - lx)), (1, 1, ly * lx)):
            yy, xx = y0 + dy, x0 + dx
            ok = inside & (yy >= 0) & (yy <= H - 1) & (xx >= 0) & (xx <= W - 1)   # cuh:55-78
            idx = (yy.clamp(0, H - 1) * W + xx.clamp(0, W - 1))
            tap = v[bidx, idx, midx]                                        # [B,Lq,M,P,D]
            acc = acc + tap * (wt * ok)[..., None]
        out = out + (acc * w[:, :, :, l, :, None]).sum(3)
        start += H * W
    return out.reshape(B, Lq, M * D)


def msda_core_grid_sample(value, shapes, loc, w):
    """Same quantity through F.grid_sample (the formulation of ms_deform_attn.py:39-59), used as a cross-check."""
    B, S, M, D = value.shape
    _, Lq, _, L, P, _ = loc.shape
    vals = value.split([int(h) * int(w_) for h, w_ in shapes], dim=1)
    grids = 2 * loc - 1
    sampled = []
    for l, (H, W) in enumerate(shapes):
        vl = vals[l].flatten(2).transpose(1, 2).reshape(B * M, D, int(H), int(W))
        gl = grids[:, :, :, l].transpose(1, 2).flatten(0, 1)
        sampled.append(F.grid_sample(vl, gl, mode="bilinear", padding_mode="zeros", align_corners=False))
    aw = w.transpose(1, 2).reshape(B * M, 1, Lq, L * P)
    out = (torch.stack(sampled, dim=-2).flatten(-2) * aw).sum(-1).view(B, M * D, Lq)
    return out.transpose(1, 2).contiguous()


def msda_module(sd: Dict[str, torch.Tensor], p: str, query, ref, src, shapes, n_heads=8, n_points=4, core=msda_core):
    """MSDeformAttn.forward — ms_deform_attn.py:116-153 (no padding mask on this path)."""
    B, Lq, C = query.shape
    S = src.shape[1]
    L = len(shapes)
    value = F.linear(src, sd[p + ".value_proj.weight"], sd[p + ".value_proj.bias"]).view(B, S, n_heads, C // n_heads)
    off = F.linear(query, sd[p + ".sampling_offsets.weight"], sd[p + ".sampling_offsets.bias"])
    off = off.view(B, Lq, n_heads, L, n_points, 2)
    aw = F.linear(query, sd[p + ".attention_weights.weight"], sd[p + ".attention_weights.bias"])
    aw = F.softmax(aw.view(B, Lq, n_heads, L * n_points), -1).view(B, Lq, n_heads, L, n_points)
    shp = torch.as_tensor([[int(h), int(w)] for h, w in shapes], device=query.device, dtype=torch.float32)
    if ref.shape[-1] == 2:
        normalizer = torch.stack([shp[:, 1], shp[:, 0]], -1)
        loc = ref[:, :, None, :, None, :] + off / normalizer[None, None, None, :, None, :]
    else:
        loc = ref[:, :, None, :, None, :2] + off / n_points * ref[:, :, None, :, None, 2:] * 0.5
    out = core(value, shapes, loc, aw)
    return F.linear(out, sd[p + ".output_proj.weight"], sd[p + ".output_proj.bias"])


def ref_kernel_case(B: int, Lq: int, shapes, M: int = 8, D: int = 32, P: int = 4, device="cuda"):
    """Seeded fp32 inputs of the comparison with the reference's MSDeformAttn CUDA kernel
    (tests/test_msda_ref_gpu.py, tests/golden/make_golden.py msda_ref): value, shapes, level starts, locations, weights."""
    L = len(shapes)
    S = sum(h * w for h, w in shapes)
    g = torch.Generator(device=device).manual_seed(5)
    value = torch.randn(B, S, M, D, device=device, generator=g)
    loc = (torch.rand(B, Lq, M, L, P, 2, device=device, generator=g) * 1.4 - 0.2).contiguous()   # some samples fall outside
    w = torch.softmax(torch.randn(B, Lq, M, L * P, device=device, generator=g), -1).view(B, Lq, M, L, P).contiguous()
    shp = torch.tensor(shapes, device=device, dtype=torch.long)
    start = torch.cat([shp.new_zeros(1), (shp[:, 0] * shp[:, 1]).cumsum(0)[:-1]]).contiguous()
    return value, shp, start, loc, w
