"""TEST INFRASTRUCTURE — restatement of the tile driver's split / blend (val_patches.py:25-92, :114-206)."""
from __future__ import annotations

import math
from typing import List, Sequence, Tuple

import numpy as np
import torch


def tile_grid(height: int, width: int, patch: int = 128, overlap: int = 16) -> Tuple[int, int, int, int]:
    """(n_h, n_w, padded_h, padded_w) — val_patches.py:49-58."""
    stride = patch - overlap
    n_h = math.ceil((height - overlap) / stride)
    n_w = math.ceil((width - overlap) / stride)
    return n_h, n_w, (n_h - 1) * stride + patch, (n_w - 1) * stride + patch


def split_image(img: np.ndarray, patch: int = 128, overlap: int = 16) -> List[np.ndarray]:
    """Zero-pad right/bottom and cut row-major tiles — val_patches.py:25-92 (HWC or HW uint8 arrays)."""
    h, w = img.shape[:2]
    n_h, n_w, ph, pw = tile_grid(h, w, patch, overlap)
    pad = ((0, ph - h), (0, pw - w)) + (((0, 0),) if img.ndim == 3 else ())
    padded = np.pad(img, pad, mode="constant", constant_values=0)
    stride = patch - overlap
    return [padded[i * stride:i * stride + patch, j * stride:j * stride + patch].astype(np.uint8)
            for i in range(n_h) for j in range(n_w)]


def blend_window(patch: int = 512, fade: int = 64, dtype=torch.float32) -> torch.Tensor:
    """val_patches.py:155-167: ones with linear ramps (i+1)/fade multiplied onto all four edges."""
    win = torch.ones((patch, patch), dtype=dtype)
    for i in range(fade):
        f = (i + 1) / fade
        win[i, :] *= f
        win[-(i + 1), :] *= f
        win[:, i] *= f
        win[:, -(i + 1)] *= f
    return win


def merge_tiles(tiles: Sequence[torch.Tensor], original_size: Tuple[int, int], patch: int = 512, overlap: int = 64):
    """val_patches.py:114-206.  NB the grid is derived from the hard-coded LQ geometry 128/16 (:133-148)."""
    oh, ow = original_size
    n_h, n_w, ph, pw = tile_grid(oh, ow, 128, 16)
    scale = patch / 128
    fh, fw = int(ph * scale), int(pw * scale)
    dev, dt = tiles[0].device, tiles[0].dtype
    canvas = torch.zeros((1, 3, fh, fw), device=dev, dtype=dt)
    weight = torch.zeros((1, 1, fh, fw), device=dev, dtype=dt)
    win = blend_window(patch, overlap, dt).to(dev)
    stride = patch - overlap
    k = 0
    for i in range(n_h):
        for j in range(n_w):
            if k >= len(tiles):
                break
            ys, xs = i * stride, j * stride
            canvas[:, :, ys:ys + patch, xs:xs + patch] += tiles[k] * win
            weight[:, :, ys:ys + patch, xs:xs + patch] += win
            k += 1
    out = canvas / weight.clamp(min=1e-8)
    return out[:, :, :int(oh * scale), :int(ow * scale)]


def resize_tile_reference(tile_u8, out_size: int, coeff_fn):
    """numpy restatement of PIL's two fixed-point resampling passes (Pillow Resample.c: ImagingResampleHorizontal_8bpc
    then ImagingResampleVertical_8bpc) driven by per-output-index tables ``coeff_fn(in_size, out_size) -> (bounds,
    coeffs)``; the CPU test pins the product's tables (tair_b200.tiles.pil_bicubic_coeffs) against PIL through it."""
    import numpy as np
    h, w = tile_u8.shape[:2]
    bx, cx = coeff_fn(w, out_size)
    by, cy = coeff_fn(h, out_size)
    t = tile_u8.astype(np.int64)
    tmp = np.zeros((h, out_size, 3), np.int64)
    for ox in range(out_size):
        x0, n = bx[ox]
        tmp[:, ox] = np.clip(((1 << 21) + (t[:, x0:x0 + n] * cx[ox, :n, None].astype(np.int64)).sum(1)) >> 22, 0, 255)
    out = np.zeros((out_size, out_size, 3), np.int64)
    for oy in range(out_size):
        y0, n = by[oy]
        out[oy] = np.clip(((1 << 21) + (tmp[y0:y0 + n] * cy[oy, :n, None, None].astype(np.int64)).sum(0)) >> 22, 0, 255)
    return out.astype(np.uint8)


def tiled_fn_case():
    """Seeded input, tile function and (size, stride) cases of the make_tiled_fn comparison (tests/test_host_cpu.py,
    tests/golden/make_golden.py tiled)."""
    x = torch.randn(1, 4, 40, 56, generator=torch.Generator().manual_seed(1))
    return x, (lambda t: torch.tanh(t) * 3), ((16, 8), (16, 12), (32, 20))
