"""Tile-level restoration driver: the val_patches.py image loop (val_patches.py:296-391) re-organised for B200.

Reference: for every 128x128 LQ tile, sequentially and at batch 1: bicubic x4 -> SwinIR -> prepare_condition ->
50-step val_sample -> VAE decode -> clamp; then merge_patches_with_overlap.  Here tiles are independent work units:
they are sharded round-robin over ranks (``tiles.shard_tiles``), batched ``tile_batch`` at a time through the
CUDA-graph step, decoded, reassembled with ONE all-gather and blended by one kernel.  Noise is keyed by the GLOBAL
tile index, so the restored image is bit-identical for every world size and batch size.

Stages around the denoising loop (val_patches.py:318-370):
    cleaner(lq)   : (b,3,512,512) in [0,1] -> cleaned image.  SwinIR (SURVEY.md §8f rank 3) is not on our kernels yet:
                    pass the torch module (or any callable); default = identity.
    cond_fn(lq)   : -> {"c_txt": (b,77,1024), "c_img": (b,4,64,64)}.  Default: ``cldm.prepare_condition(cleaner(lq), [""]*b)``
                    i.e. the kernel VAE encoder + the kernel OpenCLIP text encoder of ``cldm`` (cldm.py:143-158).
    decode_fn(z)  : (b,4,64,64) latent -> (b,3,512,512) in [0,1].  Default: ``(cldm.vae_decode(z) + 1) / 2`` (kernel VAE).
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional

import numpy as np
import torch

from . import tiles as T


def _tile_to_tensor(tile, size: int = 512) -> torch.Tensor:
    """PIL bicubic 128 -> 512 and /255, as val_patches.py:291-294,318 (T.Resize(BICUBIC) + T.ToTensor())."""
    from PIL import Image
    arr = np.asarray(tile.resize((size, size), Image.BICUBIC), dtype=np.float32) / 255.0
    if arr.ndim == 2:
        arr = np.repeat(arr[:, :, None], 3, axis=2)
    return torch.from_numpy(arr).permute(2, 0, 1)


class _TileNoise:
    """Per-tile random streams keyed by the global tile index (start noise first, then one draw per step)."""

    def __init__(self, indices: List[int], seed: int, device):
        self.gens = []
        for p in indices:
            g = torch.Generator(device=device)
            g.manual_seed(seed * 1000003 + p)
            self.gens.append(g)
        self.device = device

    def draw(self) -> torch.Tensor:
        return torch.stack([torch.randn((4, 64, 64), generator=g, device=self.device) for g in self.gens])


@torch.no_grad()
def restore_image(lq: np.ndarray, cldm, sampler, *, cond_fn: Optional[Callable] = None,
                  decode_fn: Optional[Callable] = None, cleaner: Optional[Callable] = None, ts_model=None,
                  steps: int = 50, tile_batch: int = 16, cfg_scale: float = 1.0, uncond_fn: Optional[Callable] = None,
                  seed: int = 25, group=None, use_cuda_graph: bool = True, cfg=None) -> torch.Tensor:
    """lq: (H,W,3) uint8 low-quality image -> (1,3,4H,4W) restored image on every rank.

    ``sampler`` is any sampler of ``tair_b200.sampler``: ``SpacedSampler`` (the reference's 50-step DDPM), or
    ``DDIMSampler`` / ``DPMSolverSampler`` / ``UniPCSampler`` (one network evaluation per step, usually run with fewer
    ``steps``).  The
    step noise is drawn per tile either way, so the result does not depend on ``tile_batch``."""
    import torch.distributed as dist
    dev = next(cldm.parameters()).device
    if cond_fn is None:
        if cldm.vae is None or cldm.clip is None:
            raise RuntimeError("restore_image: pass cond_fn, or build ControlLDM with vae_cfg and clip_cfg")
        cond_fn = lambda x: cldm.prepare_condition(x if cleaner is None else cleaner(x), [""] * x.shape[0])
    if decode_fn is None:
        if cldm.vae is None:
            raise RuntimeError("restore_image: pass decode_fn, or build ControlLDM with vae_cfg")
        decode_fn = lambda z: (cldm.vae_decode(z) + 1) / 2
    world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
    rank = dist.get_rank(group) if world > 1 else 0
    # tile front-end on the GPU: the padded LQ image is uploaded once, tiles are cropped + resized on the device with
    # PIL's exact fixed-point bicubic arithmetic (bit-identical to split_image_with_overlap + resize + ToTensor)
    front = T.TileFrontEnd(lq, dev)
    n = len(front)
    mine = T.shard_tiles(n, rank, world)
    decoded = []
    for s in range(0, len(mine), tile_batch):
        idx = mine[s:s + tile_batch]
        b = len(idx)
        lq512 = front.tiles(idx)
        cond = cond_fn(lq512)
        uncond = uncond_fn(lq512) if (uncond_fn is not None and cfg_scale != 1.0) else None
        noise = _TileNoise(idx, seed, dev)
        x_T = noise.draw()
        sampler.noise_fn = lambda i, x, _n=noise: _n.draw()
        try:
            if ts_model is not None:
                z, _ = sampler.val_sample(cldm, dev, steps, (b, 4, 64, 64), cond, uncond, cfg_scale, x_T=x_T,
                                          progress=False, cfg=cfg, pure_cldm=cldm, ts_model=ts_model,
                                          use_cuda_graph=use_cuda_graph)
            else:
                z, _ = sampler.sample(cldm, dev, steps, (b, 4, 64, 64), cond, uncond, cfg_scale, x_T=x_T, progress=False,
                                      use_cuda_graph=use_cuda_graph)
        finally:
            sampler.noise_fn = None
        decoded.append(decode_fn(z).clamp(0, 1).float())
    local = torch.cat(decoded, 0) if decoded else torch.zeros((0, 3, 512, 512), device=dev)
    all_tiles = T.gather_tiles(local, n, group)
    return T.merge_patches_with_overlap(all_tiles, lq.shape[:2], 512, 64)


def save_image(img: torch.Tensor, path: str) -> None:
    """(1,3,H,W) or (3,H,W) image in [0,1] -> 8-bit PNG/JPEG (host side; val_patches.py writes the restored image with
    torchvision's ToPILImage, i.e. mul(255) and a truncating byte cast)."""
    from PIL import Image
    t = img.detach()
    if t.dim() == 4:
        t = t[0]
    arr = t.clamp(0, 1).mul(255).byte().permute(1, 2, 0).cpu().numpy()
    Image.fromarray(arr).save(path)
