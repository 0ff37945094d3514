#!/usr/bin/env python
"""Benchmark of the TeReDiff patch-denoising hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference]

One bench "step" = one complete 50-step spaced-sampler denoise of a batch of 16 synthetic 512x512 patches
(latent 4x64x64) per GPU through IRControlNet + SD2.1 UNet + the fused sampler update — BASELINE.json configs[1].
Random-init (non-degenerate) weights of the val architecture, synthetic conditioning, bf16 tensor-core compute.

value      : patches/s with all inputs resident in HBM (CUDA-graph replay of the step), max over ranks, weak scaling.
e2e        : same metric through the public API (SpacedSampler.sample) with pinned HOST inputs copied H2D and the
             final latent read back D2H inside the timed region.
full_step  : configs[2] — the whole TeReDiff step at B=16: the above + the TESTR text-spotting head on every step's
             decoder features + detection post-processing + string decode + prompt + OpenCLIP re-encode
             (SpacedSampler.val_sample, spaced_sampler.py:246-328); patches/s and ms per denoising step.
e2e_pixels : configs[3] — pixels to pixels through pipeline.restore_image (val_patches.py:296-391): a HOST uint8 512x512
             LQ image -> 25 overlapping tiles -> GPU front-end (crop + PIL-exact bicubic) -> SwinIR -> VAE encode + CLIP
             -> 50-step val_sample with TESTR feedback -> VAE decode -> ONE NCCL all_gather_into_tensor -> blend kernel
             -> restored 2048x2048 image back on the HOST.  At --gpus N the 25 tiles are sharded over the ranks
             (strong scaling; the collective and the blend are inside the timed region).
roofline   : dominant kernel family (3x3 implicit-GEMM conv, 47% of the FLOPs) timed live with CUDA events on the
             launching stream: algorithmic FLOPs / summed launch durations, against MEASURED_PEAKS.json.
cpu_baseline      : the reference's CPU path on the host cores (the real reference modules when the reference tree is
                    importable — $TAIR_REF, /root/reference, baseline/_ref — else the oracle port), bounded sample.
gpu_eager_baseline: the oracle port on cuda in fp32 with TF32 off ("the reference PyTorch path" on the same box), B=16.
cfg_sweep  : configs[4] reduced — classifier-free guidance (cond/uncond stacked, scale 4.0) at 1 / 4 / 16 / 32 tiles per GPU.
--impl reference  : the CPU path as its own arm, all host threads, same metric/config, extrapolated from a bounded sample.
--dump-outputs DIR: after the timed steps, write what the last timed step of each timed path returned to its caller as
                    DIR/<name>.npy (float32).  The global RNG is seeded once before the warm-up, so two builds run with
                    the same arguments get the same inputs and can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "patches_per_s_50step_512px"
UNIT = "patches/s"
SAMPLER_STEPS = 50
BATCH = 16
STEP_SEED = 4321                # global RNG seed set once before the warm-up (the sampler's per-step noise)
DUMP_LIMIT_BYTES = 64 << 20
# algorithmic work per tile-step, SURVEY.md §8(d) [probe]: conv3x3 504.3 + linear 366.5 + SDPA 176.5 + conv1x1 26.0 GFLOP
GFLOP_PER_TILE_STEP = 1073.4
# §8(d) memory-bound algorithmic bytes per tile-step (bf16 activations, read + write once)
GN_BYTES_PER_TILE_STEP = 59.1e6 * 4
LN_BYTES_PER_TILE_STEP = 48.7e6 * 4

VAE_CFG = dict(ddconfig=dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128,
                             ch_mult=[1, 2, 4, 4], num_res_blocks=2, attn_resolutions=[], dropout=0.0), embed_dim=4)
CLIP_CFG = dict(embed_dim=1024, vision_cfg=None, layer="penultimate",
                text_cfg=dict(context_length=77, vocab_size=49408, width=1024, heads=16, layers=24))
SWINIR_CFG = dict(img_size=64, patch_size=1, in_chans=3, embed_dim=180, depths=[6] * 8, num_heads=[6] * 8, window_size=8,
                  mlp_ratio=2, sf=8, img_range=1.0, upsampler="nearest+conv", resi_connection="1conv", unshuffle=True,
                  unshuffle_scale=8)


def full_cfgs():
    u = dict(in_channels=4, out_channels=4, model_channels=320, attention_resolutions=[4, 2, 1], num_res_blocks=2,
             channel_mult=[1, 2, 4, 4], num_head_channels=64, use_spatial_transformer=True,
             use_linear_in_transformer=True, transformer_depth=1, context_dim=1024, legacy=False)
    c = dict(u)
    c.pop("out_channels")
    c["hint_channels"] = 4
    return u, c


def hash_tokenizer(texts):
    """Stand-in for open_clip.tokenize when the CLIP merge table (OpenAI data, not redistributed) is absent: same
    (n,77) int64 contract, <start> ids... <end>; the text encoder's work does not depend on the ids."""
    import torch
    out = torch.zeros((len(texts), 77), dtype=torch.long)
    for i, s in enumerate(texts):
        ids = [49406] + [zlib.crc32(w.encode()) % 49000 for w in s.split(None, 76)[:75]] + [49407]
        out[i, :len(ids)] = torch.tensor(ids)
    return out


def workload_config(n_gpus, graph=True):
    return {"workload": "configs[1]: batch of 16 synthetic 512^2 patches bf16 per B200 "
                        "(IRControlNet + SD2.1 UNet + sampler-update kernels only), 50-step spaced sampler",
            "batch_per_gpu": BATCH, "sampler_steps": SAMPLER_STEPS, "latent": [4, 64, 64], "context": [77, 1024],
            "cfg_scale": 1.0, "weights": "random-init (seeded, non-degenerate)", "cuda_graph": graph,
            "l2": "256 MiB buffer written between timed steps; weights (2.4 GB bf16) exceed L2",
            "parallelism": f"dp{n_gpus} (independent patches per rank, no data-path collective; the sharded image with "
                           f"its all-gather + blend is measured as e2e_pixels)",
            # identical text in both arms so that their configs compare equal
            "reference_arm": "--impl reference is EXTRAPOLATED: it times a bounded sample (1-3 denoising steps of ONE patch "
                             "per bench step) of this workload on the host cores and scales by 50 steps x 16 patches"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def dump_outputs(path, outputs):
    """Write each host array of ``outputs`` as ``path/<name>.npy``, float64 kept, everything else as float32."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(v if v.dtype == np.float64 else v.astype(np.float32)) for k, v in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


class ClockSampler:
    """Polls nvidia-smi during the timed region (recipe's clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = []
        for i, name in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap")):
            if any(r[i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(float(r[2]) for r in self.rows)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (the only places that execute oracle/ or the reference tree)
# ---------------------------------------------------------------------------------------------------------------------
def _host_threads() -> int:
    import torch
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0)) or n
    except Exception:
        pass
    torch.set_num_threads(n)     # torchrun exports OMP_NUM_THREADS=1: without this the CPU arm would run single-threaded
    return torch.get_num_threads()


def _cpu_step_fn(state_dicts):
    """-> (one(i, x) -> x_prev, kind).  The real reference modules when the tree is importable, else the oracle port."""
    import torch
    from oracle import ref_harness as RH
    from oracle import sampler as OS
    from oracle import unet as OU
    usd, csd = state_dicts
    sched = OS.make_schedule(OS.diffusion_betas(), SAMPLER_STEPS)
    tabs = OS.tables_to_torch(sched)
    ts = sched["timesteps"][::-1]
    torch.manual_seed(0)
    hint, ctx = torch.randn(1, 4, 64, 64), torch.randn(1, 77, 1024)
    if RH.available():
        try:
            RH.install()
            from terediff.model.cldm import ControlLDM as RefCLDM
            from terediff.sampler.spaced_sampler import SpacedSampler as RefSampler
            u, c = RH.build_unet(), RH.build_controlnet()
            u.load_state_dict(usd)
            c.load_state_dict(csd)
            cldm = RefCLDM.__new__(RefCLDM)       # the reference forward() without its 438 M-parameter VAE / CLIP
            torch.nn.Module.__init__(cldm)
            cldm.unet, cldm.controlnet, cldm.control_scales = u, c, [1.0] * 13
            s = RefSampler(OS.diffusion_betas(), "v", False)
            s.make_schedule(SAMPLER_STEPS)

            def one_ref(i, x):
                model_t = torch.full((1,), int(ts[i]), dtype=torch.long)
                t = torch.full((1,), SAMPLER_STEPS - 1 - i, dtype=torch.long)
                return s.p_sample(cldm, x, model_t, t, dict(c_txt=ctx, c_img=hint), None, 1.0)[0]
            return one_ref, "reference"
        except Exception as e:  # pragma: no cover - the port is always available
            print(f"[bench] reference tree present but not importable ({e}); using the oracle port", file=sys.stderr)

    def one(i, x):
        model_t = torch.full((1,), int(ts[i]), dtype=torch.long)
        t = torch.full((1,), SAMPLER_STEPS - 1 - i, dtype=torch.long)
        v, _ = OU.cldm_forward(usd, csd, x, model_t, ctx, hint)
        return OS.p_sample_update(tabs, x, v, t, torch.randn_like(x))[0]
    return one, "port"


def cpu_baseline(state_dicts, seconds=20.0, max_steps=4, step_fn=None):
    """B=1, full-size ControlNet+UNet forward + sampler update per step on the host cores, fp32."""
    import torch
    cores = _host_threads()
    one, kind = step_fn or _cpu_step_fn(state_dicts)
    x = torch.randn(1, 4, 64, 64)
    with torch.no_grad():
        x = one(0, x)  # warm-up
        t0, n = time.perf_counter(), 0
        while n < max_steps and (n == 0 or time.perf_counter() - t0 < seconds):
            x = one(n + 1, x)
            n += 1
        dt = (time.perf_counter() - t0) / n
    what = "the reference's own modules (ControlLDM.forward + SpacedSampler.p_sample)" if kind == "reference" else "fp32 torch oracle port"
    return {"value": 1.0 / (dt * SAMPLER_STEPS), "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{n} of 50 denoising steps of 1 patch (ControlNet+UNet+update, {what}), "
                      f"{dt:.2f} s/step, extrapolated x50", "s_per_step": dt}


def run_reference(args):
    """--impl reference: the reference's CPU path, all host threads, same metric/config (extrapolated from a bounded
    sample: a full 16-patch 50-step denoise would take ~20 minutes per bench step on the host)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import weights as OW
    man = json.load(open(os.path.join(ROOT, "tests", "golden", "manifests.json")))
    sds = (OW.seeded_state_dict(man["unet_full"]), OW.seeded_state_dict(man["controlnet_full"]))
    fn = _cpu_step_fn(sds)
    K, W = args.steps, max(1, args.warmup)
    per = 1 if K > 3 else 3          # denoising steps per bench step: the whole run stays within a few minutes
    for _ in range(min(W, 2)):
        cpu_baseline(sds, seconds=1.0, max_steps=1, step_fn=fn)
    vals = [cpu_baseline(sds, seconds=15.0, max_steps=per, step_fn=fn) for _ in range(K)]
    dt = sum(v["s_per_step"] for v in vals) / len(vals)
    best = vals[0]
    value = 1.0 / (dt * SAMPLER_STEPS)
    cfg = workload_config(args.gpus, graph=True)     # same config object as the tair arm (cuda_graph is its setting)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt * SAMPLER_STEPS * BATCH,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": best["cores"], "kind": best["kind"],
                             "sample": f"EXTRAPOLATED x50 steps x16 patches from {len(vals)} bench step(s) of {per} denoising "
                                       f"step(s) of ONE patch each: " + best["sample"].replace(f"{best['s_per_step']:.2f} s/step", f"{dt:.2f} s/step (mean)")},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def gpu_eager_baseline(model, dev, steps=3):
    """The oracle port (fp32 torch, TF32 off) on cuda at the bench batch: 'the reference PyTorch path' on this box."""
    import torch
    from oracle import sampler as OS
    from oracle import unet as OU
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    usd = {k: v.detach().float() for k, v in model.unet.state_dict().items()}
    csd = {k: v.detach().float() for k, v in model.controlnet.state_dict().items()}
    sched = OS.make_schedule(OS.diffusion_betas(), SAMPLER_STEPS)
    tabs = OS.tables_to_torch(sched, dev)
    g = torch.Generator(device=dev).manual_seed(5)
    x = torch.randn((BATCH, 4, 64, 64), device=dev, generator=g)
    hint = torch.randn((BATCH, 4, 64, 64), device=dev, generator=g)
    ctx = torch.randn((BATCH, 77, 1024), device=dev, generator=g)
    mt = torch.full((BATCH,), 500, device=dev, dtype=torch.long)
    tt = torch.full((BATCH,), 25, device=dev, dtype=torch.long)

    def one(x):
        v, _ = OU.cldm_forward(usd, csd, x, mt, ctx, hint)
        return OS.p_sample_update(tabs, x, v, tt, torch.randn_like(x))[0]
    with torch.no_grad():
        one(x)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            x = one(x)
        b.record()
        torch.cuda.synchronize()
    ms = a.elapsed_time(b) / steps
    return {"value": BATCH / (ms * 1e-3 * SAMPLER_STEPS), "unit": UNIT, "ms_per_denoise_step": ms, "kind": "port",
            "what": f"oracle port (eager fp32 torch, TF32 off) on cuda, B={BATCH}, {steps} denoising steps, extrapolated x50"}


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="tair", choices=["tair", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip full_step / e2e_pixels / cfg_sweep / gpu_eager_baseline")
    ap.add_argument("--no-cfg-sweep", action="store_true", help="skip the classifier-free-guidance batch sweep (configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of every timed path as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl tair only")
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from tair_b200 import _lib
    _lib.lib()          # builds in-tree when missing / stale; raises when the CUDA library cannot be had (no fallback)
    from tair_b200 import ops, pipeline
    from tair_b200.init import nondegenerate_init_
    from tair_b200.model import ControlLDM
    from tair_b200.model.gaussian_diffusion import val_diffusion
    from tair_b200.sampler import SpacedSampler

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    extras = not args.no_extras

    unet_cfg, cn_cfg = full_cfgs()
    model = (ControlLDM(unet_cfg, VAE_CFG, CLIP_CFG, cn_cfg) if extras else ControlLDM(unet_cfg, cn_cfg)).to(dev).eval()
    nondegenerate_init_(model.unet, 1234)
    nondegenerate_init_(model.controlnet, 1235)
    betas = val_diffusion().betas
    sampler = SpacedSampler(betas, "v", False)

    g = torch.Generator(device=dev).manual_seed(100 + rank)
    x_T = torch.randn((BATCH, 4, 64, 64), device=dev, generator=g)
    c_img = torch.randn((BATCH, 4, 64, 64), device=dev, generator=g)
    c_txt = torch.randn((BATCH, 77, 1024), device=dev, generator=g)
    host = [t.cpu().pin_memory() for t in (x_T, c_img, c_txt)]
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
    use_graph = not args.no_graph
    outputs = {}     # name -> host array: what the last timed step of each timed path returned (--dump-outputs)

    def denoise(x0, ci, ct):
        z, _ = sampler.sample(model, dev, SAMPLER_STEPS, (BATCH, 4, 64, 64), dict(c_txt=ct, c_img=ci), None, 1.0,
                              x_T=x0, progress=False, use_cuda_graph=use_graph)
        return z

    def step_resident():
        flush.fill_(1)
        return denoise(x_T, c_img, c_txt)

    def step_e2e():
        flush.fill_(1)
        xs = [h.to(dev, non_blocking=True) for h in host]
        return denoise(*xs).cpu()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last_local_ms = [0.0]

    def timed(fn, k):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(k):
            out = fn()
        b.record()
        barrier()
        ms = a.elapsed_time(b) / k
        last_local_ms[0] = ms
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    torch.manual_seed(STEP_SEED)     # the sampler's per-step noise: the same sequence in every run with the same arguments
    for _ in range(W):
        z = step_resident()
    torch.cuda.synchronize()
    assert torch.isfinite(z).all(), "non-finite latent after warm-up"
    with ClockSampler(local) as clk:
        ms, z = timed(step_resident, K)
    outputs["latent"] = z.cpu().numpy()
    clocks = clk.summary()
    per_rank = None
    if world > 1:   # which rank sets the max: per-rank time and SM clock of the headline region (GPUs of one box differ by 1-3 %)
        mine = torch.tensor([last_local_ms[0], float(clocks.get("sm_mhz") or 0.0)], device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"ms_per_denoise": [round(float(t[0]), 2) for t in allr], "sm_mhz": [float(t[1]) for t in allr]}
    for _ in range(1):
        step_e2e()
    ms_e2e, z_e2e = timed(step_e2e, K)
    outputs["e2e_latent"] = z_e2e.numpy()

    # ---- live per-family kernel timing (CUDA events on the launching stream), one eager denoising step ----
    timer = ops.KernelTimer()
    sampler.make_schedule(SAMPLER_STEPS)
    sampler.to(dev)
    mt = torch.full((BATCH,), 500, device=dev, dtype=torch.long)
    tt = torch.full((BATCH,), 25, device=dev, dtype=torch.long)
    cond = dict(c_txt=c_txt, c_img=c_img)
    # one stream for this measurement: with the ControlNet on its own stream two kernels can share the GPU and the
    # per-launch event times would no longer be per-kernel times
    overlap, model.overlap_controlnet = model.overlap_controlnet, False
    for _ in range(2):
        sampler.p_sample(model, x_T, mt, tt, cond, None, 1.0)
    torch.cuda.synchronize()
    ops.reset_launch_count()
    ops.set_timer(timer)
    sampler.p_sample(model, x_T, mt, tt, cond, None, 1.0)
    ops.set_timer(None)
    model.overlap_controlnet = overlap
    fam = timer.summary()
    launches_per_step = ops.launch_count()
    pk = peaks()
    conv = fam["conv3x3"]
    conv_tflops = conv["work"] / (conv["ms"] * 1e-3) / 1e12
    n_conv = conv["launches"]
    roofline = {"kernel": "gemm_tc_kernel<BN> (implicit-GEMM 3x3 conv, tcgen05/TMA)", "bound": "tensor",
                "achieved": conv_tflops, "peak": pk["tc_sustained"], "unit": "TFLOP/s",
                "frac": conv_tflops / pk["tc_sustained"],
                # ncu dram__bytes_read+write of ONE launch of the most frequent conv (B=16, 64x64, 320->320;
                # profiles/round2_ncu_full_step_kernels.csv, gemm_tc_kernel<160>, 119 us): 43.9 MB read + 5.4 MB written
                # against 42 + 42 MB algorithmic in + out — the output stays in the 126 MB L2 for its consumer
                "traffic": 49.3e6, "traffic_unit": "B per launch (64x64 320->320 conv, ncu --set full, round 2)",
                "peak_source": pk["source"] + ", sustained bf16 (kernel timed inside a long step)",
                "launches_per_denoise_step": n_conv, "avg_launch_ms": conv["ms"] / n_conv,
                "flop_per_launch_avg": conv["work"] / n_conv}
    breakdown = {}
    for k, v in fam.items():
        e = {"launches": v["launches"], "ms": round(v["ms"], 4)}
        if k in ("conv3x3", "gemm", "attention"):
            e["tflops"] = round(v["work"] / (v["ms"] * 1e-3) / 1e12, 1)
            e["frac_of_tensor_peak"] = round(e["tflops"] / pk["tc_sustained"], 3)
        else:
            e["gbs"] = round(v["work"] / (v["ms"] * 1e-3) / 1e9, 1)
            e["frac_of_hbm_peak"] = round(e["gbs"] / pk["hbm"], 3)
        breakdown[k] = e
    # norm families against SURVEY §8(d)'s ALGORITHMIC bytes (4 B per element: one bf16 read + one bf16 write), whatever
    # the kernels actually move
    gn_ms = sum(v["ms"] for k, v in fam.items() if k.startswith("groupnorm"))
    ln_ms = sum(v["ms"] for k, v in fam.items() if k.startswith("layernorm"))
    norms = {"groupnorm_ms": round(gn_ms, 4), "layernorm_ms": round(ln_ms, 4), "family_ms": round(gn_ms + ln_ms, 4),
             "bytes_basis": "SURVEY 8(d): 59.1 M (GroupNorm) / 48.7 M (LayerNorm) elements x 4 B per tile-step"}
    if gn_ms > 0:
        norms["groupnorm_frac_of_hbm_on_algorithmic_bytes"] = round(GN_BYTES_PER_TILE_STEP * BATCH / (gn_ms * 1e-3) / 1e9 / pk["hbm"], 3)
    if ln_ms > 0:
        norms["layernorm_frac_of_hbm_on_algorithmic_bytes"] = round(LN_BYTES_PER_TILE_STEP * BATCH / (ln_ms * 1e-3) / 1e9 / pk["hbm"], 3)

    value = BATCH * world / (ms * 1e-3)
    e2e_val = BATCH * world / (ms_e2e * 1e-3)
    h2d = sum(h.numel() * h.element_size() for h in host)
    d2h = BATCH * 4 * 64 * 64 * 4
    step_ms = ms / SAMPLER_STEPS
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": workload_config(world, use_graph),
            "unet_step_latency_ms": step_ms,
            "model_tflops": GFLOP_PER_TILE_STEP * BATCH / step_ms,
            "model_frac_of_tensor_peak": GFLOP_PER_TILE_STEP * BATCH / step_ms / pk["tc_sustained"],
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e},
            "gpu_launches": int(launches_per_step * SAMPLER_STEPS * K),
            "gpu_launches_per_denoise_step": int(launches_per_step),
            "clocks": clocks, "per_rank": per_rank, "roofline": roofline, "kernel_breakdown_one_step": breakdown, "norm_families": norms}

    if extras:
        from types import SimpleNamespace
        from tair_b200.model.swinir import SwinIR
        from tair_b200.testr import TransformerDetector, default_cfg
        nondegenerate_init_(model.vae, 1236)
        nondegenerate_init_(model.clip, 1237)
        model.clip.attach_tokenizer(hash_tokenizer)
        det = TransformerDetector(default_cfg(str(dev))).to(dev).eval()
        nondegenerate_init_(det, 99)
        cleaner = SwinIR(**SWINIR_CFG).to(dev).eval()
        nondegenerate_init_(cleaner, 77)
        vcfg = SimpleNamespace(exp_args=SimpleNamespace(mode="VAL", prompt_style="CAPTION"))

        # ---- configs[2]: full step (TESTR + detection post-processing + prompt + CLIP re-encode), B = 16 per GPU ----
        c_txt0 = model.clip.encode([""] * BATCH)

        def full_denoise():
            flush.fill_(1)
            cond2 = dict(c_txt=c_txt0.clone(), c_img=c_img)
            z2, res = sampler.val_sample(model, dev, SAMPLER_STEPS, (BATCH, 4, 64, 64), cond2, None, 1.0, x_T=x_T,
                                         progress=False, cfg=vcfg, pure_cldm=model, ts_model=det, use_cuda_graph=use_graph)
            return z2, res
        full_denoise()
        ms_full, (z2, res2) = timed(full_denoise, K)
        assert torch.isfinite(z2).all()
        outputs["full_step_latent"] = z2.cpu().numpy()
        outputs["full_step_polygons_last_step_tile0"] = np.asarray(res2[-1]["pred_polys"], np.float32).reshape(-1, 16, 2)
        ops.reset_launch_count()
        full_denoise()
        torch.cuda.synchronize()
        line["full_step"] = {"workload": "configs[2]: B=16 per GPU, IRControlNet + UNet + sampler update + TESTR head "
                                         "(MSDeformAttn encoder/decoder) + detection post-processing + string decode + prompt "
                                         "+ OpenCLIP re-encode on every one of the 50 steps (val_sample)",
                             "value": BATCH * world / (ms_full * 1e-3), "unit": UNIT, "ms_per_denoise": ms_full,
                             "ms_per_denoise_step": ms_full / SAMPLER_STEPS, "timed_denoises": K,
                             "detections_last_step_tile0": len(res2[-1]["pred_texts"]),
                             "gpu_launches_outside_the_step_graph_per_denoise": int(ops.launch_count()),
                             "tokenizer": "hash stand-in (CLIP merge table not shipped)"}

        # ---- configs[3]: pixels to pixels, 512x512 LQ -> 25 tiles sharded over the ranks -> all-gather -> blend ----
        # a DIFFERENT image per call: restoring one image over and over would find every prompt of the previous pass in
        # the text encoder's prompt memo and skip the OpenCLIP re-encode that a real stream of images pays
        lqs = [np.random.default_rng(i).integers(0, 256, (512, 512, 3), dtype=np.uint8) for i in range(K + 1)]
        lq = lqs[0]
        n_tiles = 25
        PIX_TILE_BATCH = 32   # >= 25: a rank denoises all of its tiles as ONE batch (16 + 9 in two passes cost 5 % more)
        calls = [0]

        def restore():
            flush.fill_(1)
            lq = lqs[calls[0] % len(lqs)]
            calls[0] += 1
            out = pipeline.restore_image(lq, model, sampler, steps=SAMPLER_STEPS, tile_batch=PIX_TILE_BATCH, ts_model=det, cfg=vcfg,
                                         cleaner=lambda x: cleaner(x).clamp(0, 1), use_cuda_graph=use_graph)
            return out.cpu()
        restore()       # graph captures for this rank's tile-batch sizes (image 0; the timed calls restore images 1..K)
        req0, enc0 = model.clip.prompts_requested, model.clip.prompts_encoded
        ms_pix, img = timed(restore, K)
        req1, enc1 = model.clip.prompts_requested, model.clip.prompts_encoded
        assert tuple(img.shape) == (1, 3, 2048, 2048) and torch.isfinite(img).all()
        crc = zlib.crc32(img.numpy().tobytes())
        outputs["e2e_pixels_image"] = img.numpy()
        line["e2e_pixels"] = {"workload": "configs[3]: HOST uint8 512x512 LQ image -> 25 overlapping 128^2 tiles -> GPU crop + "
                                          "PIL-exact bicubic x4 -> SwinIR -> VAE encode + CLIP -> 50-step val_sample with TESTR "
                                          "feedback -> VAE decode -> all_gather_into_tensor (NCCL) -> blend kernel -> 2048x2048 "
                                          "fp32 image on the HOST (pipeline.restore_image)",
                              "value": n_tiles / (ms_pix * 1e-3), "unit": UNIT, "ms_per_image": ms_pix, "tiles": n_tiles,
                              "tiles_per_rank_max": (n_tiles + world - 1) // world, "tile_batch": PIX_TILE_BATCH, "scaling": "strong",
                              "collective": "none (1 rank)" if world == 1 else "1 x all_gather_into_tensor of decoded tiles + blend, inside the timed region",
                              "h2d_bytes_per_image": int(lq.nbytes), "d2h_bytes_per_image": int(img.numel() * 4),
                              "timed_images": K, "images": "a different synthetic image per call",
                              "prompts_per_image_this_rank": {"requested": (req1 - req0) // K, "encoded_by_openclip": (enc1 - enc0) // K},
                              "image_crc32": f"{crc:08x}"}

    if extras and not args.no_cfg_sweep:
        # ---- configs[4], reduced to what one bench run can afford: classifier-free guidance (cond / uncond stacked as
        # batch 2, scale 4.0, SURVEY §8a hazard 6) at several tiles-per-GPU batch sizes, one 50-step denoise each.  The
        # full 3840x2160 image is 700 tiles; tools/config4_sweep.py runs it (and batch 64) outside the bench budget. ----
        sweep = {}
        un_txt = torch.randn((1, 77, 1024), device=dev, generator=g)
        for bsz in (1, 4, 16, 32):
            xs = torch.randn((bsz, 4, 64, 64), device=dev, generator=g)
            ci = torch.randn((bsz, 4, 64, 64), device=dev, generator=g)
            ct = torch.randn((bsz, 77, 1024), device=dev, generator=g)
            un = dict(c_txt=un_txt.expand(bsz, -1, -1).contiguous(), c_img=ci)

            def cfg_denoise():
                flush.fill_(1)
                z3, _ = sampler.sample(model, dev, SAMPLER_STEPS, (bsz, 4, 64, 64), dict(c_txt=ct, c_img=ci), un, 4.0, x_T=xs,
                                       progress=False, use_cuda_graph=use_graph)
                return z3
            cfg_denoise()
            ms_c, z3 = timed(cfg_denoise, K)
            assert torch.isfinite(z3).all()
            outputs[f"cfg_sweep_latent_b{bsz}"] = z3.cpu().numpy()
            sweep[str(bsz)] = {"patches_per_s": bsz * world / (ms_c * 1e-3), "ms_per_denoise_step": ms_c / SAMPLER_STEPS}
        line["cfg_sweep"] = {"workload": "configs[4] (reduced): CFG scale 4.0 with cond/uncond stacked as batch 2 per tile, tiles-per-GPU "
                                         "batch sweep, 50-step sampler, ControlNet + UNet + fused CFG update; --steps timed denoises per batch",
                             "tiles_per_gpu": sweep, "unit": UNIT}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        usd = {k: v.detach().float().cpu() for k, v in model.unet.state_dict().items()}
        csd = {k: v.detach().float().cpu() for k, v in model.controlnet.state_dict().items()}
        line["cpu_baseline"] = {k: v for k, v in cpu_baseline((usd, csd)).items() if k != "s_per_step"}
        if extras:
            try:
                line["gpu_eager_baseline"] = gpu_eager_baseline(model, dev)
            except Exception as e:  # e.g. out of memory next to the resident models: report, do not fail the bench
                line["gpu_eager_baseline"] = {"unavailable": str(e)[:200]}
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
