"""Spaced-50 vs DDIM-25 vs DPM-Solver++(2M)-20 vs UniPC-2 at 10 and 15 steps at the bench batch (B=16, synthetic weights),
in one process, alternating.

For each sampler: a whole `sample` run (ControlNet + UNet + update per step, CUDA graph) and a whole `val_sample` run
(+ TESTR head, detection post-processing, prompt and CLIP re-encode per step), timed with a host clock around work that
ends in a device synchronise.  Reports ms per step, s per batch and patches/s, and the fused multistep and UniPC update
kernels against tair_sampler_update (CUDA events around graph replays of 200 back-to-back launches on the [16, 4, 64, 64] latent,
which stays in L2).  The GPU name and power limit are read in the same run.  Prints the result as JSON, and writes it
to the file given with --out."""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from bench import full_cfgs  # noqa: E402
from tair_b200 import ops  # noqa: E402
from tair_b200.init import nondegenerate_init_  # noqa: E402
from tair_b200.model import ControlLDM  # noqa: E402
from tair_b200.model.clip import FrozenOpenCLIPEmbedder  # noqa: E402
from tair_b200.model.gaussian_diffusion import val_diffusion  # noqa: E402
from tair_b200.sampler import DDIMSampler, DPMSolverSampler, SpacedSampler, UniPCSampler  # noqa: E402
from tair_b200.testr import TransformerDetector, default_cfg  # noqa: E402

B, REPS = 16, int(os.environ.get("REPS", "3"))
dev = torch.device("cuda:0")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(dev), "nvidia_smi": q}


def hash_tok(texts):
    out = torch.zeros((len(texts), 77), dtype=torch.long)
    for i, s_ in enumerate(texts):
        ids = [49406] + [zlib.crc32(w.encode()) % 49000 for w in s_.split()][:75] + [49407]
        out[i, :len(ids)] = torch.tensor(ids)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    info_before = gpu_info()
    model = ControlLDM(*full_cfgs()).to(dev).eval()
    nondegenerate_init_(model, 1234)
    clip = FrozenOpenCLIPEmbedder(1024, None, dict(context_length=77, vocab_size=49408, width=1024, heads=16, layers=24),
                                  layer="penultimate").to(dev).eval()
    nondegenerate_init_(clip, 7)
    clip.attach_tokenizer(hash_tok)
    model.attach_clip(clip)
    det = TransformerDetector(default_cfg("cuda")).to(dev).eval()
    nondegenerate_init_(det, 99)
    betas = val_diffusion().betas
    configs = [("spaced", SpacedSampler(betas), 50), ("ddim", DDIMSampler(betas), 25),
               ("dpmpp2m", DPMSolverSampler(betas), 20),
               # one instance per step count: a schedule change re-allocates the tables and drops the captured graphs
               ("unipc2_", UniPCSampler(betas, order=2), 10), ("unipc2_", UniPCSampler(betas, order=2), 15)]
    g = torch.Generator(device=dev).manual_seed(0)
    x_T = torch.randn((B, 4, 64, 64), device=dev, generator=g)
    c_img = torch.randn((B, 4, 64, 64), device=dev, generator=g)
    c_txt0 = clip.encode([""] * B)
    vcfg = SimpleNamespace(exp_args=SimpleNamespace(mode="VAL", prompt_style="CAPTION"))

    def run(kind, s, n):
        cond = dict(c_txt=c_txt0.clone(), c_img=c_img)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if kind == "sample":
            z, _ = s.sample(model, dev, n, (B, 4, 64, 64), cond, None, 1.0, x_T=x_T, progress=False, use_cuda_graph=True)
        else:
            z, _ = s.val_sample(model, dev, n, (B, 4, 64, 64), cond, None, 1.0, x_T=x_T, progress=False, cfg=vcfg,
                                pure_cldm=model, ts_model=det, use_cuda_graph=True)
        torch.cuda.synchronize()
        assert torch.isfinite(z).all()
        return time.perf_counter() - t0

    times = {(name + str(n), kind): [] for name, _, n in configs for kind in ("sample", "val_sample")}
    for name, s, n in configs:           # warm-up: graph capture, autotuning, CLIP cache
        for kind in ("sample", "val_sample"):
            run(kind, s, n)
    for _ in range(REPS):
        for name, s, n in configs:
            for kind in ("sample", "val_sample"):
                times[name + str(n), kind].append(run(kind, s, n))

    res = {"batch": B, "reps": REPS, "gpu_before": info_before, "runs": {}}
    for name, s, n in configs:
        for kind in ("sample", "val_sample"):
            ts = times[name + str(n), kind]
            best, med = min(ts), sorted(ts)[len(ts) // 2]
            res["runs"][f"{name}{n}_{kind}"] = {
                "steps": n, "s_per_batch_all": [round(t, 4) for t in ts], "s_per_batch_median": round(med, 4),
                "ms_per_step_median": round(med * 1e3 / n, 3), "ms_per_step_min": round(best * 1e3 / n, 3),
                "patches_per_s_median": round(B / med, 3)}
            print(name, n, kind, res["runs"][f"{name}{n}_{kind}"], flush=True)

    # the update kernels alone
    x, v, nz = (torch.randn((B, 4, 64, 64), device=dev, generator=g) for _ in range(3))
    t = torch.full((B,), 10, device=dev, dtype=torch.long)
    spaced, ms = configs[0][1], configs[2][1]
    spaced.make_schedule(50)
    spaced.to(dev)
    ms.make_schedule(20)
    ms.to(dev)
    out = torch.empty_like(x)
    hist = ms.x0_history(x)
    uni = {}
    for order in (2, 3):    # a corrected step of full order: every state slot is read
        u = uni[order] = UniPCSampler(betas, order=order)
        u.make_schedule(20)
        u.to(dev)

    def ev(fn, n=200, reps=10):
        """us per launch: n launches captured in one CUDA graph, replayed reps times (no host overhead per launch)."""
        fn()
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(n):
                fn()
        gr.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(True), torch.cuda.Event(True)
        a.record()
        for _ in range(reps):
            gr.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / (n * reps)
    kern = {}
    for _ in range(3):   # alternate
        kern.setdefault("sampler_update_us", []).append(ev(lambda: ops.sampler_update(x, v, nz, t, spaced._tables(), out=out)))
        kern.setdefault("sampler_multistep_update_us", []).append(
            ev(lambda: ops.sampler_multistep_update(x, v, nz, t, ms._tables(), x0_hist=hist, out=out)))
        for order, u in uni.items():
            xc, h = u.state_buffers(x)
            kern.setdefault(f"sampler_unipc_update_k{order}_us", []).append(
                ev(lambda: ops.sampler_unipc_update(x, v, t, u.unipc_table, x_corr=xc, x0_hist=h, out=out)))
    res["update_kernel"] = {k: [round(u, 3) for u in vals] for k, vals in kern.items()}
    res["update_kernel"]["note"] = ("per launch, 200 launches per CUDA graph replayed 10 times; "
                                    "[16,4,64,64] fp32 operands stay in L2")
    res["gpu_after"] = gpu_info()
    print(json.dumps(res, indent=1), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
