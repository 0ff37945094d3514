"""Generate the committed golden fixtures by running the UNMODIFIED reference (imported from /root/reference
through oracle/ref_harness.py).  Run here (build container) only:

    python tests/golden/make_golden.py [unet] [sched] [msda] [merge] [testr] [manifest] [vae] [clip] [tok] [swinir] [feedback]
                                       [tiled] [msda_ref (on a GPU)]

The reference has no tests or known-answer vectors of its own for this path (SURVEY.md §4), so these fixtures —
outputs of the reference's own modules on seeded inputs/weights — are what pins the oracle; the GPU box, which has
no reference tree, checks the oracle (and through it the CUDA path) against them.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import ref_harness as H  # noqa: E402
from oracle import weights as Wt  # noqa: E402

NARROW = dict(model_channels=64, context_dim=128)


def seeded(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(shape, generator=g) * scale


def gen_manifest():
    path = os.path.join(HERE, "manifests.json")
    out = json.load(open(path)) if os.path.exists(path) else {}
    for name, kw in (("narrow", NARROW), ("full", {})):
        out[f"unet_{name}"] = Wt.manifest_of(H.build_unet(**kw))
        out[f"controlnet_{name}"] = Wt.manifest_of(H.build_controlnet(**kw))
    ts = H.build_testr()
    out["testr"] = Wt.manifest_of(ts)
    with open(os.path.join(HERE, "manifests.json"), "w") as f:
        json.dump(out, f)
    print("manifests:", {k: len(v) for k, v in out.items()})


def gen_unet():
    u, c = H.build_unet(**NARROW), H.build_controlnet(**NARROW)
    u.load_state_dict(Wt.seeded_state_dict(Wt.manifest_of(u)))
    c.load_state_dict(Wt.seeded_state_dict(Wt.manifest_of(c)))
    B = 2
    x, hint = seeded((B, 4, 32, 32), 1), seeded((B, 4, 32, 32), 2)
    ctx = seeded((B, 77, 128), 3)
    t = torch.tensor([999, 500])
    with torch.no_grad():
        ctrl = c(x=x, hint=hint, timesteps=t, context=ctx)
        out, feats = u(x=x, timesteps=t, context=ctx, control=[k.clone() for k in ctrl], only_mid_control=False)
    np.savez_compressed(os.path.join(HERE, "unet_narrow.npz"), t=t.numpy(), out=out.numpy(),
                        ctrl0=ctrl[0][:, ::4, ::2, ::2].numpy(), ctrl12=ctrl[12].numpy()[:, ::4],
                        **{f"feat{i}": f[:, ::4, ::2, ::2].numpy() for i, f in enumerate(feats)})
    print("unet_narrow: out std", out.std().item())


def gen_sched():
    H.install()
    from terediff.model.gaussian_diffusion import enforce_zero_terminal_snr, make_beta_schedule
    from terediff.sampler.spaced_sampler import SpacedSampler
    betas = enforce_zero_terminal_snr(make_beta_schedule("linear", 1000, linear_start=0.00085, linear_end=0.0120))
    s = SpacedSampler(betas, "v", False)
    s.make_schedule(50)
    names = ["sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod",
             "sqrt_recipm1_alphas_cumprod", "posterior_variance", "posterior_log_variance_clipped",
             "posterior_mean_coef1", "posterior_mean_coef2"]
    d = {n: getattr(s, n).numpy() for n in names}
    d["timesteps"] = s.timesteps
    # one p_sample through the reference with a stub model and injected noise
    x, v, noise = seeded((2, 4, 8, 8), 11), seeded((2, 4, 8, 8), 12), seeded((2, 4, 8, 8), 13)
    orig = torch.randn_like
    for idx in (49, 7, 0):
        t = torch.full((2,), idx, dtype=torch.long)
        torch.randn_like = lambda _x: noise
        try:
            xp, _ = s.p_sample(lambda _x, _t, _c: (v, None), x, t, t, {}, None, 1.0)
        finally:
            torch.randn_like = orig
        d[f"x_prev_t{idx}"] = xp.numpy()
    np.savez_compressed(os.path.join(HERE, "schedule_50.npz"), **d)
    print("schedule_50: timesteps", s.timesteps[:4], "...", s.timesteps[-3:])


def gen_msda():
    H.install()
    from testr.adet.layers.ms_deform_attn import ms_deform_attn_core_pytorch
    shapes = [(8, 8), (4, 6), (3, 3)]
    S = sum(h * w for h, w in shapes)
    B, M, D, Lq, L, P = 2, 8, 32, 24, 3, 4
    value = seeded((B, S, M, D), 21)
    loc = torch.rand((B, Lq, M, L, P, 2), generator=torch.Generator().manual_seed(22)) * 1.4 - 0.2
    w = torch.softmax(seeded((B, Lq, M, L * P), 23), -1).view(B, Lq, M, L, P)
    out = ms_deform_attn_core_pytorch(value, shapes, loc, w)
    np.savez_compressed(os.path.join(HERE, "msda_case.npz"), shapes=np.array(shapes), out=out.numpy())
    print("msda_case: out std", out.std().item())


def gen_merge():
    H.install()
    import val_patches as vp
    d = {}
    for name, (oh, ow) in (("a", (200, 300)), ("b", (128, 128)), ("c", (130, 250))):
        n = len(vp.split_image_with_overlap(__import__("PIL.Image", fromlist=["Image"]).fromarray(
            np.zeros((oh, ow, 3), np.uint8)), 128, 16))
        g = torch.Generator().manual_seed(31)
        tl = [torch.rand((1, 3, 512, 512), generator=g) for _ in range(n)]
        m = vp.merge_patches_with_overlap(tl, (oh, ow), 512, 64)
        d[f"{name}_size"] = np.array([oh, ow, n])
        d[f"{name}_sum"] = np.array(m.double().sum().item())
        d[f"{name}_sample"] = m[0, :, ::37, ::41].numpy()
    np.savez_compressed(os.path.join(HERE, "merge_case.npz"), **d)
    print("merge_case:", {k: v.tolist() for k, v in d.items() if k.endswith("size")})


def gen_testr():
    ts = H.build_testr()
    ts.load_state_dict(Wt.seeded_state_dict(Wt.manifest_of(ts)), strict=False)
    B = 1
    feats = [seeded((B, 1280, 16, 16), 41), seeded((B, 1280, 32, 32), 42), seeded((B, 640, 64, 64), 43),
             seeded((B, 320, 64, 64), 44)]
    with torch.no_grad():
        out = ts.testr(feats)
        _, res = ts(feats, None, "VAL")
    r = res[0]
    np.savez_compressed(os.path.join(HERE, "testr_full.npz"), pred_logits=out["pred_logits"].numpy(),
                        pred_ctrl_points=out["pred_ctrl_points"].numpy(), pred_texts=out["pred_texts"].numpy(),
                        enc_logits=out["enc_outputs"]["pred_logits"].numpy()[:, ::8],
                        n_inst=np.array(len(r.scores)), scores=r.scores.numpy(), polygons=r.polygons.numpy(),
                        recs=r.recs.numpy())
    print("testr_full: instances", len(r.scores), "logit std", out["pred_logits"].std().item())


def gen_vae():
    H.install()
    from terediff.model.vae import AutoencoderKL
    dd = dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=[1, 2, 4, 4],
              num_res_blocks=2, attn_resolutions=[], dropout=0.0)
    vae = AutoencoderKL(dd, 4).eval()
    full = Wt.manifest_of(vae)
    man = {k: v for k, v in full.items() if k.startswith(("decoder.", "post_quant_conv."))}
    sd = Wt.seeded_state_dict(full)
    vae.load_state_dict(sd)
    z = seeded((1, 4, 16, 16), 51)
    x = seeded((1, 3, 64, 64), 52).clamp(-1, 1)
    with torch.no_grad():
        img = vae.decode(z)
        moments = vae.encode(x).parameters
    import json
    mf = json.load(open(os.path.join(HERE, "manifests.json")))
    mf["vae_decoder"] = man
    mf["vae"] = full
    json.dump(mf, open(os.path.join(HERE, "manifests.json"), "w"))
    np.savez_compressed(os.path.join(HERE, "vae_decode.npz"), img=img.numpy()[:, :, ::2, ::2], moments=moments.numpy())
    print("vae_decode: img std", img.std().item(), "keys", len(man))


def gen_clip():
    H.install()
    from terediff.model.clip import FrozenOpenCLIPEmbedder
    m = FrozenOpenCLIPEmbedder(1024, dict(image_size=224, layers=32, width=1280, head_width=80, patch_size=14),
                               dict(context_length=77, vocab_size=49408, width=1024, heads=16, layers=24),
                               layer="penultimate").eval()
    man = Wt.manifest_of(m)
    m.load_state_dict(Wt.seeded_state_dict(man), strict=False)
    tokens = torch.randint(0, 49408, (2, 77), generator=torch.Generator().manual_seed(71))
    with torch.no_grad():
        z = m(tokens)
    mf = json.load(open(os.path.join(HERE, "manifests.json")))
    mf["clip_text"] = man
    json.dump(mf, open(os.path.join(HERE, "manifests.json"), "w"))
    np.savez_compressed(os.path.join(HERE, "clip_text.npz"), tokens=tokens.numpy(), z=z.numpy()[:, ::4, ::2])
    print("clip_text: z std", z.std().item(), "keys", len(man))


SWINIR_CFG = dict(img_size=64, patch_size=1, in_chans=3, embed_dim=180, depths=[6] * 8, num_heads=[6] * 8, window_size=8,
                  mlp_ratio=2, sf=8, img_range=1.0, upsampler="nearest+conv", resi_connection="1conv", unshuffle=True,
                  unshuffle_scale=8)


def gen_swinir():
    H.install()
    from terediff.model.swinir import SwinIR
    m = SwinIR(**SWINIR_CFG).eval()
    man = Wt.manifest_of(m)
    sd = Wt.seeded_state_dict(man)
    # keep the integer index buffer and the 0/-100 masks of the reference, seed everything else
    for k, v in m.state_dict().items():
        if k.endswith("relative_position_index") or k.endswith("attn_mask"):
            sd[k] = v.clone()
    m.load_state_dict(sd)
    x = torch.rand((1, 3, 128, 128), generator=torch.Generator().manual_seed(81))
    with torch.no_grad():
        y = m(x)
    mf = json.load(open(os.path.join(HERE, "manifests.json")))
    mf["swinir"] = man
    json.dump(mf, open(os.path.join(HERE, "manifests.json"), "w"))
    np.savez_compressed(os.path.join(HERE, "swinir.npz"), x=x.numpy(), y=y.numpy())
    print("swinir: y std", y.std().item(), "keys", len(man))


def gen_feedback():
    """val_sample with the text-spotting feedback loop (spaced_sampler.py:246-328), run through the UNMODIFIED reference:
    its ControlLDM.forward over the full-size ControlledUnetModel + ControlNet, its TransformerDetector and its
    SpacedSampler.val_sample; 3 steps, batch 1, injected noise, HashClip stand-in for the frozen text encoder."""
    H.install()
    from types import SimpleNamespace
    from terediff.model.cldm import ControlLDM
    from terediff.model.gaussian_diffusion import enforce_zero_terminal_snr, make_beta_schedule
    from terediff.sampler.spaced_sampler import SpacedSampler
    from oracle.val_loop import HashClip
    mf = json.load(open(os.path.join(HERE, "manifests.json")))
    u, c = H.build_unet(), H.build_controlnet()
    u.load_state_dict(Wt.seeded_state_dict(mf["unet_full"]))
    c.load_state_dict(Wt.seeded_state_dict(mf["controlnet_full"]))
    ts = H.build_testr()
    ts.load_state_dict(Wt.seeded_state_dict(mf["testr"]), strict=False)
    cldm = ControlLDM.__new__(ControlLDM)          # the reference forward() without building the 438 M-parameter VAE/CLIP
    torch.nn.Module.__init__(cldm)
    cldm.unet, cldm.controlnet, cldm.control_scales, cldm.clip = u, c, [1.0] * 13, HashClip()
    betas = enforce_zero_terminal_snr(make_beta_schedule("linear", 1000, linear_start=0.00085, linear_end=0.0120))
    s = SpacedSampler(betas, "v", False)
    steps = 3
    x_T, c_img = seeded((1, 4, 64, 64), 9800), seeded((1, 4, 64, 64), 9900)
    noises = [seeded((1, 4, 64, 64), 10000 + i) for i in range(steps)]
    cond = dict(c_txt=cldm.clip.encode(""), c_img=c_img)
    cfg = SimpleNamespace(exp_args=SimpleNamespace(mode="VAL", prompt_style="CAPTION"))
    it = iter(noises)
    xs = []
    orig = torch.randn_like
    orig_p = s.p_sample

    def p_sample(*a, **k):
        out = orig_p(*a, **k)
        xs.append(out[0].clone())
        return out
    s.p_sample = p_sample
    torch.randn_like = lambda _x: next(it)
    try:
        with torch.no_grad():
            x, res = s.val_sample(cldm, "cpu", steps, (1, 4, 64, 64), cond, None, 1.0, x_T=x_T, progress=False, cfg=cfg,
                                  pure_cldm=cldm, ts_model=ts)
    finally:
        torch.randn_like = orig
    np.savez_compressed(os.path.join(HERE, "val_feedback.npz"), x=torch.cat(xs).numpy(),
                        **{f"polys{i}": np.stack(r["pred_polys"]) if r["pred_polys"] else np.zeros((0, 16, 2), np.int32)
                           for i, r in enumerate(res)})
    json.dump({"steps": steps, "timesteps": [int(r["timestep"]) for r in res], "pred_texts": [r["pred_texts"] for r in res],
               "pred_prompt": [r["pred_prompt"] for r in res]}, open(os.path.join(HERE, "val_feedback.json"), "w"), indent=1)
    print("val_feedback:", [(int(r["timestep"]), len(r["pred_texts"])) for r in res], "x std", x.std().item())


def gen_tiled():
    """The reference's make_tiled_fn (terediff/utils/common.py:175-234) where its tree is present.  Without it,
    tair_b200.legacy.make_tiled_fn, which the live comparison with the reference found torch.equal on exactly these
    inputs and cases (the committed tiled_fn.npz was written that way)."""
    if H.available():
        H.install()
        from terediff.utils.common import make_tiled_fn
        src = "reference"
    else:
        from tair_b200.legacy import make_tiled_fn
        src = "tair_b200.legacy (equal to the reference)"
    from oracle.tiles import tiled_fn_case
    x, fn, cases = tiled_fn_case()
    np.savez_compressed(os.path.join(HERE, "tiled_fn.npz"),
                        **{f"out_{size}_{stride}": make_tiled_fn(fn, size, stride, progress=False)(x).numpy()
                           for size, stride in cases})
    print("tiled_fn from", src)


MSDA_REF_CASES = [(2, 300, [(16, 16), (32, 32), (64, 64), (64, 64)]), (3, 77, [(8, 8), (4, 6), (3, 3)]),
                  (1, 9472, [(16, 16), (32, 32), (64, 64), (64, 64)])]
MSDA_REF_ROWS = 32


def msda_ref_key(B, Lq, shapes):
    return f"B{B}_Lq{Lq}_L{len(shapes)}"


def gen_msda_ref(out_dir=HERE):
    """On a GPU: the reference's own MSDeformAttn CUDA kernel (oracle/_ref/libmsda_ref.so, oracle/build_ref.sh) on the
    seeded inputs of tests/test_msda_ref_gpu.py, a fixed seeded sample of MSDA_REF_ROWS output rows per case.  Without
    that library, tair_msda_forward in fp32, which was measured bit-identical to the reference kernel on exactly these
    inputs (max |difference| 0.0 on all three cases; the committed msda_ref_cases.npz was written that way)."""
    import ctypes as C
    from oracle.msda import ref_kernel_case
    ref_so = os.path.join(os.path.dirname(os.path.dirname(HERE)), "oracle", "_ref", "libmsda_ref.so")
    d = {}
    for i, (B, Lq, shapes) in enumerate(MSDA_REF_CASES):
        value, shp, start, loc, w = ref_kernel_case(B, Lq, shapes)
        if os.path.exists(ref_so):
            out = torch.empty(B, Lq, 8 * 32, device="cuda")
            rc = C.CDLL(ref_so).msda_ref_forward_f32(*(C.c_void_p(t.data_ptr()) for t in (value, shp, start, loc, w, out)),
                                                     B, value.shape[1], 8, 32, len(shapes), Lq, 4,
                                                     C.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0
            src = "reference kernel"
        else:
            from tair_b200 import ops
            out = ops.msda_forward(value, shp, start, loc, w)
            src = "tair_msda_forward (bit-identical to the reference kernel)"
        rows = np.sort(np.random.default_rng(i).choice(B * Lq, MSDA_REF_ROWS, replace=False))
        k = msda_ref_key(B, Lq, shapes)
        d[k + "_rows"] = rows
        d[k + "_out"] = out.reshape(B * Lq, -1).cpu().numpy()[rows]
    np.savez_compressed(os.path.join(out_dir, "msda_ref_cases.npz"), **d)
    print("msda_ref_cases from", src)


TOKENIZER_CASES = ["", "A realistic scene where the texts \"HELLO\", \"world\" appear clearly on signs.",
                   "it's  a  test &amp;amp; more!!!  123 4.5", "na\u00efve caf\u00e9 \u2014 \u65e5\u672c\u8a9e", "x" * 400,
                   "<start_of_text> hi <end_of_text>", "don't we'll I'm they've you'd HE'S", "  \t\n  ",
                   "exit, 24, OPEN, coffee, P, no-parking"]


def gen_tok():
    H.install()
    import random
    import string
    from terediff.model.open_clip import tokenizer as RT
    rnd = random.Random(0)
    cases = TOKENIZER_CASES + ["".join(rnd.choice(string.printable) for _ in range(rnd.randint(0, 120))) for _ in range(40)]
    ids = RT.tokenize(cases)
    json.dump({"texts": cases, "ids": [[int(v) for v in row] for row in ids]},
              open(os.path.join(HERE, "tokenizer_cases.json"), "w"))
    print("tokenizer_cases:", len(cases))


if __name__ == "__main__":
    what = sys.argv[1:] or ["manifest", "unet", "sched", "msda", "merge", "testr"]
    torch.manual_seed(0)
    for w in what:
        {"manifest": gen_manifest, "unet": gen_unet, "sched": gen_sched, "msda": gen_msda, "merge": gen_merge,
         "testr": gen_testr, "vae": gen_vae, "clip": gen_clip, "tok": gen_tok, "swinir": gen_swinir, "feedback": gen_feedback,
         "tiled": gen_tiled, "msda_ref": gen_msda_ref}[w]()
