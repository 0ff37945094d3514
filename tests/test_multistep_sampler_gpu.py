"""DDIM and DPM-Solver++(2M) on the B200: the fused multistep update bit for bit against a torch fp32 restatement, the
samplers against the float64 oracle on an analytic model, and the loops (CUDA graph, rescaled CFG, batch independence,
text-spotting feedback, tile driver) on the full-size seeded ControlLDM."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_pipeline_gpu import cond_fn, decode_fn, narrow_model
from test_sampler_gpu import STEP_TOL, HashClip, full_cfgs, inputs

pytestmark = pytest.mark.gpu


def ref_update(x, v, noise, t, tabs, hist, v_uncond=None, cfg_scale=1.0):
    """The kernel's arithmetic in torch fp32, in the kernel's order; history not read where c == 0."""
    ex = lambda tb: tb.gather(0, t).view(-1, *([1] * (x.dim() - 1)))   # noqa: E731
    P, Q, a, b, c, d = (ex(tb) for tb in tabs)
    if v_uncond is not None:
        v = v_uncond + cfg_scale * (v - v_uncond)
    x0 = P * x - Q * v
    h = torch.where(c == 0, torch.zeros_like(hist), hist)
    return ((b * x0 + a * x) + c * h) + d * noise, x0


def test_multistep_update_bit_exact(cuda_lib):
    from oracle import weights
    from tair_b200 import ops
    g = torch.Generator().manual_seed(5)
    tabs = [torch.rand(10, generator=g).cuda() for _ in range(6)]
    tabs[4][[0, 7]] = 0.0                                     # c == 0 on rows 0 and 7
    x, v, vu, nz, hist = (weights.seeded_randn((3, 4, 64, 64), 2000 + k).cuda() for k in range(5))
    t = torch.tensor([7, 2, 5], device="cuda")                 # a different row per sample, one with c == 0
    scale_dev = torch.full((1,), 3.5, device="cuda")
    for kw in (dict(), dict(v_uncond=vu, cfg_scale=4.0), dict(v_uncond=vu, cfg_scale=1.0, cfg_scale_dev=scale_dev)):
        scale = 3.5 if "cfg_scale_dev" in kw else kw.get("cfg_scale", 1.0)
        h = hist.clone()
        out = ops.sampler_multistep_update(x, v, nz, t, tabs, x0_hist=h, **kw)
        ref, x0 = ref_update(x, v, nz, t, tabs, hist, kw.get("v_uncond"), scale)
        assert torch.equal(out, ref) and torch.equal(h, x0), kw
    # c == 0 everywhere the batch looks: NaN history is not read, and now holds x0
    t0 = torch.tensor([0, 7, 0], device="cuda")
    h = torch.full_like(x, float("nan"))
    out = ops.sampler_multistep_update(x, v, nz, t0, tabs, x0_hist=h)
    ref, x0 = ref_update(x, v, nz, t0, tabs, torch.zeros_like(x))
    assert torch.isfinite(out).all() and torch.equal(out, ref) and torch.equal(h, x0)


class AnalyticModel:
    """v-prediction of data x0 ~ N(mu, s^2), with abar read from a device table (capturable in a CUDA graph)."""

    def __init__(self, betas, mu, s):
        self.abar = torch.tensor(np.cumprod(1.0 - betas), dtype=torch.float64, device="cuda")
        self.mu, self.s = mu, s

    def __call__(self, x, model_t, cond):
        ab = self.abar[model_t].view(-1, 1, 1, 1)
        al, x64 = ab.sqrt(), x.double()
        x0 = self.mu + al * self.s ** 2 / (ab * self.s ** 2 + (1 - ab)) * (x64 - al * self.mu)
        return ((al * x64 - x0) / (1 - ab).sqrt()).float(), None


@pytest.mark.parametrize("kind", ["ddim", "dpmpp2m"])
def test_analytic_model_matches_float64_oracle(cuda_lib, kind):
    from oracle import multistep_sampler as OM, sampler as OS
    from tair_b200.sampler import DDIMSampler, DPMSolverSampler
    betas = OS.diffusion_betas()
    s = (DDIMSampler if kind == "ddim" else DPMSolverSampler)(betas)
    model = AnalyticModel(betas, 0.3, 0.7)
    x_T = torch.randn((2, 4, 64, 64), generator=torch.Generator().manual_seed(9)).cuda()
    ref = []
    OM.sample_loop(OM.GaussianData(0.3, 0.7).x0_hat, betas, 20, x_T.double().cpu().numpy(), kind, trace=ref)
    outs = []
    for graph in (True, False):
        s.trace = []
        out, _ = s.sample(model, "cuda", 20, tuple(x_T.shape), {}, None, 1.0, x_T=x_T, progress=False,
                          use_cuda_graph=graph)
        for i, (rec, r) in enumerate(zip(s.trace, ref)):
            err = np.abs(rec["x"].double().cpu().numpy() - r).max() / np.abs(r).max()
            assert err < 1e-5, (graph, i, err)
        outs.append(out)
    s.trace = None
    assert torch.equal(outs[0], outs[1])


@pytest.fixture(scope="module")
def cldm(cuda_lib, manifests):
    from oracle import weights
    from tair_b200.model import ControlLDM
    usd = weights.seeded_state_dict(manifests["unet_full"])
    csd = weights.seeded_state_dict(manifests["controlnet_full"])
    m = ControlLDM(*full_cfgs())
    m.unet.load_state_dict(usd)
    m.controlnet.load_state_dict(csd)
    return m.cuda().eval(), {k: v.cuda() for k, v in usd.items()}, {k: v.cuda() for k, v in csd.items()}


def make(kind, **kw):
    from tair_b200.model.gaussian_diffusion import val_diffusion
    from tair_b200.sampler import DDIMSampler, DPMSolverSampler
    betas = val_diffusion().betas
    if kind == "dpmpp2m":
        return DPMSolverSampler(betas, "v", kw.get("rescale_cfg", False))
    return DDIMSampler(betas, "v", kw.get("rescale_cfg", False), eta=kw.get("eta", 0.0))


N_TF = 20


@pytest.mark.parametrize("kind,eta", [("ddim", 0.0), ("ddim", 1.0), ("dpmpp2m", 0.0)])
@pytest.mark.parametrize("i", [0, 1, 2, N_TF - 1])
def test_teacher_forced_step(cldm, kind, eta, i):
    """One step of the product (bf16 network + fused update) against the fp32 oracle network + the float64 textbook
    update; from i >= 1 the history holds the same x0_hat the oracle is given (step 2 is the first second-order step)."""
    from oracle import multistep_sampler as OM, sampler as OS, unet as OU, weights
    m, usd, csd = cldm
    s = make(kind, eta=eta)
    s.make_schedule(N_TF)
    s.to("cuda")
    taus, abar, abar_next = OM.schedule(OS.diffusion_betas(), N_TF)
    x, c_img, c_txt = inputs(2, seed=60 + i)
    noise = weights.seeded_randn((2, 4, 64, 64), 600 + i).cuda()
    m_prev = weights.seeded_randn((2, 4, 64, 64), 700 + i).cuda()
    s.x0_history(x).copy_(m_prev)
    model_t = torch.full((2,), int(taus[i]), device="cuda", dtype=torch.long)
    t = torch.full((2,), N_TF - 1 - i, device="cuda", dtype=torch.long)
    with torch.no_grad():
        v, _ = OU.cldm_forward(usd, csd, x, model_t, c_txt, c_img)
    x64, v64, z64, mp64 = (a.double().cpu().numpy() for a in (x, v, noise, m_prev))
    m0 = np.sqrt(abar[i]) * x64 - np.sqrt(1 - abar[i]) * v64
    if kind == "ddim":
        ref = OM.ddim_step(x64, m0, abar[i], abar_next[i], eta, z64)
    else:
        ref = OM.dpmpp2m_step(x64, m0, abar[i], abar_next[i], mp64 if i else None, abar[i - 1] if i else None)
    out, _ = s.p_sample(m, x, model_t, t, dict(c_txt=c_txt, c_img=c_img), None, 1.0, noise=noise)
    err = np.abs(out.double().cpu().numpy() - ref).max() / np.abs(ref).max()
    assert err < STEP_TOL, err


def run_both(s, m, steps, x_T, cond, uncond=None, scale=1.0, noises=None):
    outs = []
    s.noise_fn = None if noises is None else (lambda i, x: noises[i])
    try:
        for graph in (True, False):
            o, _ = s.sample(m, "cuda", steps, tuple(x_T.shape), cond, uncond, scale, x_T=x_T, progress=False,
                            use_cuda_graph=graph)
            outs.append(o)
    finally:
        s.noise_fn = None
    return outs


@pytest.mark.parametrize("kind,eta", [("ddim", 0.0), ("ddim", 1.0), ("dpmpp2m", 0.0)])
def test_sample_graph_equals_eager(cldm, kind, eta):
    from oracle import weights
    m = cldm[0]
    s = make(kind, eta=eta)
    x_T, c_img, c_txt = inputs(1, seed=71)
    noises = [weights.seeded_randn((1, 4, 64, 64), 1700 + k).cuda() for k in range(4)]
    g, e = run_both(s, m, 4, x_T, dict(c_txt=c_txt, c_img=c_img), noises=noises)
    assert torch.isfinite(g).all() and torch.equal(g, e)


def test_graph_follows_schedule_changes(cldm):
    """4 -> 3 -> 4 steps on one sampler: the tables and the history follow the schedule, graph == eager each time."""
    m = cldm[0]
    s = make("dpmpp2m")
    x_T, c_img, c_txt = inputs(1, seed=72)
    for steps in (4, 3, 4):
        g, e = run_both(s, m, steps, x_T, dict(c_txt=c_txt, c_img=c_img))
        assert torch.equal(g, e), steps


def test_rescaled_cfg_uses_one_graph(cldm):
    from oracle import weights
    m = cldm[0]
    s = make("dpmpp2m", rescale_cfg=True)
    x_T, c_img, c_txt = inputs(1, seed=73)
    un = dict(c_txt=weights.seeded_randn((1, 77, 1024), 1773).cuda(), c_img=c_img)
    g, e = run_both(s, m, 4, x_T, dict(c_txt=c_txt, c_img=c_img), un, 4.0)
    assert torch.equal(g, e)
    assert len(s._graphs) == 1 and all(st.graph is not None for st in s._graphs.values())


def test_bench_batch_tiles_equal_single_tiles(cldm):
    """B=16, a second-order DPM-Solver++ step (history read): tiles 0, 7 and 15 equal the same tile run alone."""
    from oracle import weights
    m = cldm[0]
    s = make("dpmpp2m")
    s.make_schedule(N_TF)
    s.to("cuda")
    B, i = 16, 5
    x, c_img, c_txt = inputs(B, seed=74)
    hist = weights.seeded_randn((B, 4, 64, 64), 1774).cuda()
    noise = torch.zeros_like(x)
    model_t = torch.full((B,), int(s.timesteps[N_TF - 1 - i]), device="cuda", dtype=torch.long)
    t = torch.full((B,), N_TF - 1 - i, device="cuda", dtype=torch.long)
    assert s.ms_c[N_TF - 1 - i].item() != 0.0
    s.x0_history(x).copy_(hist)
    out, _ = s.p_sample(m, x, model_t, t, dict(c_txt=c_txt, c_img=c_img), None, 1.0, noise=noise)
    for b in (0, 7, 15):
        sl = slice(b, b + 1)
        s.x0_history(x[sl]).copy_(hist[sl])
        one, _ = s.p_sample(m, x[sl], model_t[sl], t[sl], dict(c_txt=c_txt[sl], c_img=c_img[sl]), None, 1.0,
                            noise=noise[sl])
        assert torch.equal(one, out[sl]), b


def test_val_sample_with_text_spotting_feedback(cldm, manifests):
    from oracle import weights
    from tair_b200.testr import TransformerDetector, default_cfg
    m = cldm[0]
    det = TransformerDetector(default_cfg("cuda"))
    det.load_state_dict(weights.seeded_state_dict(manifests["testr"]))
    det = det.cuda().eval()
    old = m.clip
    m.attach_clip(HashClip())
    s = make("dpmpp2m")
    B = 2
    x_T, c_img, _ = inputs(B, seed=75)
    cfg = SimpleNamespace(exp_args=SimpleNamespace(mode="VAL", prompt_style="CAPTION"))
    try:
        outs = []
        for graph in (True, False):
            cond = dict(c_txt=m.clip.encode([""] * B), c_img=c_img)
            first = cond["c_txt"].clone()
            x, res = s.val_sample(m, "cuda", 3, (B, 4, 64, 64), cond, None, 1.0, x_T=x_T, progress=False, cfg=cfg,
                                  pure_cldm=m, ts_model=det, use_cuda_graph=graph)
            assert torch.isfinite(x).all() and not torch.equal(cond["c_txt"], first)
            assert [r["timestep"] for r in res] == [999, 500, 0]
            for r in res:
                assert set(r) >= {"timestep", "pred_texts", "pred_prompt", "pred_polys"}
                assert len(r["batch_prompts"]) == B and len(r["pred_texts"]) == len(r["pred_polys"])
            outs.append(x)
        assert torch.equal(outs[0], outs[1])
    finally:
        m.attach_clip(old)


def test_restore_image_is_independent_of_tile_batching(cuda_lib, manifests):
    from tair_b200 import pipeline
    m = narrow_model(manifests)
    s = make("dpmpp2m")
    lq = np.random.default_rng(0).integers(0, 256, (200, 300, 3), dtype=np.uint8)   # 2 x 3 tiles
    a = pipeline.restore_image(lq, m, s, cond_fn=cond_fn, decode_fn=decode_fn, steps=4, tile_batch=4)
    b = pipeline.restore_image(lq, m, s, cond_fn=cond_fn, decode_fn=decode_fn, steps=4, tile_batch=1)
    assert a.shape == (1, 3, 800, 1200) and torch.isfinite(a).all() and torch.equal(a, b)
