"""UniPC on the B200: the fused update bit for bit against a torch fp32 restatement of its documented evaluation order,
the sampler against the float64 paper-form oracle on an analytic model, and the loops (CUDA graph, schedule and order
changes, rescaled CFG, batch independence, text-spotting feedback, tile driver, two samplers on one model) on the
full-size seeded ControlLDM."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from test_multistep_sampler_gpu import N_TF, AnalyticModel, cldm, run_both  # noqa: F401  (cldm is a fixture)
from test_pipeline_gpu import cond_fn, decode_fn, narrow_model
from test_sampler_gpu import STEP_TOL, HashClip, inputs

pytestmark = pytest.mark.gpu


def ref_update(x, v, t, table, x_corr, hist, v_uncond=None, cfg_scale=1.0):
    """The kernel's arithmetic in torch fp32, in the documented order: each term added (left to right, from 0) only
    where its coefficient is non-zero; then the state update.  -> (x_next, x_corr, x0_hist) after the step."""
    K = hist.shape[0]
    rows = table[t]
    col = lambda j: rows[:, j].view(-1, *([1] * (x.dim() - 1)))   # noqa: E731
    if v_uncond is not None:
        v = v_uncond + cfg_scale * (v - v_uncond)
    x0 = col(0) * x - col(1) * v

    def acc(terms):
        out = torch.zeros_like(x)
        for c, term in terms:
            out = torch.where(c != 0, out + c * term, out)
        return out
    xc = acc([(col(2), x), (col(3), x_corr), (col(4), x0)] + [(col(5 + k), hist[k]) for k in range(K)])
    xn = acc([(col(8), xc), (col(9), x0)] + [(col(10 + k), hist[k]) for k in range(K)])
    return xn, xc, torch.stack([x0] + [hist[k - 1] for k in range(1, K)])


def same(a, b):
    """Bit equality that also lets NaN (a stale slot the shift moved on) equal NaN."""
    return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(a.nan_to_num(0.0), b.nan_to_num(0.0))


def test_unipc_update_bit_exact(cuda_lib):
    from oracle import weights
    from tair_b200 import _lib, ops
    g = torch.Generator().manual_seed(11)
    table = (torch.rand(10, 16, generator=g) - 0.3)
    table[:, 13:] = 0.0
    table[7, 2:13] = 0.0                                        # a first step: no correction, first-order predictor
    table[7, 2], table[7, 9] = 1.0, 0.7
    table[4, 2] = 0.0                                           # corrector of order 1, predictor of order 2
    table[4, 6:8] = 0.0
    table[4, 11:13] = 0.0
    table = table.cuda()
    shape = (3, 4, 64, 64)
    x, v, vu = (weights.seeded_randn(shape, 3000 + k).cuda() for k in range(3))
    xc0 = weights.seeded_randn(shape, 3010).cuda()
    t = torch.tensor([7, 4, 2], device="cuda")
    scale_dev = torch.full((1,), 3.5, device="cuda")
    for K in (1, 2, 3):
        hist0 = weights.seeded_randn((K,) + shape, 3020 + K).cuda()
        # state that no coefficient of the sample's row uses is NaN: sample 0 (row 7) uses none, sample 1 (row 4)
        # uses x_corr and h0 only
        xc0n, hist0n = xc0.clone(), hist0.clone()
        xc0n[0] = float("nan")
        hist0n[:, 0] = float("nan")
        hist0n[1:, 1] = float("nan")
        for kw in (dict(), dict(v_uncond=vu, cfg_scale=4.0), dict(v_uncond=vu, cfg_scale=1.0, cfg_scale_dev=scale_dev)):
            scale = 3.5 if "cfg_scale_dev" in kw else kw.get("cfg_scale", 1.0)
            for xcs, hs in ((xc0, hist0), (xc0n, hist0n)):
                xc, h = xcs.clone(), hs.clone()
                out = ops.sampler_unipc_update(x, v, t, table, x_corr=xc, x0_hist=h, **kw)
                rn, rc, rh = ref_update(x, v, t, table, xcs, hs, kw.get("v_uncond"), scale)
                assert torch.isfinite(out).all() and torch.isfinite(xc).all(), (K, kw)
                assert torch.equal(out, rn) and torch.equal(xc, rc) and same(h, rh), (K, kw)
        # a step without correction returns xc = x exactly
        assert torch.equal(xc[0], x[0])
    # validation errors come back through tair_last_error()
    xc, h = xc0.clone(), weights.seeded_randn((2,) + shape, 3030).cuda()
    with pytest.raises(_lib.TairError, match="x_next must not alias"):
        ops.sampler_unipc_update(x, v, t, table, x_corr=xc, x0_hist=h, out=x)
    with pytest.raises(_lib.TairError, match="x_corr and x0_hist must not alias"):
        ops.sampler_unipc_update(x, v, t, table, x_corr=h[1], x0_hist=h)
    out = torch.empty_like(x)
    rc = _lib.lib().tair_sampler_unipc_update(x.data_ptr(), v.data_ptr(), None, 1.0, None, out.data_ptr(),
                                              xc.data_ptr(), h.data_ptr(), t.data_ptr(), table.data_ptr(), 4, 3,
                                              4 * 64 * 64, None)
    assert rc == -1 and b"history depth" in _lib.lib().tair_last_error()


@pytest.mark.parametrize("order,corrector", [(1, True), (2, True), (3, True), (2, False)])
def test_analytic_model_matches_float64_oracle(cuda_lib, order, corrector):
    from oracle import sampler as OS, unipc_sampler as OU
    from tair_b200.sampler import UniPCSampler
    betas = OS.diffusion_betas()
    s = UniPCSampler(betas, order=order, corrector=corrector)
    model = AnalyticModel(betas, 0.3, 0.7)
    x_T = torch.randn((2, 4, 64, 64), generator=torch.Generator().manual_seed(19)).cuda()
    ref = []
    OU.sample_loop(OU.GaussianData(0.3, 0.7).x0_hat, betas, 20, x_T.double().cpu().numpy(), "unipc", order=order,
                   corrector=corrector, trace=ref)
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


def make(order=2, **kw):
    from tair_b200.model.gaussian_diffusion import val_diffusion
    from tair_b200.sampler import UniPCSampler
    return UniPCSampler(val_diffusion().betas, "v", kw.get("rescale_cfg", False), order=order,
                        corrector=kw.get("corrector", True))


@pytest.mark.parametrize("order", [2, 3])
@pytest.mark.parametrize("i", [0, 1, 2, 5, N_TF - 1])
def test_teacher_forced_step(cldm, order, i):
    """One step of the product (bf16 network + fused update) against the fp32 oracle network + the float64 paper-form
    corrector and predictor, from the same seeded state (corrected latent and x0 history of the previous steps)."""
    from oracle import multistep_sampler as OM, sampler as OS, unet as OU, unipc_sampler as OP, weights
    m, usd, csd = cldm
    s = make(order)
    s.make_schedule(N_TF)
    s.to("cuda")
    orders = s.host_tables(N_TF)["orders"]
    taus, abar, abar_next = OM.schedule(OS.diffusion_betas(), N_TF)
    x, c_img, c_txt = inputs(2, seed=80 + i)
    xc_prev = weights.seeded_randn((2, 4, 64, 64), 800 + i).cuda()
    hist = weights.seeded_randn((order, 2, 4, 64, 64), 900 + i).cuda()      # h_k = x0 of step i-1-k
    x_corr, x0_hist = s.state_buffers(x)
    x_corr.copy_(xc_prev)
    x0_hist.copy_(hist)
    model_t = torch.full((2,), int(taus[i]), device="cuda", dtype=torch.long)
    t = torch.full((2,), N_TF - 1 - i, device="cuda", dtype=torch.long)
    with torch.no_grad():
        v, _ = OU.cldm_forward(usd, csd, x, model_t, c_txt, c_img)
    x64, v64, xc64 = (a.double().cpu().numpy() for a in (x, v, xc_prev))
    h64 = hist.double().cpu().numpy()
    m0 = np.sqrt(abar[i]) * x64 - np.sqrt(1 - abar[i]) * v64
    n_hist = min(i, order)
    ms = [h64[k] for k in reversed(range(n_hist))]                           # oldest first
    lams = [OM._lam(abar[i - 1 - k]) for k in reversed(range(n_hist))]
    ref, ref_xc, p = OP.unipc_step(x64, xc64, m0, ms, lams, abar[i], abar[i - 1] if i else None, abar_next[i], order,
                                   int(orders[i - 1]) if i else None, i, N_TF)
    assert p == orders[i]
    out, _ = s.p_sample(m, x, model_t, t, dict(c_txt=c_txt, c_img=c_img), None, 1.0)
    err = np.abs(out.double().cpu().numpy() - ref).max() / np.abs(ref).max()
    assert err < STEP_TOL, err
    err = np.abs(x_corr.double().cpu().numpy() - ref_xc).max() / np.abs(ref_xc).max()
    assert err < STEP_TOL, err


@pytest.mark.parametrize("order,corrector", [(1, True), (2, True), (3, True), (3, False)])
def test_sample_graph_equals_eager(cldm, order, corrector):
    m = cldm[0]
    s = make(order, corrector=corrector)
    x_T, c_img, c_txt = inputs(1, seed=81)
    g, e = run_both(s, m, 6, x_T, dict(c_txt=c_txt, c_img=c_img))
    assert torch.isfinite(g).all() and torch.equal(g, e)


def test_graph_follows_schedule_and_order_changes(cldm):
    """10 -> 15 steps, then order 2 -> 3 -> 2 on one sampler: graph == eager each time, and the order-3 run equals a
    fresh order-3 sampler's."""
    m = cldm[0]
    s = make(2)
    x_T, c_img, c_txt = inputs(1, seed=82)
    cond = dict(c_txt=c_txt, c_img=c_img)
    res = {}
    for steps, order in ((10, 2), (15, 2), (15, 3), (15, 2)):
        s.order = order
        g, e = run_both(s, m, steps, x_T, cond)
        assert torch.equal(g, e), (steps, order)
        if (steps, order) in res:
            assert torch.equal(res[steps, order], g), (steps, order)
        res[steps, order] = g
    fresh, _ = make(3).sample(m, "cuda", 15, tuple(x_T.shape), cond, None, 1.0, x_T=x_T, progress=False,
                              use_cuda_graph=True)
    assert torch.equal(fresh, res[15, 3]) and not torch.equal(res[15, 2], res[15, 3])


def test_rescaled_cfg_uses_one_graph(cldm):
    from oracle import weights
    m = cldm[0]
    s = make(2, rescale_cfg=True)
    x_T, c_img, c_txt = inputs(1, seed=83)
    un = dict(c_txt=weights.seeded_randn((1, 77, 1024), 1883).cuda(), c_img=c_img)
    g, e = run_both(s, m, 5, x_T, dict(c_txt=c_txt, c_img=c_img), un, 4.0)
    assert torch.equal(g, e)
    assert len(s._graphs) == 1 and all(st.graph is not None for st in s._graphs.values())


def test_bench_batch_tiles_equal_single_tiles(cldm):
    """B=16, a third-order step with correction (every state slot read): tiles 0, 7 and 15 equal the same tile alone."""
    from oracle import weights
    m = cldm[0]
    s = make(3)
    s.make_schedule(N_TF)
    s.to("cuda")
    B, i = 16, 5
    x, c_img, c_txt = inputs(B, seed=84)
    xc_prev = weights.seeded_randn((B, 4, 64, 64), 1884).cuda()
    hist = weights.seeded_randn((3, B, 4, 64, 64), 1885).cuda()
    model_t = torch.full((B,), int(s.timesteps[N_TF - 1 - i]), device="cuda", dtype=torch.long)
    t = torch.full((B,), N_TF - 1 - i, device="cuda", dtype=torch.long)
    assert (s.unipc_table[N_TF - 1 - i, 5:8] != 0).all() and (s.unipc_table[N_TF - 1 - i, 10:12] != 0).all()
    xc, h = s.state_buffers(x)
    xc.copy_(xc_prev)
    h.copy_(hist)
    out, _ = s.p_sample(m, x, model_t, t, dict(c_txt=c_txt, c_img=c_img), None, 1.0)
    for b in (0, 7, 15):
        sl = slice(b, b + 1)
        xc1, h1 = s.state_buffers(x[sl])
        xc1.copy_(xc_prev[sl])
        h1.copy_(hist[:, sl])
        one, _ = s.p_sample(m, x[sl], model_t[sl], t[sl], dict(c_txt=c_txt[sl], c_img=c_img[sl]), None, 1.0)
        assert torch.equal(one, out[sl]), b


def test_two_samplers_alternating_on_one_model(cldm):
    """UniPC-2 and UniPC-3 stepping alternately on one model give what each gives alone (no shared state)."""
    m = cldm[0]
    x_T, c_img, c_txt = inputs(1, seed=85)
    cond = dict(c_txt=c_txt, c_img=c_img)
    N = 6
    alone = [make(o).sample(m, "cuda", N, tuple(x_T.shape), cond, None, 1.0, x_T=x_T, progress=False)[0]
             for o in (2, 3)]
    a, b = make(2), make(3)
    xs = {}
    for s in (a, b):
        s.make_schedule(N)
        s.to("cuda")
        xs[s] = x_T.clone()
    for i in range(N):
        for s in (a, b):
            model_t = torch.full((1,), int(s.timesteps[N - 1 - i]), device="cuda", dtype=torch.long)
            t = torch.full((1,), N - 1 - i, device="cuda", dtype=torch.long)
            xs[s], _ = s.p_sample(m, xs[s], model_t, t, cond, None, 1.0)
    assert torch.equal(xs[a], alone[0]) and torch.equal(xs[b], alone[1])
    # whole graph-replayed runs, alternating
    for _ in range(2):
        for s, ref in ((a, alone[0]), (b, alone[1])):
            out, _ = s.sample(m, "cuda", N, tuple(x_T.shape), cond, None, 1.0, x_T=x_T, progress=False,
                              use_cuda_graph=True)
            assert torch.equal(out, ref)


def test_val_sample_with_text_spotting_feedback(cldm, manifests):
    from oracle import weights
    from tair_b200.testr import TransformerDetector, default_cfg
    m = cldm[0]
    det = TransformerDetector(default_cfg("cuda"))
    det.load_state_dict(weights.seeded_state_dict(manifests["testr"]))
    det = det.cuda().eval()
    old = m.clip
    m.attach_clip(HashClip())
    s = make(2)
    B = 2
    x_T, c_img, _ = inputs(B, seed=86)
    cfg = SimpleNamespace(exp_args=SimpleNamespace(mode="VAL", prompt_style="CAPTION"))
    try:
        outs = []
        for graph in (True, False):
            cond = dict(c_txt=m.clip.encode([""] * B), c_img=c_img)
            first = cond["c_txt"].clone()
            x, res = s.val_sample(m, "cuda", 4, (B, 4, 64, 64), cond, None, 1.0, x_T=x_T, progress=False, cfg=cfg,
                                  pure_cldm=m, ts_model=det, use_cuda_graph=graph)
            assert torch.isfinite(x).all() and not torch.equal(cond["c_txt"], first)
            assert [r["timestep"] for r in res] == [999, 666, 333, 0]
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
    s = make(3)
    lq = np.random.default_rng(1).integers(0, 256, (200, 300, 3), dtype=np.uint8)   # 2 x 3 tiles
    a = pipeline.restore_image(lq, m, s, cond_fn=cond_fn, decode_fn=decode_fn, steps=5, tile_batch=4)
    b = pipeline.restore_image(lq, m, s, cond_fn=cond_fn, decode_fn=decode_fn, steps=5, tile_batch=1)
    assert a.shape == (1, 3, 800, 1200) and torch.isfinite(a).all() and torch.equal(a, b)
