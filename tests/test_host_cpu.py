"""Host-side logic that needs no GPU: character codec and prompt templates (terediff/dataset/utils.py:18-40,
spaced_sampler.py:298-317), the Instances container (detectron2 structures/instances.py:8-144), the respaced schedule
tables against the reference fixture, and the GroupNorm-free pieces of the sampler API."""
import numpy as np
import pytest
import torch

from tair_b200 import prompt
from tair_b200.testr.structures import Instances


def test_character_table_and_codec_round_trip():
    assert len(prompt.CTLABELS) == 95 and prompt.CTLABELS[0] == " " and prompt.CTLABELS[-1] == "~"
    assert prompt.CTLABELS[33] == "A" and prompt.CTLABELS[65] == "a" and prompt.CTLABELS[16] == "0"
    for word in ("EXIT", "no-parking", "24/7 OPEN!", "", "x" * 25):
        idx = prompt.encode(word)
        assert len(idx) == 25 and all(i == 96 for i in idx[len(word):])
        assert prompt.decode(idx) == word                      # decode stops at the first pad index
    assert prompt.decode([33, 34, 200, 35]) == "AB"            # ... or at any index outside the table
    assert prompt.decode(torch.tensor([40, 41, 96, 96])) == "HI"


def test_prompt_templates_match_reference_strings():
    assert prompt.build_prompt(["EXIT", "24"], "CAPTION") == \
        'A realistic scene where the texts "EXIT", "24" appear clearly on signs, boards, buildings, or other objects.'
    assert prompt.build_prompt([], "CAPTION") == \
        "A realistic scene where the texts  appear clearly on signs, boards, buildings, or other objects."
    assert prompt.build_prompt(["a", "b"], "TAG") == '"a", "b"'
    with pytest.raises(ValueError):
        prompt.build_prompt(["a"], "POEM")


def test_decode_texts_batches_instances():
    a, b = Instances((512, 512)), Instances((512, 512))
    a.recs = torch.tensor([prompt.encode("STOP"), prompt.encode("go")])
    a.polygons = torch.arange(64, dtype=torch.float32).view(2, 32) + 0.7
    b.recs = torch.zeros((0, 25), dtype=torch.long)
    b.polygons = torch.zeros((0, 32))
    texts, polys = prompt.decode_texts([a, b])
    assert texts == [["STOP", "go"], []]
    assert len(polys[0]) == 2 and polys[0][0].shape == (16, 2) and polys[0][0].dtype == np.int32 and polys[1] == []
    assert polys[0][1][0, 0] == 32                            # float -> int32 truncation as .astype(np.int32)


def test_instances_container_semantics():
    r = Instances((480, 640))
    assert r.image_size == (480, 640)
    with pytest.raises(NotImplementedError):                   # as detectron2: an empty container has no length
        len(r)
    r.scores = torch.tensor([0.9, 0.6, 0.8])
    r.set("recs", torch.zeros((3, 25), dtype=torch.long))
    assert len(r) == 3 and r.has("scores") and not r.has("polygons")
    assert set(r.get_fields()) == {"scores", "recs"} and torch.equal(r.get("scores"), r.scores)
    with pytest.raises(AssertionError):
        r.polygons = torch.zeros((2, 32))                      # every field must share the instance count
    with pytest.raises(AttributeError):
        _ = r.beziers


def test_spaced_schedule_matches_reference_fixture(golden):
    """make_schedule(50) on the CPU: the respaced timestep set and all eight fp32 tables of the reference
    (spaced_sampler.py:77-121), including the inf at the zero-terminal-SNR end of sqrt_recip*_alphas_cumprod."""
    from tair_b200.model.gaussian_diffusion import val_diffusion
    from tair_b200.sampler import SpacedSampler
    g = golden("schedule_50.npz")
    s = SpacedSampler(val_diffusion().betas, "v", False)
    s.make_schedule(50)
    assert np.array_equal(np.asarray(s.timesteps), g["timesteps"]) and len(s.timesteps) == 50
    for name in ("sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod",
                 "sqrt_recipm1_alphas_cumprod", "posterior_variance", "posterior_log_variance_clipped",
                 "posterior_mean_coef1", "posterior_mean_coef2"):
        got = getattr(s, name).numpy()
        assert got.dtype == np.float32 and np.array_equal(got, g[name], equal_nan=True), name
    assert np.isinf(s.sqrt_recip_alphas_cumprod.numpy()[-1])


def _shapes(m, skip_suffix=()):
    return {k: list(v.shape) for k, v in m.state_dict().items() if not k.endswith(tuple(skip_suffix))}


def test_state_dict_names_and_shapes_equal_the_reference(manifests):
    """Checkpoint compatibility without a GPU: every parameter / buffer name and shape of the product modules equals
    the reference module's (tests/golden/manifests.json was generated from the reference constructors)."""
    from tair_b200.model import ControlLDM
    from tair_b200.model.clip import FrozenOpenCLIPEmbedder
    from tair_b200.model.swinir import SwinIR
    from tair_b200.model.vae import AutoencoderKL
    from tair_b200.testr import TransformerDetector, default_cfg
    u = dict(in_channels=4, out_channels=4, model_channels=64, attention_resolutions=[4, 2, 1], num_res_blocks=2,
             channel_mult=[1, 2, 4, 4], num_head_channels=64, use_spatial_transformer=True,
             use_linear_in_transformer=True, transformer_depth=1, context_dim=128, legacy=False)
    c = dict(u)
    c.pop("out_channels")
    c["hint_channels"] = 4
    m = ControlLDM(u, c)
    assert _shapes(m.unet) == manifests["unet_narrow"]
    assert _shapes(m.controlnet) == manifests["controlnet_narrow"]
    dd = dict(double_z=True, z_channels=4, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=[1, 2, 4, 4],
              num_res_blocks=2, attn_resolutions=[], dropout=0.0)
    assert _shapes(AutoencoderKL(dd, 4)) == manifests["vae"]
    clip = FrozenOpenCLIPEmbedder(1024, None, dict(context_length=77, vocab_size=49408, width=1024, heads=16, layers=24),
                                  layer="penultimate")
    assert _shapes(clip) == manifests["clip_text"]
    sw = SwinIR(img_size=64, patch_size=1, in_chans=3, embed_dim=180, depths=[6] * 8, num_heads=[6] * 8, window_size=8,
                mlp_ratio=2, sf=8, img_range=1.0, upsampler="nearest+conv", resi_connection="1conv", unshuffle=True,
                unshuffle_scale=8)
    assert _shapes(sw, ("relative_position_index",)) == manifests["swinir"]
    det = TransformerDetector(default_cfg("cpu"))
    assert _shapes(det) == manifests["testr"]


def test_checkpoint_loading_surface_of_controlldm():
    """cldm.py:33-90: load_pretrained_sd maps the SD-2.1 prefixes, load_controlnet_from_unet widens the 8-channel input
    conv with zeros, load_controlnet_from_ckpt is strict; Diffusion.to() is a no-op like val_patches.py:240 expects."""
    import torch
    from tair_b200.model import ControlLDM
    from tair_b200.model.gaussian_diffusion import val_diffusion
    u = dict(in_channels=4, out_channels=4, model_channels=32, attention_resolutions=[4, 2, 1], num_res_blocks=1,
             channel_mult=[1, 2], num_head_channels=32, use_spatial_transformer=True, use_linear_in_transformer=True,
             transformer_depth=1, context_dim=64, legacy=False)
    c = dict(u)
    c.pop("out_channels")
    c["hint_channels"] = 4
    m = ControlLDM(u, c)
    g = torch.Generator().manual_seed(0)
    ckpt = {"model.diffusion_model." + k: torch.randn(v.shape, generator=g) for k, v in m.unet.state_dict().items()}
    ckpt["cond_stage_model.unrelated"] = torch.zeros(1)
    some = next(iter(m.unet.state_dict()))
    del ckpt["model.diffusion_model." + some]
    unused, missing = m.load_pretrained_sd(ckpt)
    assert unused == {"cond_stage_model.unrelated"} and missing == {"model.diffusion_model." + some}
    for k, v in m.unet.state_dict().items():
        if k != some:
            assert torch.equal(v, ckpt["model.diffusion_model." + k])
    assert not any(p.requires_grad for p in m.unet.parameters()) and m.unet.train() is m.unet and not m.unet.training
    widened, kept = m.load_controlnet_from_unet()
    assert widened == {"input_blocks.0.0.weight"}
    w = m.controlnet.state_dict()["input_blocks.0.0.weight"]
    assert w.shape[1] == 8 and torch.equal(w[:, :4], m.unet.state_dict()["input_blocks.0.0.weight"]) and (w[:, 4:] == 0).all()
    assert all(k.startswith(("zero_convs", "middle_block_out")) for k in kept)
    sd = {k: torch.randn(v.shape, generator=g) for k, v in m.controlnet.state_dict().items()}
    m.load_controlnet_from_ckpt(sd)
    assert all(torch.equal(v, sd[k]) for k, v in m.controlnet.state_dict().items())
    import pytest
    with pytest.raises(RuntimeError):
        m.load_controlnet_from_ckpt({k: v for k, v in list(sd.items())[1:]})
    d = val_diffusion()
    assert d.to("cpu") is d and len(d.betas) == 1000
    assert m.cast_dtype(torch.float16) is m


def test_sampler_parameterisations_and_graph_key():
    """'eps' selects the recip tables (spaced_sampler.py:133-139,176-179); unknown names raise; the graph key follows
    the step count (tables are re-allocated when it changes)."""
    import pytest
    from tair_b200.model.gaussian_diffusion import val_diffusion
    from tair_b200.sampler import SpacedSampler
    s = SpacedSampler(val_diffusion().betas, "eps", False)
    s.make_schedule(10)
    assert s._tables()[0] is s.sqrt_recip_alphas_cumprod and s._tables()[1] is s.sqrt_recipm1_alphas_cumprod
    k10 = s._graph_key("x")
    s._graphs["dummy"] = object()
    s.make_schedule(10)
    assert s._graph_key("x") == k10 and "dummy" in s._graphs           # same shape: tables updated in place
    s.make_schedule(7)
    assert s._graph_key("x") != k10 and not s._graphs                  # re-allocated: stale graphs dropped
    with pytest.raises(ValueError):
        SpacedSampler(val_diffusion().betas, "x0", False)


def test_make_tiled_fn_matches_reference_semantics():
    """terediff/utils/common.py:125-234: window list (edge-flush last window), gaussian weights (asymmetric midpoints),
    weighted accumulation; an identity fn must be reproduced exactly up to round-off, tile bounds reach fn as kwargs."""
    import numpy as np
    import torch
    from tair_b200 import legacy as L
    assert L.sliding_windows(10, 12, 8, 4) == [(0, 8, 0, 8), (0, 8, 4, 12), (2, 10, 0, 8), (2, 10, 4, 12)]
    assert L.sliding_windows(8, 8, 8, 4) == [(0, 8, 0, 8)]
    w = L.gaussian_weights(4, 4)
    var = 0.01
    wx = [np.exp(-(x - 1.5) ** 2 / 16 / (2 * var)) / np.sqrt(2 * np.pi * var) for x in range(4)]
    wy = [np.exp(-(y - 2.0) ** 2 / 16 / (2 * var)) / np.sqrt(2 * np.pi * var) for y in range(4)]
    assert np.allclose(w, np.outer(wy, wx), rtol=1e-12)
    x = torch.randn(2, 3, 20, 28, generator=torch.Generator().manual_seed(0))
    seen = []

    def fn(t, tag, hi, hi_end, wi, wi_end):
        seen.append((hi, hi_end, wi, wi_end))
        assert tag == "t" and t.shape[-2:] == (8, 8)
        return t * 2
    y = L.make_tiled_fn(fn, 8, 6)(x, "t")
    assert torch.allclose(y, 2 * x, atol=1e-5) and seen == L.sliding_windows(20, 28, 8, 6)
    up = L.make_tiled_fn(lambda t: torch.nn.functional.interpolate(t, scale_factor=2), 8, 8, scale=2, weight="uniform")(x[..., :16, :24])
    assert up.shape == (2, 3, 32, 48)


def test_reference_make_tiled_fn_agrees(golden):
    """Same inputs through the reference's make_tiled_fn: its outputs are stored in tests/golden/tiled_fn.npz
    (make_golden.py tiled)."""
    import torch
    from oracle.tiles import tiled_fn_case
    from tair_b200.legacy import make_tiled_fn
    g = golden("tiled_fn.npz")
    x, fn, cases = tiled_fn_case()
    for size, stride in cases:
        assert torch.equal(make_tiled_fn(fn, size, stride, progress=False)(x), torch.from_numpy(g[f"out_{size}_{stride}"]))


def test_vectorised_decode_matches_scalar_decode():
    import numpy as np
    from tair_b200 import prompt as P
    rng = np.random.default_rng(0)
    recs = rng.integers(0, 97, (500, 25))
    recs[::7, 3] = 96          # early terminator
    recs[5] = rng.integers(0, 95, 25)   # no terminator at all
    recs[6, 0] = 95            # empty string
    assert P.decode_batch(recs) == [P.decode(r) for r in recs]
    assert P.decode_batch(recs.astype(np.uint8)) == [P.decode(r) for r in recs]
    assert P.decode_batch(np.zeros((0, 25), np.uint8)) == []
    scores = rng.random((2, 100)).astype(np.float32)
    polys = (rng.random((2, 100, 32)) * 512).astype(np.float32)
    texts, pg = P.texts_and_polys(scores, polys, recs[:200].reshape(2, 100, 25), 0.5)
    for b in range(2):
        keep = scores[b] >= 0.5
        assert texts[b] == [P.decode(r) for r in recs[:200].reshape(2, 100, 25)[b][keep]]
        assert all(np.array_equal(a, p.reshape(16, 2).astype(np.int32)) for a, p in zip(pg[b], polys[b][keep]))
