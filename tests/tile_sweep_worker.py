"""Tile sweep of the GEMM and the implicit-GEMM 3x3 conv (csrc/gemm_tc.cu), shared by tests/test_gemm_tiles_gpu.py and
run by it as a worker process of its own.

The case table, the seeded inputs and ``run()`` live here so that both processes compute exactly the same thing.  As a
script (``python tests/tile_sweep_worker.py``) it runs every 2-CTA-relevant case at the tuned tile and at every forced
``TAIR_GEMM_BN``, checks that all of them are bit-identical, and prints one ``DIGEST <case> <bn> <sha256>`` line per
(case, BN).  It is a separate process because ``TAIR_GEMM_2CTA`` is read once per process: the parent runs it under
``TAIR_GEMM_2CTA=0`` (no 2-CTA pair anywhere) and ``=2`` (every legal BN - 128, 160, 256 - as a 2-CTA pair)."""
import contextlib
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BNS = (64, 96, 128, 160, 192, 224, 256)

# GEMM shapes (name, M, N, K) from the project's call sites.  Which edge of the tile space each one reaches:
GEMMS = {
    # CLIP text encoder q|k|v, one prompt of 77 tokens: M < 128, a single M tile; under 2-CTA the peer CTA's tile lies
    # wholly outside M
    "clip_qkv": (77, 2304, 768),
    # TESTR decoder, B=16 x 100 queries: tiles_m = 13 (odd, >= 3) with a ragged last tile; num_kb = 4 < 8
    "testr_dec": (1600, 256, 256),
    # UNet 64x64 level at B=16: more than 3 x 148 tiles for every BN, so every persistent CTA / pair drains at least
    # three tiles and the double-buffered TMEM accumulator wraps its phase; N = 320 is ragged for 96/128/192/224/256
    "unet64": (65536, 320, 320),
    # UNet 16x16 level at B=16: N = 1280 ragged for 96/192/224, exact for the rest; num_kb = 20 >= 16, the use_2cta threshold
    "unet16": (4096, 1280, 1280),
    # SwinIR MLP fc2 (hidden 360): K not a multiple of 64 (TMA zero fill of the K tail), num_kb = 6 < 8
    "swinir_fc2": (4096, 192, 360),
    # K tail at num_kb = 16 (no single call site has both): the deep-K loop with a zero-filled last k-block
    "k_tail_deep": (1000, 640, 1000),
    # TESTR control-point head (256 -> 2): N % 32 != 0 and a 4-byte output row, the generic thread-per-row epilogue
    "testr_coord": (1600, 2, 256),
    # N = 72 keeps a 16-byte output row but N % 32 != 0: the generic TMA-store epilogue's column tail; M = 300, K = 200
    "ragged_72": (300, 72, 200),
    # transformer feed-forward GEGLU of the 64x64 level (8 x 320 interleaved rows): BN = 256 is the only legal tile
    "geglu_ff": (4096, 2560, 320),
    # GEGLU with N % 256 != 0: BN = 128 is the only legal tile
    "geglu_384": (1000, 384, 192),
}

# Epilogue variants of the GEMM sweep
GEMM_VARIANTS = ("plain", "bias_silu", "bias_gelu", "bias_res", "rg16_periodic", "rg32_slice", "out_fp32", "out_slice", "ln")
# ... of which these can run as a 2-CTA pair (bf16 output with 16-byte aligned rows); the others are 1-CTA only
TWO_CTA_VARIANTS = ("plain", "bias_silu", "bias_gelu", "bias_res", "rg16_periodic", "rg32_slice", "ln", "geglu")

# 3x3 convs (name, B, H, Cin, Cout, stride, pad), H = W
CONVS = {
    "unet64": (16, 64, 320, 320, 1, 1),           # UNet levels at B=16
    "unet32": (16, 32, 640, 640, 1, 1),
    "unet16": (16, 16, 1280, 1280, 1, 1),
    "unet_down8": (16, 16, 1280, 1280, 2, 1),     # stride 2 into 8x8: the default takes the 3-way split-K path
    "vae_down": (1, 256, 256, 256, 2, 0),         # VAE encoder downsampler: pad = 0, i.e. F.pad(x, (0, 1, 0, 1))
    "conv_out": (16, 64, 320, 4, 1, 1),           # UNet conv_out: Cout = 4
    "swinir_body": (1, 64, 192, 192, 1, 1),       # SwinIR conv_after_body on the 192-wide padded trunk
    "odd_b5_4x4": (5, 4, 320, 320, 1, 1),         # one M tile spans all 5 images and extends past the batch
    "odd_b3_8x8": (3, 8, 256, 320, 1, 1),         # 2 M tiles, the second half past the batch
}
CONV_VARIANTS = ("bias", "bias_rg_res", "bias_silu")


def gemm_variants(name):
    """Legal epilogue variants of one GEMM case."""
    M, N, K = GEMMS[name]
    if name.startswith("geglu"):
        return ("geglu",)
    v = [x for x in GEMM_VARIANTS if not (x == "rg16_periodic" and N % 32 != 0)]   # bf16 rows need the row-add epilogue
    if N % 4 != 0:
        v.remove("ln")   # folded LayerNorm needs N % 4 == 0
    return tuple(v)


def splitk_conv(name):
    B, H, Cin, Cout, stride, pad = CONVS[name]
    Ho = (H + pad - 2) // stride + 1
    # ops.conv3x3 lends the workspace (Cin >= 448) and tair_conv3x3_bf16 uses it (num_kb >= 64, Cout % 4 == 0)
    return Ho * Ho <= 64 and Cin >= 448 and 9 * (Cin // 64) >= 64 and Cout % 4 == 0


def rn(*shape, scale=1.0, seed=0):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(*shape, device="cuda", generator=g) * scale


def fresh(shape, dtype):
    """An output buffer full of NaN: a tile the kernel does not store stays NaN and fails every comparison."""
    import torch
    return torch.full(shape, float("nan"), device="cuda", dtype=dtype)


@contextlib.contextmanager
def forced_bn(bn):
    """Force the N tile (TAIR_GEMM_BN is read on every call, before the tune cache); None leaves the tuner in charge."""
    old = os.environ.pop("TAIR_GEMM_BN", None)
    if bn is not None:
        os.environ["TAIR_GEMM_BN"] = str(bn)
    try:
        yield
    finally:
        os.environ.pop("TAIR_GEMM_BN", None)
        if old is not None:
            os.environ["TAIR_GEMM_BN"] = old


def gemm_inputs(name, variant):
    """Seeded inputs of one GEMM case: a dict of the operands and the epilogue tensors the variant uses."""
    import torch
    M, N, K = GEMMS[name]
    s = 1000 * (list(GEMMS).index(name) + 1)
    d = dict(a=rn(M, K, seed=s).bfloat16(), w=rn(N, K, scale=K ** -0.5, seed=s + 1).bfloat16())
    n_out = N // 2 if variant == "geglu" else N
    if variant != "plain":
        d["bias"] = rn(N, scale=0.5, seed=s + 2)
    if variant in ("bias_res", "geglu"):
        d["res"] = rn(M, n_out, seed=s + 3).bfloat16()
    if variant == "rg16_periodic":
        d["rg"], d["rpg"] = rn(100, N, seed=s + 4).bfloat16(), -100
    if variant == "rg32_slice":   # a column slice of a wider buffer: 4-byte offset, ldg % 4 != 0 (vec_rg == false)
        R = 64
        d["rg"], d["rpg"] = rn((M + R - 1) // R, N + 5, seed=s + 5)[:, 1:N + 1], R
    if variant == "ln":           # raw rows far from zero mean, as a LayerNorm input
        from tair_b200 import ops
        d["a"] = (rn(M, K, scale=1.5, seed=s) + 3.0 * rn(M, 1, seed=s + 6)).bfloat16()
        d["ln"] = (ops.row_stats(d["a"]), d["w"].float().sum(1).contiguous())
    if variant == "out_slice":    # bf16 output as a column slice with ldc % 8 != 0 (vec_out == false)
        d["out_buf"] = torch.empty(M, N + 3, device="cuda", dtype=torch.bfloat16)   # refilled with NaN by every run
    return d


def run_gemm(ops, d, variant):
    import torch
    M, N = d["a"].shape[0], d["w"].shape[0]
    kw = dict(bias=d.get("bias"), residual=d.get("res"))
    if "rg" in d:
        kw.update(rowgroup=d["rg"], rows_per_group=d["rpg"])
    if variant == "out_slice":
        d["out_buf"].fill_(float("nan"))
        kw["out"] = d["out_buf"][:, 1:N + 1]
    else:
        kw["out"] = fresh((M, N // 2 if variant == "geglu" else N), torch.float32 if variant == "out_fp32" else torch.bfloat16)
    if variant == "bias_silu":
        kw["act"] = ops.ACT_SILU
    elif variant == "bias_gelu":
        kw["act"] = ops.ACT_GELU
    elif variant == "geglu":
        kw["act"] = ops.ACT_GEGLU
    elif variant == "ln":
        kw["ln"] = d["ln"]
    return ops.gemm(d["a"], d["w"], **kw)


def conv_inputs(name, variant):
    B, H, Cin, Cout, stride, pad = CONVS[name]
    Ho = (H + pad - 2) // stride + 1
    s = 5000 + 1000 * list(CONVS).index(name)
    d = dict(x=rn(B, H, H, Cin, seed=s).bfloat16(), w=rn(Cout, 9 * Cin, scale=(9 * Cin) ** -0.5, seed=s + 1).bfloat16(),
             bias=rn(Cout, scale=0.5, seed=s + 2))
    if variant == "bias_rg_res":   # per-image fp32 rows as an unaligned column slice (_Step.emb_for), plus a residual
        d["rg"], d["rpg"] = rn(B, Cout + 5, seed=s + 3)[:, 1:Cout + 1], Ho * Ho
        d["res"] = rn(B, Ho, Ho, Cout, seed=s + 4).bfloat16()
    return d


def run_conv(ops, name, d, variant):
    import torch
    B, H, Cin, Cout, stride, pad = CONVS[name]
    Ho = (H + pad - 2) // stride + 1
    kw = dict(stride=stride, pad=pad, bias=d["bias"], residual=d.get("res"), out=fresh((B, Ho, Ho, Cout), torch.bfloat16))
    if "rg" in d:
        kw.update(rowgroup=d["rg"], rows_per_group=d["rpg"])
    if variant == "bias_silu":
        kw["act"] = ops.ACT_SILU
    return ops.conv3x3(d["x"], d["w"], **kw)


def run(ops, kind, name, variant, d, bn=None):
    """One launch of the case into a NaN-filled output (forced tile, or the tuned one when bn is None)."""
    def once():
        return run_gemm(ops, d, variant) if kind == "gemm" else run_conv(ops, name, d, variant)
    with forced_bn(bn):
        if bn is None:
            once()   # the first call of a shape tunes, running every candidate into its output: keep a later call's only
        return once()


def inputs(kind, name, variant):
    return gemm_inputs(name, variant) if kind == "gemm" else conv_inputs(name, variant)


def legal_bns(kind, name, variant):
    """The forced BNs a case accepts: every BN, except that a GEGLU weight is interleaved for exactly one."""
    if variant == "geglu":
        from tair_b200.model.attention import geglu_tile
        return (geglu_tile(GEMMS[name][1]),)
    return BNS


def digest(t) -> str:
    import torch
    t = t.contiguous()
    return hashlib.sha256(t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).cpu().numpy().tobytes()).hexdigest()


def worker_cases():
    """(kind, name, variant) of the 2-CTA sweep."""
    out = [("gemm", n, v) for n in GEMMS for v in gemm_variants(n) if v in TWO_CTA_VARIANTS]
    out += [("conv", n, v) for n in CONVS for v in CONV_VARIANTS]
    return out


def main():
    import torch
    from tair_b200 import ops
    torch.backends.cuda.matmul.allow_tf32 = False
    for kind, name, variant in worker_cases():
        d = inputs(kind, name, variant)
        tag = f"{kind}:{name}:{variant}"
        ref = None
        if not (kind == "conv" and splitk_conv(name)):   # the split-K default sums in another order: not compared
            ref = run(ops, kind, name, variant, d).clone()
            print(f"DIGEST {tag} tuned {digest(ref)}", flush=True)
        for bn in legal_bns(kind, name, variant):
            out = run(ops, kind, name, variant, d, bn)
            if ref is None:
                ref = out.clone()
            assert torch.equal(out, ref), f"{tag}: BN={bn} differs from the first output of this process"
            print(f"DIGEST {tag} {bn} {digest(out)}", flush=True)
        del d, ref
    torch.cuda.synchronize()
    print("WORKER OK", flush=True)


if __name__ == "__main__":
    main()
