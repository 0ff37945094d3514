"""Every tile and split choice of the GEMM / conv / attention dispatchers, bit for bit and element by element.

The GEMM and the implicit-GEMM 3x3 conv run on one of ten kernel instantiations (gemm_tc_kernel<BN> for seven BN,
gemm_tc2_kernel<BN> as a 2-CTA pair for three), picked at run time by the tile autotuner; deep-K convs on the 8x8 level
take a 3-way split-K and splitk_reduce_kernel; the key/value-stationary attention kernel streams a batch-dependent number
of query tiles per CTA.  The tuner promises that all candidates give bit-identical results, and the batch-independence,
graph-replay and world-size tests elsewhere rely on it.  Here every candidate is forced in turn and must
- equal the tuned output bit for bit, and
- lie inside a per-element bound around a float64 reference computed from the same bf16 inputs, epilogue included:

      |out - ref| <= u_out |ref| + d_act * (acc_err + fp32 epilogue roundings) + act_slack

  u_out = 2^-8 for bf16 and 2^-24 for fp32 outputs.  acc_err is the fp32 accumulation error of the MMA chain (see
  acc_err below).  d_act bounds the slope of the activation, act_slack its fp32 evaluation error.

A relative max-abs tolerance over a whole tensor would let a wrong tile whose values are a few times smaller than the
tensor's maximum pass; the per-element bound does not, and test_checker_rejects_broken_tiles proves it on broken
outputs.  Every launch writes into a NaN-filled output, so a tile a candidate fails to store cannot borrow the values an
earlier candidate left in a recycled buffer; the tuned output is taken from a call after the one that tuned, because
tuning runs every candidate into the caller's output.  2-CTA pairs are reached through tests/tile_sweep_worker.py in processes of their own (TAIR_GEMM_2CTA is read
once per process).  Run with -s to see the worst err/bound ratio of each family."""
import math
import os
import re
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if HERE not in sys.path:
    sys.path.insert(0, HERE)
import tile_sweep_worker as tsw  # noqa: E402

pytestmark = pytest.mark.gpu

U_BF16, U_FP32 = 2.0 ** -8, 2.0 ** -24
ACT_SLACK = 4e-6          # fp32 evaluation of the A&S erf (GELU) and of __expf / __fdividef (SiLU), times (1 + |x|)
D_ACT = 1.13              # max slope of GELU (1.129) and SiLU (1.100)
ATTN_P_ROUNDING = 2.0     # c in 2^-8 |ref| + c 2^-8 (P |V|): bf16 rounding of P before the PV MMA


def acc_err(mag, K):
    """Bound on the fp32 accumulation error of sum_k a[m,k] w[n,k] over K, given mag = sum_k |a w|: one fp32 rounding
    (2^-23, truncation allowed) of the running sum per 16-deep MMA step, plus the 16 products of each step aligned with
    at least fp32 precision.  The linear worst case K 2^-22 mag is 32x looser and, at K = 9 x 2560, too loose to notice a
    dropped 64-wide k-block (test_checker_rejects_broken_tiles)."""
    return (math.ceil(K / 16) + 16) * 2.0 ** -23 * mag


WORST: dict = {}


def note(family, ratio):
    WORST[family] = max(WORST.get(family, 0.0), ratio)


@pytest.fixture(scope="module", autouse=True)
def _report_worst_ratios():
    yield
    if WORST:
        print("\nworst |out - ref| / bound: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(WORST.items())))


@pytest.fixture(scope="module")
def ops(cuda_lib):
    from tair_b200 import ops as o
    return o


def check(out, ref, bound, what):
    """Element-wise |out - ref| <= bound (NaN fails); returns the worst |out - ref| / bound."""
    d = (out.double() - ref).abs()
    ok = d <= bound
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{what}: {bad.shape[0]} of {d.numel()} elements outside the float64 bound; first at {i}: "
                             f"out {out[i].item():.6g} ref {ref[i].item():.6g} bound {bound[i].item():.3g}")
    return (d / bound.clamp_min(1e-300)).max().item()


def _rows_of(rg, rpg, M):
    """The row-group add expanded to [M, N] float64 (rows_per_group > 0: row m / rpg; < 0: periodic, row m % -rpg)."""
    m = torch.arange(M, device=rg.device)
    return rg.double()[m // rpg if rpg > 0 else m % (-rpg)]


def _gelu_tanh(x):
    return 0.5 * x * (1 + torch.tanh(math.sqrt(2 / math.pi) * (x + 0.044715 * x ** 3)))


def epilogue_ref(acc, mag, K, *, bias=None, rg=None, res=None, act="none", ln=None, geglu_tile=0, out_fp32=False):
    """float64 epilogue on the float64 accumulator; returns (ref, bound).  Argument order follows the kernels: folded
    LayerNorm, bias and row group before the activation, residual after it."""
    err = acc_err(mag, K)
    if ln is not None:   # acc' = rstd * acc - mean * rstd * colsum, evaluated as fmaf(acc, rstd, (-mean * rstd) * colsum)
        stats, cs = ln
        mean, rstd = stats[:, :1].double(), stats[:, 1:].double()
        shift = mean * rstd * cs.double()[None, :]
        err = rstd * err + 2.0 ** -22 * (rstd * acc.abs() + shift.abs())
        acc = rstd * acc - shift
    pre, addends = acc, 0
    if bias is not None:
        pre = pre + bias.double()
        addends = addends + bias.double().abs()
    if rg is not None:
        pre = pre + rg
        addends = addends + rg.abs()
    if bias is not None or rg is not None:
        err = err + 2.0 ** -23 * (acc.abs() + addends)    # two fp32 additions
    if act == "geglu":   # value / gate halves of each geglu_tile-wide column tile; tanh-form GELU as in gelu_tanh_f
        M, N = pre.shape
        v4, e4 = pre.view(M, N // geglu_tile, 2, geglu_tile // 2), err.view(M, N // geglu_tile, 2, geglu_tile // 2)
        val, gate, ev, eg = (t.reshape(M, N // 2) for t in (v4[:, :, 0], v4[:, :, 1], e4[:, :, 0], e4[:, :, 1]))
        g = _gelu_tanh(gate)
        post = val * g
        # tanh.approx.f32: relative error <= 2^-11 of tanh, i.e. <= 2^-12 |gate| in gelu_tanh
        err = g.abs() * ev + D_ACT * val.abs() * eg + val.abs() * (2.0 ** -11 * gate.abs() + ACT_SLACK) + 2.0 ** -23 * post.abs()
    elif act == "gelu":
        post = 0.5 * pre * (1 + torch.erf(pre / math.sqrt(2)))
        err = D_ACT * err + ACT_SLACK * (1 + pre.abs())
    elif act == "silu":
        post = pre * torch.sigmoid(pre)
        err = D_ACT * err + ACT_SLACK * (1 + pre.abs())
    elif act == "relu":
        post = pre.clamp_min(0)
    else:
        post = pre
    if res is not None:
        post = post + res.double()
        err = err + 2.0 ** -24 * (post.abs() + res.double().abs())
    u = U_FP32 if out_fp32 else U_BF16
    return post, u * post.abs() + (1 + u) * err   # |round(y) - ref| <= u |y| + |y - ref|, |y - ref| <= err


ACT_OF = {"bias_silu": "silu", "bias_gelu": "gelu", "geglu": "geglu"}


def gemm_ref(d, variant):
    A, W = d["a"].double(), d["w"].double()
    M, K = A.shape
    kw = dict(bias=d.get("bias"), res=d.get("res"), act=ACT_OF.get(variant, "none"), ln=d.get("ln"),
              out_fp32=variant == "out_fp32")
    if "rg" in d:
        kw["rg"] = _rows_of(d["rg"], d["rpg"], M)
    if variant == "geglu":
        from tair_b200.model.attention import geglu_tile
        kw["geglu_tile"] = geglu_tile(W.shape[0])
    return epilogue_ref(A @ W.t(), A.abs() @ W.abs().t(), K, **kw)


def conv_acc(x, w, stride, pad):
    """float64 3x3 conv of channels-last x [B,H,W,Cin] with w [Cout, 9*Cin]: (acc, |x| * |w|) as [M, Cout]."""
    Cout, Cin = w.shape[0], x.shape[3]
    xn = x.double().permute(0, 3, 1, 2)
    if pad == 0:
        xn = F.pad(xn, (0, 1, 0, 1))   # the VAE downsampler's asymmetric padding
    wn = w.double().view(Cout, 3, 3, Cin).permute(0, 3, 1, 2)
    p = 1 if pad == 1 else 0
    acc = F.conv2d(xn, wn, stride=stride, padding=p).permute(0, 2, 3, 1).reshape(-1, Cout)
    mag = F.conv2d(xn.abs(), wn.abs(), stride=stride, padding=p).permute(0, 2, 3, 1).reshape(-1, Cout)
    return acc, mag


def conv_ref(d, acc, mag, act="none", out_fp32=False):
    K = d["w"].shape[1]
    M = acc.shape[0]
    rg = _rows_of(d["rg"], d["rpg"], M) if "rg" in d else None
    res = d["res"].reshape(M, -1) if "res" in d else None
    return epilogue_ref(acc, mag, K, bias=d.get("bias"), rg=rg, res=res, act=act, out_fp32=out_fp32)


def rn(*shape, scale=1.0, seed=0):
    return tsw.rn(*shape, scale=scale, seed=seed)


def fresh(*shape, dtype=torch.bfloat16):
    """NaN-filled output: every comparison below sees only what this one launch stored (see tsw.fresh)."""
    return tsw.fresh(shape, dtype)


# ---------------------------------------------------------------------------------------------------------------------
# 1. the checker rejects broken tiles


def test_checker_rejects_broken_tiles(ops):
    """A verified output passes; the same output with (a) two 32-column groups swapped inside one N tile of one 128-row
    block, or (b) one 64-wide k-block missing from one 128-row tile, is rejected - also at K = 9 x 2560 (split-K conv)."""
    M, N, K = 512, 320, 640
    a, w = rn(M, K, seed=1).bfloat16(), rn(N, K, scale=K ** -0.5, seed=2).bfloat16()
    ops.gemm(a, w)   # tunes
    out = ops.gemm(a, w, out=fresh(M, N))
    A, W = a.double(), w.double()
    ref, bound = epilogue_ref(A @ W.t(), A.abs() @ W.abs().t(), K)
    check(out, ref, bound, "verified GEMM")
    swapped = out.clone()
    swapped[128:256, 32:64], swapped[128:256, 64:96] = out[128:256, 64:96], out[128:256, 32:64]
    with pytest.raises(AssertionError):
        check(swapped, ref, bound, "(a) swapped column groups")
    dropped = (out.double() - torch.nn.functional.pad(A[128:256, 64:128] @ W[:128, 64:128].t(), (0, N - 128, 128, M - 256)))
    with pytest.raises(AssertionError):
        check(dropped.bfloat16(), ref, bound, "(b) dropped k-block")
    # deep K: 8x8 2560 -> 1280 at B=2 (split-K); drop channels [640, 704) of the centre tap from the first 128 rows
    B, H, Cin, Cout = 2, 8, 2560, 1280
    x, wc = rn(B, H, H, Cin, seed=3).bfloat16(), rn(Cout, 9 * Cin, scale=(9 * Cin) ** -0.5, seed=4).bfloat16()
    outc = ops.conv3x3(x, wc, out=fresh(B, H, H, Cout)).view(-1, Cout)
    acc, mag = conv_acc(x, wc, 1, 1)
    ref, bound = epilogue_ref(acc, mag, 9 * Cin)
    check(outc, ref, bound, "verified split-K conv")
    c0 = 4 * Cin + 640
    part = x.double().view(-1, Cin)[:128, 640:704] @ wc.double()[:, c0:c0 + 64].t()
    with pytest.raises(AssertionError):
        check((outc.double() - F.pad(part, (0, 0, 0, outc.shape[0] - 128))).bfloat16(), ref, bound, "deep dropped k-block")


# ---------------------------------------------------------------------------------------------------------------------
# 2. GEMM candidate sweep (1-CTA in this process; 2-CTA pairs in test_two_cta_sweep_digests)

GEMM_CASES = [(n, v) for n in tsw.GEMMS for v in tsw.gemm_variants(n)]


@pytest.mark.parametrize("name,variant", GEMM_CASES, ids=[f"{n}-{v}" for n, v in GEMM_CASES])
def test_gemm_every_tile(ops, name, variant):
    from tair_b200._lib import TairError
    d = tsw.inputs("gemm", name, variant)
    tuned = tsw.run(ops, "gemm", name, variant, d).clone()
    ref, bound = gemm_ref(d, variant)
    note("gemm fp32 out" if variant == "out_fp32" else "gemm", check(tuned, ref, bound, f"{name} {variant} tuned"))
    legal = tsw.legal_bns("gemm", name, variant)
    for bn in tsw.BNS:
        if bn not in legal:   # GEGLU at a BN the weight is not interleaved for: refused, not silently wrong
            with pytest.raises(TairError):
                tsw.run(ops, "gemm", name, variant, d, bn)
            continue
        out = tsw.run(ops, "gemm", name, variant, d, bn)
        assert torch.equal(out, tuned), f"{name} {variant}: BN={bn} is not bit-identical to the tuned tile"
        if variant == "out_slice":   # the columns around the slice keep their NaN
            N = d["w"].shape[0]
            assert d["out_buf"][:, 0].isnan().all() and d["out_buf"][:, N + 1:].isnan().all(), f"BN={bn}"


# ---------------------------------------------------------------------------------------------------------------------
# 3. conv candidate sweep

CONV_CASES = [(n, v) for n in tsw.CONVS for v in tsw.CONV_VARIANTS]
_conv_acc_cache: dict = {}


def _conv_acc_for(name, d):
    if name not in _conv_acc_cache:   # the accumulator does not depend on the epilogue variant
        _conv_acc_cache.clear()
        B, H, Cin, Cout, stride, pad = tsw.CONVS[name]
        _conv_acc_cache[name] = conv_acc(d["x"], d["w"], stride, pad)
    return _conv_acc_cache[name]


@pytest.mark.parametrize("name,variant", CONV_CASES, ids=[f"{n}-{v}" for n, v in CONV_CASES])
def test_conv_every_tile(ops, name, variant):
    d = tsw.inputs("conv", name, variant)
    acc, mag = _conv_acc_for(name, d)
    ref, bound = conv_ref(d, acc, mag, act=ACT_OF.get(variant, "none"))
    default = tsw.run(ops, "conv", name, variant, d).clone()
    Cout = d["w"].shape[0]
    fam = "splitk_conv" if tsw.splitk_conv(name) else "conv"
    note(fam, check(default.view(-1, Cout), ref, bound, f"conv {name} {variant} default"))
    first = None
    for bn in tsw.BNS:
        out = tsw.run(ops, "conv", name, variant, d, bn)
        if tsw.splitk_conv(name):   # the default is the split-K sum: the single-pass tiles agree among themselves
            if first is None:
                first = out.clone()
                note("conv", check(first.view(-1, Cout), ref, bound, f"conv {name} {variant} BN={bn}"))
            assert torch.equal(out, first), f"conv {name} {variant}: BN={bn} differs from BN={tsw.BNS[0]}"
        else:
            assert torch.equal(out, default), f"conv {name} {variant}: BN={bn} is not bit-identical to the tuned tile"


# ---------------------------------------------------------------------------------------------------------------------
# 2-CTA pairs: the worker process under TAIR_GEMM_2CTA=0 and =2


def _worker_digests(mode):
    env = dict(os.environ)
    env.pop("TAIR_GEMM_BN", None)
    env["TAIR_GEMM_2CTA"] = str(mode)
    res = subprocess.run([sys.executable, os.path.join(HERE, "tile_sweep_worker.py")], capture_output=True, text=True,
                         timeout=900, env=env, cwd=ROOT)
    assert res.returncode == 0 and "WORKER OK" in res.stdout, \
        f"TAIR_GEMM_2CTA={mode} worker failed:\n{res.stdout[-2000:]}\n{res.stderr[-4000:]}"
    out = {}
    for tag, bn, h in re.findall(r"^DIGEST (\S+) (\S+) ([0-9a-f]{64})$", res.stdout, re.M):
        out.setdefault(tag, {})[f"{bn}/2cta={mode}"] = h
    return out


def test_two_cta_sweep_digests(ops):
    """Every case of the sweep gives one digest across all BN, the tuned tile, both TAIR_GEMM_2CTA modes and this
    process's own tuned output."""
    runs = [_worker_digests(0), _worker_digests(2)]
    cases = tsw.worker_cases()
    for kind, name, variant in cases:
        tag = f"{kind}:{name}:{variant}"
        d = tsw.inputs(kind, name, variant)
        split = kind == "conv" and tsw.splitk_conv(name)
        mine = tsw.digest(tsw.run(ops, kind, name, variant, d, tsw.BNS[0] if split else None))
        seen = {**runs[0].get(tag, {}), **runs[1].get(tag, {})}
        assert len(seen) == 2 * (len(tsw.legal_bns(kind, name, variant)) + (0 if split else 1)), (tag, sorted(seen))
        assert set(seen.values()) == {mine}, f"{tag}: digests differ across BN / CTA mode: {seen} (this process: {mine})"


# ---------------------------------------------------------------------------------------------------------------------
# 4. split-K conv (Ho * Wo <= 64 and 9 * Cin / 64 >= 64: ops.conv3x3 lends the workspace)

SPLITK_LAYERS = {"8x8_1280": (16, 8, 1280, 1280, 1), "8x8_2560_1280": (16, 8, 2560, 1280, 1),
                 "16to8_s2_1280": (16, 16, 1280, 1280, 2),
                 "8x8_1280_b32": (32, 8, 1280, 1280, 1)}   # CFG-stacked batch: 16 x 5 tiles x 3 splits > 148 SMs
SPLITK_EPILOGUES = ("bias", "rg_per_image", "rg_periodic", "residual", "gelu", "silu", "relu", "out_fp32")


def _splitk_inputs(layer):
    B, H, Cin, Cout, stride = SPLITK_LAYERS[layer]
    s = 9000 + 100 * list(SPLITK_LAYERS).index(layer)
    return (rn(B, H, H, Cin, seed=s).bfloat16(), rn(Cout, 9 * Cin, scale=(9 * Cin) ** -0.5, seed=s + 1).bfloat16(),
            rn(Cout, scale=0.5, seed=s + 2))


@pytest.mark.parametrize("layer", list(SPLITK_LAYERS))
def test_splitk_conv_epilogues_and_single_pass(ops, layer):
    B, H, Cin, Cout, stride = SPLITK_LAYERS[layer]
    x, w, bias = _splitk_inputs(layer)
    Ho = H // stride
    M = B * Ho * Ho
    acc, mag = conv_acc(x, w, stride, 1)
    for epi in SPLITK_EPILOGUES:
        kw, d = dict(stride=stride, bias=bias), dict(w=w, bias=bias)
        if epi == "rg_per_image":
            d["rg"], d["rpg"] = rn(B, Cout, seed=1), Ho * Ho
        elif epi == "rg_periodic":
            d["rg"], d["rpg"] = rn(Ho * Ho, Cout, seed=2), -Ho * Ho
        elif epi == "residual":
            d["res"] = rn(B, Ho, Ho, Cout, seed=3).bfloat16()
            kw["residual"] = d["res"]
        if "rg" in d:
            kw.update(rowgroup=d["rg"], rows_per_group=d["rpg"])
        act = epi if epi in ("gelu", "silu", "relu") else "none"
        if act != "none":
            kw["act"] = {"gelu": ops.ACT_GELU, "silu": ops.ACT_SILU, "relu": ops.ACT_RELU}[act]
        kw["out"] = fresh(B, Ho, Ho, Cout, dtype=torch.float32 if epi == "out_fp32" else torch.bfloat16)
        out = ops.conv3x3(x, w, **kw).view(M, Cout)
        ref, bound = conv_ref(d, acc, mag, act=act, out_fp32=epi == "out_fp32")
        note("splitk_conv fp32 out" if epi == "out_fp32" else "splitk_conv", check(out, ref, bound, f"split-K {layer} {epi}"))
    # split against single pass, fp32 output: each within `bound` of the float64 result, so within 2 x bound of each other
    ref, bound = conv_ref(dict(w=w, bias=bias), acc, mag, out_fp32=True)
    split = ops.conv3x3(x, w, stride=stride, bias=bias, out=fresh(B, Ho, Ho, Cout, dtype=torch.float32)).view(M, Cout)
    with tsw.forced_bn(256):
        single = ops.conv3x3(x, w, stride=stride, bias=bias, out=fresh(B, Ho, Ho, Cout, dtype=torch.float32)).view(M, Cout)
    note("conv fp32 out", check(single, ref, bound, f"single pass {layer}"))
    note("splitk_conv vs single pass", check(split, single.double(), 2 * bound, f"split-K vs single pass {layer}"))


def test_splitk_conv_batch_independent(ops):
    """8x8 1280 -> 1280 with bias + per-image fp32 rows + residual: B = 1, 16 and 32 give the same bits per image (the split
    depends on the layer geometry, never on the batch)."""
    Cin = Cout = 1280
    x = rn(32, 8, 8, Cin, seed=11).bfloat16()
    w = rn(Cout, 9 * Cin, scale=(9 * Cin) ** -0.5, seed=12).bfloat16()
    bias, rg, res = rn(Cout, seed=13), rn(32, Cout, seed=14), rn(32, 8, 8, Cout, seed=15).bfloat16()

    def conv(lo, hi):
        return ops.conv3x3(x[lo:hi].contiguous(), w, bias=bias, rowgroup=rg[lo:hi].contiguous(), rows_per_group=64,
                           residual=res[lo:hi].contiguous(), out=fresh(hi - lo, 8, 8, Cout))
    o32 = conv(0, 32)
    assert torch.equal(conv(0, 16), o32[:16])
    assert torch.equal(conv(16, 32), o32[16:])
    for i in (0, 9, 31):
        assert torch.equal(conv(i, i + 1)[0], o32[i]), i


def test_bf16_rowgroup_refused_on_splitk_layers(ops):
    """bf16 row groups exist only in the row-add epilogue of the single-pass kernels: a split-K layer refuses them with a
    TairError, while the same call on a 16x16 layer succeeds and is right."""
    from tair_b200._lib import TairError
    Cin = Cout = 1280
    w = rn(Cout, 9 * Cin, scale=(9 * Cin) ** -0.5, seed=21).bfloat16()
    rg = rn(2, Cout, seed=22).bfloat16()
    with pytest.raises(TairError):
        ops.conv3x3(rn(2, 8, 8, Cin, seed=23).bfloat16(), w, rowgroup=rg, rows_per_group=64)
    x = rn(2, 16, 16, Cin, seed=24).bfloat16()
    ops.conv3x3(x, w, rowgroup=rg, rows_per_group=256)   # tunes
    out = ops.conv3x3(x, w, rowgroup=rg, rows_per_group=256, out=fresh(2, 16, 16, Cout)).view(-1, Cout)
    acc, mag = conv_acc(x, w, 1, 1)
    ref, bound = conv_ref(dict(w=w, rg=rg, rpg=256), acc, mag)
    note("conv", check(out, ref, bound, "16x16 bf16 row group"))


# ---------------------------------------------------------------------------------------------------------------------
# 5. capture path: the uncached closed-form tile against the tuned one


def test_capture_closed_form_tile_matches_tuned(ops):
    M, N, K = 1237, 640, 320     # an M no other test uses: the tune cache cannot hold this shape yet
    a, w, bias = rn(M, K, seed=31).bfloat16(), rn(N, K, scale=K ** -0.5, seed=32).bfloat16(), rn(N, seed=33)
    ops.gemm(a[:128], w)   # library loaded and initialised outside the capture
    out = fresh(M, N)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.gemm(a, w, bias=bias, out=out)
    g.replay()
    torch.cuda.synchronize()
    ops.gemm(a, w, bias=bias)   # first eager call: tunes and caches (every candidate writes its output)
    eager = ops.gemm(a, w, bias=bias, out=fresh(M, N))   # one launch of the cached choice
    assert torch.equal(out, eager)
    A, W = a.double(), w.double()
    ref, bound = epilogue_ref(A @ W.t(), A.abs() @ W.abs().t(), K, bias=bias)
    note("gemm", check(out, ref, bound, "captured GEMM"))


# ---------------------------------------------------------------------------------------------------------------------
# 6. key/value-stationary attention: query tiles per CTA


@pytest.mark.parametrize("B,H,Lq,Lk", [(2, 5, 4096, 77), (16, 10, 1024, 77), (3, 20, 200, 50), (2, 3, 128, 1)])
def test_kvs_attention_every_chunking(ops, monkeypatch, B, H, Lq, Lk):
    """TAIR_KVS_CHUNKS = 1, 2, 3 and q_tiles (values above q_tiles are ignored, leaving the default) and the default give
    the same bits, inside 2^-8 |ref| + c 2^-8 (P |V|) of float64 softmax attention."""
    C = H * 64
    q = rn(B * Lq, C, scale=1.5, seed=41).bfloat16()
    k, v = rn(B * Lk, C, scale=1.5, seed=42).bfloat16(), rn(B * Lk, C, seed=43).bfloat16()
    monkeypatch.delenv("TAIR_KVS_CHUNKS", raising=False)
    default = ops.attention(q, k, v, B=B, H=H, Lq=Lq, Lk=Lk, out=fresh(B * Lq, C))
    q_tiles = (Lq + 127) // 128
    for chunks in sorted({1, 2, 3, q_tiles}):
        monkeypatch.setenv("TAIR_KVS_CHUNKS", str(chunks))
        out = ops.attention(q, k, v, B=B, H=H, Lq=Lq, Lk=Lk, out=fresh(B * Lq, C))
        assert torch.equal(out, default), f"chunks={chunks}"
    monkeypatch.delenv("TAIR_KVS_CHUNKS")

    def heads(t, L):
        return t.double().view(B, L, H, 64).transpose(1, 2)
    P = torch.softmax(heads(q, Lq) @ heads(k, Lk).transpose(-1, -2) / 8.0, dim=-1)
    Vh = heads(v, Lk)
    ref = (P @ Vh).transpose(1, 2).reshape(B * Lq, C)
    pv = (P @ Vh.abs()).transpose(1, 2).reshape(B * Lq, C)
    note("attention", check(default, ref, U_BF16 * ref.abs() + ATTN_P_ROUNDING * U_BF16 * pv, f"attention {B, H, Lq, Lk}"))
