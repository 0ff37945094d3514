"""Thin torch-tensor front end over the C ABI (``include/tair_b200.h``).

torch supplies device memory and the current stream; all arithmetic happens in
the sm_100a kernels of ``libtair_b200.so``.  Every function raises if handed a
CPU tensor — there is deliberately no fallback path.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import ACT_GEGLU, ACT_GELU, ACT_NONE, ACT_RELU, ACT_SILU, Epilogue, TairError  # noqa: F401

BF16 = torch.bfloat16


class KernelTimer:
    """Optional per-family CUDA-event timing of the launches issued through this module (used by bench.py to
    measure the dominant kernel live, on the launching stream).  Off by default: zero overhead on the hot path."""

    def __init__(self):
        self.records = {}   # family -> list of (start_event, end_event, work)
        self.shapes = {}    # family -> list of shape tags, parallel to records

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for fam, recs in self.records.items():
            ms = sum(a.elapsed_time(b) for a, b, _ in recs)
            out[fam] = dict(launches=len(recs), ms=ms, work=sum(w for _, _, w in recs))
        return out

    def by_shape(self):
        """(family, shape tag) -> launches / ms / work, for tools/shape_breakdown.py."""
        torch.cuda.synchronize()
        out = {}
        for fam, recs in self.records.items():
            for (a, b, w), tag in zip(recs, self.shapes[fam]):
                d = out.setdefault((fam, tag), dict(launches=0, ms=0.0, work=0.0))
                d["launches"] += 1
                d["ms"] += a.elapsed_time(b)
                d["work"] += w
        return out


_timer: Optional[KernelTimer] = None


def set_timer(t: Optional[KernelTimer]) -> None:
    global _timer
    _timer = t


class _timed:
    __slots__ = ("fam", "work", "a", "tag")

    def __init__(self, fam: str, work: float, tag=None):
        self.fam, self.work, self.tag = fam, work, tag

    def __enter__(self):
        if _timer is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if _timer is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            _timer.records.setdefault(self.fam, []).append((self.a, b, self.work))
            _timer.shapes.setdefault(self.fam, []).append(self.tag)
        return False


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _cuda(t: torch.Tensor, name: str, dtype=None) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TairError(f"{name}: expected a CUDA tensor (tair_b200 has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise TairError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    return t


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _rows(t: torch.Tensor, name: str) -> tuple[torch.Tensor, int]:
    """2-D view with unit inner stride; returns (tensor, row stride in elements)."""
    if t.dim() != 2 or t.stride(1) != 1:
        raise TairError(f"{name}: expected a 2-D tensor with contiguous rows, got {tuple(t.shape)} / {t.stride()}")
    return t, t.stride(0)


def _make_epilogue(out, M, n_out, bias, residual, rowgroup, rows_per_group, act) -> Epilogue:
    e = Epilogue()
    _cuda(out, "out")
    if out.dtype not in (BF16, torch.float32):
        raise TairError("out must be bf16 or fp32")
    o2, ldc = _rows(out, "out")
    if o2.shape[0] != M or o2.shape[1] != n_out:
        raise TairError(f"out has shape {tuple(o2.shape)}, expected {(M, n_out)}")
    e.out, e.ldc = o2.data_ptr(), ldc
    e.out_fp32 = 1 if out.dtype == torch.float32 else 0
    e.act = act
    if bias is not None:
        _cuda(bias, "bias", torch.float32)
        if not bias.is_contiguous():
            raise TairError("bias must be contiguous")
        e.bias = bias.data_ptr()
    if residual is not None:
        _cuda(residual, "residual", BF16)
        r2, ldr = _rows(residual, "residual")
        if tuple(r2.shape) != (M, n_out):
            raise TairError(f"residual has shape {tuple(r2.shape)}, expected {(M, n_out)}")
        e.residual, e.ldr = r2.data_ptr(), ldr
    if rowgroup is not None:
        _cuda(rowgroup, "rowgroup")
        if rowgroup.dtype not in (BF16, torch.float32):
            raise TairError("rowgroup must be fp32 or bf16")
        g2, ldg = _rows(rowgroup, "rowgroup")
        covered = g2.shape[0] * rows_per_group >= M if rows_per_group > 0 else (rows_per_group < 0 and g2.shape[0] >= -rows_per_group)
        if not covered or g2.shape[1] < n_out:
            raise TairError("rowgroup shape does not cover the output")
        e.rowgroup, e.ldg, e.rows_per_group = g2.data_ptr(), ldg, rows_per_group
        e.rowgroup_bf16 = 1 if rowgroup.dtype == BF16 else 0   # bf16 rows: prefetched row-add epilogue (see the header)
    return e


def gemm(a: torch.Tensor, w: torch.Tensor, *, bias=None, residual=None, rowgroup=None, rows_per_group=0,
         act: int = ACT_NONE, out: Optional[torch.Tensor] = None, out_dtype=BF16, ln=None) -> torch.Tensor:
    """``epilogue(a @ w.T)``; a [M,K] bf16, w [N,K] bf16 (nn.Linear layout).
    ``ln = (row_stats [M,2] fp32, col_sum [N] fp32)``: LayerNorm folded in (see tair_epilogue.ln_row_stats)."""
    _cuda(a, "a", BF16), _cuda(w, "w", BF16)
    a2, lda = _rows(a, "a")
    w2, ldw = _rows(w, "w")
    M, K = a2.shape
    N = w2.shape[0]
    if w2.shape[1] != K:
        raise TairError(f"gemm: K mismatch {K} vs {w2.shape[1]}")
    n_out = N // 2 if act == ACT_GEGLU else N
    if out is None:
        out = torch.empty((M, n_out), device=a.device, dtype=out_dtype)
    e = _make_epilogue(out, M, n_out, bias, residual, rowgroup, rows_per_group, act)
    if ln is not None:
        rs, cs = ln
        _cuda(rs, "ln row_stats", torch.float32), _cuda(cs, "ln col_sum", torch.float32)
        if tuple(rs.shape) != (M, 2) or cs.numel() != N or not (rs.is_contiguous() and cs.is_contiguous()):
            raise TairError("gemm: ln = (row_stats [M,2], col_sum [N]) contiguous fp32 expected")
        e.ln_row_stats, e.ln_col_sum = rs.data_ptr(), cs.data_ptr()
    with _timed("gemm", 2.0 * M * N * K, (M, N, K, act)):
        rc = _lib.lib().tair_gemm_bf16(a2.data_ptr(), lda, w2.data_ptr(), ldw, M, N, K, C.byref(e), _stream())
    _lib.check(rc, "tair_gemm_bf16")
    return out


_sk_ws: dict = {}
# A workspace that is outgrown is RETIRED, never freed: a captured CUDA graph may hold its address (graphs are captured on
# the warm-up stream, so the workspaces of that stream are shared by every graph captured there).
_retired_ws: list = []


def _splitk_workspace(device, need: int) -> torch.Tensor:
    """Scratch for split-K partial sums, one buffer per (device, stream) like the GroupNorm workspace: two streams of one
    process (ControlNet beside the UNet encoder) may run split-K convolutions at the same time."""
    key = (device, torch.cuda.current_stream().cuda_stream)
    ws = _sk_ws.get(key)
    if ws is None or ws.numel() < need:
        if ws is not None:
            _retired_ws.append(ws)
        ws = torch.empty(max(need, 16 << 20), device=device, dtype=torch.uint8)
        _sk_ws[key] = ws
    return ws


def conv3x3(x: torch.Tensor, w: torch.Tensor, *, stride: int = 1, pad: int = 1, bias=None, residual=None,
            rowgroup=None, rows_per_group=0, act: int = ACT_NONE, out: Optional[torch.Tensor] = None,
            out_dtype=BF16, real_cin: Optional[int] = None) -> torch.Tensor:
    """3x3 convolution on channels-last bf16: x [B,H,W,Cin], w [Cout, 9*Cin] -> [B,Ho,Wo,Cout].
    pad=1: PyTorch padding=1; pad=0: zero row/column on the bottom/right only (VAE downsampler).
    ``real_cin``: the layer's true input channels when x is zero-padded to the 64-channel k-block (work accounting only)."""
    _cuda(x, "x", BF16), _cuda(w, "w", BF16)
    if x.dim() != 4 or not x.is_contiguous():
        raise TairError("conv3x3: x must be a contiguous [B,H,W,C] tensor")
    B, H, W, Cin = x.shape
    Cout = w.shape[0]
    if w.dim() != 2 or w.shape[1] != 9 * Cin or not w.is_contiguous():
        raise TairError(f"conv3x3: w must be contiguous [Cout, 9*Cin], got {tuple(w.shape)}")
    Ho, Wo = (H + pad - 2) // stride + 1, (W + pad - 2) // stride + 1
    M = B * Ho * Wo
    if out is None:
        out = torch.empty((B, Ho, Wo, Cout), device=x.device, dtype=out_dtype)
    o2 = out.view(M, -1) if out.dim() == 4 else out
    r2 = residual.view(M, -1) if (residual is not None and residual.dim() == 4) else residual
    e = _make_epilogue(o2, M, Cout, bias, r2, rowgroup, rows_per_group, act)
    if Ho * Wo <= 64 and Cin >= 448:
        # deep-K layer on an (at most) 8x8 map: lend the library a per-stream scratch so it can run a 3-way split-K
        # (too few 128-row tiles to fill the SMs otherwise); see tair_epilogue.workspace in include/tair_b200.h
        ws = _splitk_workspace(x.device, 3 * M * Cout * 4)
        e.workspace, e.workspace_bytes = ws.data_ptr(), ws.numel()
    with _timed("conv3x3", 2.0 * M * Cout * 9 * (real_cin or Cin), (B, H, W, Cin, Cout, stride)):
        rc = _lib.lib().tair_conv3x3_bf16(x.data_ptr(), w.data_ptr(), B, H, W, Cin, Cout, stride, pad, C.byref(e), _stream())
    _lib.check(rc, "tair_conv3x3_bf16")
    return out


def launch_count() -> int:
    return int(_lib.lib().tair_launch_count())


def reset_launch_count() -> None:
    _lib.lib().tair_launch_count_reset()


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, B: int, H: int, Lq: int, Lk: int,
              head_dim: int = 64, scale: Optional[float] = None, causal: bool = False,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax(q k^T * scale) v per (batch, head).

    q [B*Lq, >=H*D], k/v [B*Lk, >=H*D] are 2-D bf16 views with unit inner stride (column slices of a fused
    projection buffer are fine); head h lives in columns [h*D, (h+1)*D).  Returns [B*Lq, H*D] bf16.
    """
    for t, n in ((q, "q"), (k, "k"), (v, "v")):
        _cuda(t, n, BF16)
    q2, ldq = _rows(q, "q")
    k2, ldk = _rows(k, "k")
    v2, ldv = _rows(v, "v")
    if q2.shape[0] != B * Lq or k2.shape[0] != B * Lk or v2.shape[0] != B * Lk:
        raise TairError("attention: row counts do not match B*Lq / B*Lk")
    if out is None:
        out = torch.empty((B * Lq, H * head_dim), device=q.device, dtype=BF16)
    o2, ldo = _rows(out, "out")
    if scale is None:
        scale = head_dim ** -0.5
    with _timed("attention", 4.0 * B * H * Lq * Lk * head_dim, (B, H, Lq, Lk)):
        rc = _lib.lib().tair_attention_bf16(q2.data_ptr(), ldq, k2.data_ptr(), ldk, v2.data_ptr(), ldv, o2.data_ptr(),
                                            ldo, B, H, Lq, Lk, head_dim, float(scale), int(causal), _stream())
    _lib.check(rc, "tair_attention_bf16")
    return out


# ---------------------------------------------------------------------------------------------
# memory-bound kernels
# ---------------------------------------------------------------------------------------------
_gn_ws: dict = {}


def _gn_workspace(device, B: int, groups: int) -> torch.Tensor:
    need = int(_lib.lib().tair_groupnorm_workspace_bytes(B, groups))
    key = (device, torch.cuda.current_stream().cuda_stream)
    ws = _gn_ws.get(key)
    if ws is None or ws.numel() < need:
        if ws is not None:
            _retired_ws.append(ws)
        ws = torch.empty(max(need, 1 << 20), device=device, dtype=torch.uint8)
        _gn_ws[key] = ws
    return ws


def groupnorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, *, groups: int = 32, eps: float = 1e-5,
              act: int = ACT_NONE, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm(+SiLU/GELU) on channels-last bf16 x [B, ..., C] (any number of spatial dims)."""
    _cuda(x, "x", BF16), _cuda(gamma, "gamma", torch.float32), _cuda(beta, "beta", torch.float32)
    if not x.is_contiguous():
        raise TairError("groupnorm: x must be contiguous channels-last")
    B, C = x.shape[0], x.shape[-1]
    HW = x.numel() // (B * C)
    if out is None:
        out = torch.empty_like(x)
    ws = _gn_workspace(x.device, B, groups)
    with _timed("groupnorm", 6.0 * x.numel(), tuple(x.shape)):  # bytes: two reads + one write of a bf16 tensor
        rc = _lib.lib().tair_groupnorm_nhwc(x.data_ptr(), out.data_ptr(), gamma.data_ptr(), beta.data_ptr(), B, HW, C,
                                            groups, float(eps), act, ws.data_ptr(), _stream())
    _lib.check(rc, "tair_groupnorm_nhwc")
    return out


def row_stats(x: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """(mean, rstd) per row of a bf16 [M,C] matrix -> fp32 [M,2]; the LayerNorm that owns them is folded into its
    consumer GEMM (``gemm(..., ln=(stats, col_sum))``)."""
    _cuda(x, "x", BF16)
    x2, ldx = _rows(x, "x")
    out = torch.empty((x2.shape[0], 2), device=x.device, dtype=torch.float32)
    with _timed("layernorm_stats", 4.0 * x2.numel(), tuple(x2.shape)):   # algorithmic bytes of the LayerNorm it replaces
        rc = _lib.lib().tair_row_stats(x2.data_ptr(), ldx, out.data_ptr(), x2.shape[0], x2.shape[1], float(eps), _stream())
    _lib.check(rc, "tair_row_stats")
    return out


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, *, eps: float = 1e-5,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _cuda(x, "x", BF16), _cuda(gamma, "gamma", torch.float32), _cuda(beta, "beta", torch.float32)
    x2, ldx = _rows(x, "x")
    if out is None:
        out = torch.empty((x2.shape[0], x2.shape[1]), device=x.device, dtype=BF16)
    o2, ldy = _rows(out, "out")
    with _timed("layernorm", 4.0 * x2.numel(), tuple(x2.shape)):  # bytes: one read + one write
        rc = _lib.lib().tair_layernorm(x2.data_ptr(), ldx, o2.data_ptr(), ldy, gamma.data_ptr(), beta.data_ptr(),
                                       x2.shape[0], x2.shape[1], float(eps), _stream())
    _lib.check(rc, "tair_layernorm")
    return out


def sampler_update(x, v_cond, noise, t, tables, *, v_uncond=None, cfg_scale: float = 1.0, cfg_scale_dev=None, out=None,
                   pred_x0=None):
    """tables = (A, B, posterior_mean_coef1, posterior_mean_coef2, posterior_variance) with x0 = A[t] x - B[t] v:
    fp32 CUDA vectors; t int64 [B].  ``cfg_scale_dev``: optional 1-element fp32 CUDA tensor overriding ``cfg_scale``."""
    def chk(tt, n):
        _cuda(tt, n, torch.float32)
        if not tt.is_contiguous() or tt.shape != x.shape or tt.device != x.device:
            raise TairError(f"sampler_update: {n} must be a contiguous fp32 tensor of x's shape on x's device")
        return tt
    _cuda(x, "x", torch.float32)
    for tt, n in ((x, "x"), (v_cond, "v"), (noise, "noise")):
        chk(tt, n)
    for tt, n in ((v_uncond, "v_uncond"), (out, "out"), (pred_x0, "pred_x0")):
        if tt is not None:
            chk(tt, n)
    _cuda(t, "t", torch.int64)
    if cfg_scale_dev is not None:
        _cuda(cfg_scale_dev, "cfg_scale_dev", torch.float32)
    B = x.shape[0]
    if t.numel() != B or not t.is_contiguous():
        raise TairError("sampler_update: t must be a contiguous int64 vector with one entry per sample")
    per = x.numel() // B
    if out is None:
        out = torch.empty_like(x)
    tabs = [_cuda(tb, "schedule table", torch.float32).data_ptr() for tb in tables]
    rc = _lib.lib().tair_sampler_update(x.data_ptr(), v_cond.data_ptr(), _ptr(v_uncond), float(cfg_scale),
                                        _ptr(cfg_scale_dev), noise.data_ptr(), out.data_ptr(), _ptr(pred_x0),
                                        t.data_ptr(), *tabs, B, per, _stream())
    _lib.check(rc, "tair_sampler_update")
    return out


def sampler_multistep_update(x, v_cond, noise, t, tables, *, x0_hist=None, v_uncond=None, cfg_scale: float = 1.0,
                             cfg_scale_dev=None, out=None):
    """tables = (P, Q, a, b, c, d): x0 = P[t] x - Q[t] v, x_next = ((b[t] x0 + a[t] x) + c[t] x0_hist) + d[t] noise,
    then x0_hist <- x0 in place (DDIM / DPM-Solver++(2M)).  fp32 CUDA vectors; t int64 [B].  ``x0_hist`` is not read
    where c[t] == 0 and may be None only when every c[t] used is 0."""
    def chk(tt, n):
        _cuda(tt, n, torch.float32)
        if not tt.is_contiguous() or tt.shape != x.shape or tt.device != x.device:
            raise TairError(f"sampler_multistep_update: {n} must be a contiguous fp32 tensor of x's shape on x's device")
        return tt
    _cuda(x, "x", torch.float32)
    for tt, n in ((x, "x"), (v_cond, "v"), (noise, "noise")):
        chk(tt, n)
    for tt, n in ((v_uncond, "v_uncond"), (out, "out"), (x0_hist, "x0_hist")):
        if tt is not None:
            chk(tt, n)
    _cuda(t, "t", torch.int64)
    if cfg_scale_dev is not None:
        _cuda(cfg_scale_dev, "cfg_scale_dev", torch.float32)
    B = x.shape[0]
    if t.numel() != B or not t.is_contiguous():
        raise TairError("sampler_multistep_update: t must be a contiguous int64 vector with one entry per sample")
    if len(tables) != 6:
        raise TairError("sampler_multistep_update: tables must be (P, Q, a, b, c, d)")
    per = x.numel() // B
    if out is None:
        out = torch.empty_like(x)
    tabs = [_cuda(tb, "schedule table", torch.float32).data_ptr() for tb in tables]
    rc = _lib.lib().tair_sampler_multistep_update(x.data_ptr(), v_cond.data_ptr(), _ptr(v_uncond), float(cfg_scale),
                                                  _ptr(cfg_scale_dev), noise.data_ptr(), out.data_ptr(), _ptr(x0_hist),
                                                  t.data_ptr(), *tabs, B, per, _stream())
    _lib.check(rc, "tair_sampler_multistep_update")
    return out


def sampler_unipc_update(x, v_cond, t, table, *, x_corr, x0_hist, v_uncond=None, cfg_scale: float = 1.0,
                         cfg_scale_dev=None, out=None):
    """One UniPC step from the packed fp32 [N, 16] ``table`` (columns P, Q, u, e, f, g0..g2, a, b, c0..c2, padding):
    x0 = P[t] x - Q[t] v, xc = u x + e x_corr + f x0 + sum_k g_k h_k, x_next = a xc + b x0 + sum_k c_k h_k, then
    x_corr <- xc and the history shifts (h0 <- x0, h_k <- h_{k-1}) in place.  ``x0_hist`` is a contiguous fp32
    [K, *x.shape] buffer, K in {1, 2, 3}; t int64 [B].  A state term enters a sum only where its coefficient is non-zero;
    the fp32 evaluation order is documented at ``tair_sampler_unipc_update`` in include/tair_b200.h."""
    def chk(tt, n, shape):
        _cuda(tt, n, torch.float32)
        if not tt.is_contiguous() or tt.shape != shape or tt.device != x.device:
            raise TairError(f"sampler_unipc_update: {n} must be a contiguous fp32 tensor of shape {tuple(shape)} on "
                            f"x's device")
        return tt
    _cuda(x, "x", torch.float32)
    for tt, n in ((x, "x"), (v_cond, "v"), (x_corr, "x_corr")):
        chk(tt, n, x.shape)
    for tt, n in ((v_uncond, "v_uncond"), (out, "out")):
        if tt is not None:
            chk(tt, n, x.shape)
    _cuda(x0_hist, "x0_hist", torch.float32)
    K = x0_hist.shape[0] if x0_hist.dim() == x.dim() + 1 else 0
    if not 1 <= K <= 3:
        raise TairError("sampler_unipc_update: x0_hist must have shape (K, *x.shape) with K in {1, 2, 3}")
    chk(x0_hist, "x0_hist", (K,) + tuple(x.shape))
    _cuda(t, "t", torch.int64)
    if cfg_scale_dev is not None:
        _cuda(cfg_scale_dev, "cfg_scale_dev", torch.float32)
    B = x.shape[0]
    if t.numel() != B or not t.is_contiguous():
        raise TairError("sampler_unipc_update: t must be a contiguous int64 vector with one entry per sample")
    _cuda(table, "table", torch.float32)
    if table.dim() != 2 or table.shape[1] != 16 or not table.is_contiguous() or table.device != x.device:
        raise TairError("sampler_unipc_update: table must be a contiguous fp32 [N, 16] tensor on x's device")
    per = x.numel() // B
    if out is None:
        out = torch.empty_like(x)
    rc = _lib.lib().tair_sampler_unipc_update(x.data_ptr(), v_cond.data_ptr(), _ptr(v_uncond), float(cfg_scale),
                                              _ptr(cfg_scale_dev), out.data_ptr(), x_corr.data_ptr(),
                                              x0_hist.data_ptr(), t.data_ptr(), table.data_ptr(), K, B, per, _stream())
    _lib.check(rc, "tair_sampler_unipc_update")
    return out


def timestep_embedding(t: torch.Tensor, dim: int, max_period: float = 10000.0) -> torch.Tensor:
    _cuda(t, "t", torch.int64)
    out = torch.empty((t.shape[0], dim), device=t.device, dtype=BF16)
    rc = _lib.lib().tair_timestep_embedding(t.data_ptr(), out.data_ptr(), t.shape[0], dim, float(max_period), _stream())
    _lib.check(rc, "tair_timestep_embedding")
    return out


def nchw_to_nhwc(x: torch.Tensor, c_pad: Optional[int] = None) -> torch.Tensor:
    """(B,C,H,W) fp32 -> [B,H,W,Cpad] bf16 with zero channel padding."""
    _cuda(x, "x", torch.float32)
    x = x.contiguous()
    B, C, H, W = x.shape
    cp = c_pad or C
    out = torch.empty((B, H, W, cp), device=x.device, dtype=BF16)
    rc = _lib.lib().tair_nchw_to_nhwc_bf16(x.data_ptr(), out.data_ptr(), B, C, H * W, cp, _stream())
    _lib.check(rc, "tair_nchw_to_nhwc_bf16")
    return out


def nhwc_to_nchw(x: torch.Tensor, channels: Optional[int] = None) -> torch.Tensor:
    """[B,H,W,C'] bf16 -> (B,C,H,W) fp32 keeping the first ``channels`` channels."""
    _cuda(x, "x", BF16)
    B, H, W, ld = x.shape
    if not x.is_contiguous():
        raise TairError("nhwc_to_nchw: x must be contiguous")
    C = channels or ld
    out = torch.empty((B, C, H, W), device=x.device, dtype=torch.float32)
    rc = _lib.lib().tair_nhwc_to_nchw_f32(x.data_ptr(), ld, out.data_ptr(), B, C, H * W, _stream())
    _lib.check(rc, "tair_nhwc_to_nchw_f32")
    return out


def concat_add(a: torch.Tensor, b: torch.Tensor, c: Optional[torch.Tensor] = None) -> torch.Tensor:
    """channels-last concat [a | b (+c)] for tensors [..., C1], [..., C2]."""
    _cuda(a, "a", BF16), _cuda(b, "b", BF16)
    if not (a.is_contiguous() and b.is_contiguous() and (c is None or c.is_contiguous())):
        raise TairError("concat_add: inputs must be contiguous")
    C1, C2 = a.shape[-1], b.shape[-1]
    M = a.numel() // C1
    out = torch.empty((*a.shape[:-1], C1 + C2), device=a.device, dtype=BF16)
    rc = _lib.lib().tair_concat_add(a.data_ptr(), b.data_ptr(), _ptr(c), out.data_ptr(), M, C1, C2, _stream())
    _lib.check(rc, "tair_concat_add")
    return out


def add(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _cuda(a, "a", BF16), _cuda(b, "b", BF16)
    if not (a.is_contiguous() and b.is_contiguous()) or a.shape != b.shape:
        raise TairError("add: inputs must be contiguous and of equal shape")
    if out is None:
        out = torch.empty_like(a)
    rc = _lib.lib().tair_add_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.numel(), _stream())
    _lib.check(rc, "tair_add_bf16")
    return out


def upsample2x(x: torch.Tensor) -> torch.Tensor:
    _cuda(x, "x", BF16)
    if x.dim() != 4 or not x.is_contiguous():
        raise TairError("upsample2x: x must be contiguous [B,H,W,C]")
    B, H, W, Cc = x.shape
    out = torch.empty((B, 2 * H, 2 * W, Cc), device=x.device, dtype=BF16)
    rc = _lib.lib().tair_upsample2x_nhwc(x.data_ptr(), out.data_ptr(), B, H, W, Cc, _stream())
    _lib.check(rc, "tair_upsample2x_nhwc")
    return out


def msda_forward(value: torch.Tensor, spatial_shapes: torch.Tensor, level_start_index: torch.Tensor,
                 sampling_locations: torch.Tensor, attention_weights: torch.Tensor,
                 out_dtype=None) -> torch.Tensor:
    """Same arguments as ``_C.ms_deform_attn_forward`` minus im2col_step (vision.cpp:52-55).
    value [B,S,M,D] fp32|bf16; shapes int64 [L,2]; start int64 [L]; loc fp32 [B,Lq,M,L,P,2]; w fp32 [B,Lq,M,L,P]."""
    _cuda(value, "value")
    if value.dtype not in (torch.float32, BF16):
        raise TairError("msda_forward: value must be fp32 or bf16")
    _cuda(spatial_shapes, "spatial_shapes", torch.int64), _cuda(level_start_index, "level_start_index", torch.int64)
    _cuda(sampling_locations, "sampling_locations", torch.float32)
    _cuda(attention_weights, "attention_weights", torch.float32)
    for tt, n in ((value, "value"), (sampling_locations, "sampling_locations"), (attention_weights, "attention_weights"),
                  (spatial_shapes, "spatial_shapes"), (level_start_index, "level_start_index")):
        if not tt.is_contiguous():
            raise TairError(f"msda_forward: {n} must be contiguous")
    B, S, M, D = value.shape
    _, Lq, M2, L, P, two = sampling_locations.shape
    if M2 != M or two != 2 or tuple(attention_weights.shape) != (B, Lq, M, L, P):
        raise TairError("msda_forward: inconsistent shapes")
    out_dtype = out_dtype or value.dtype
    out = torch.empty((B, Lq, M * D), device=value.device, dtype=out_dtype)
    rc = _lib.lib().tair_msda_forward(value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
                                      sampling_locations.data_ptr(), attention_weights.data_ptr(), out.data_ptr(),
                                      B, S, M, D, L, Lq, P, int(value.dtype == BF16), int(out_dtype == BF16), _stream())
    _lib.check(rc, "tair_msda_forward")
    return out


def blend_tiles(tiles: torch.Tensor, n_h: int, n_w: int, overlap: int, out_h: int, out_w: int) -> torch.Tensor:
    """tiles [P, C, T, T] fp32 in row-major grid order -> (1, C, out_h, out_w) fp32."""
    _cuda(tiles, "tiles", torch.float32)
    if tiles.dim() != 4 or tiles.shape[2] != tiles.shape[3] or not tiles.is_contiguous():
        raise TairError("blend_tiles: tiles must be contiguous [P,C,T,T]")
    P_, Cc, T, _ = tiles.shape
    out = torch.empty((1, Cc, out_h, out_w), device=tiles.device, dtype=torch.float32)
    rc = _lib.lib().tair_blend_tiles(tiles.data_ptr(), out.data_ptr(), P_, n_h, n_w, Cc, T, overlap, out_h, out_w, _stream())
    _lib.check(rc, "tair_blend_tiles")
    return out


def msda_fused(value: torch.Tensor, spatial_shapes: torch.Tensor, level_start_index: torch.Tensor, proj: torch.Tensor,
               ref: torch.Tensor, *, B: int, Lq: int, n_heads: int, n_levels: int, n_points: int,
               q_per_ref: int = 1, ref_shared: bool = False) -> torch.Tensor:
    """value bf16 [B,S,M,D]; proj fp32 [B*Lq, >= M*L*P*3] (raw offsets then raw logits); ref fp32
    [(B,) Lq/q_per_ref, L, 2|4] -> bf16 [B*Lq, M*D]."""
    _cuda(value, "value", BF16), _cuda(proj, "proj"), _cuda(ref, "ref", torch.float32)
    if proj.dtype not in (torch.float32, BF16):
        raise TairError("msda_fused: proj must be fp32 or bf16")
    _cuda(spatial_shapes, "spatial_shapes", torch.int64), _cuda(level_start_index, "level_start_index", torch.int64)
    if not (value.is_contiguous() and ref.is_contiguous()):
        raise TairError("msda_fused: value / ref must be contiguous")
    p2, ldp = _rows(proj, "proj")
    _, S, M, D = value.shape
    ref_dim = ref.shape[-1]
    n_ref = Lq // q_per_ref
    if M != n_heads or p2.shape[0] != B * Lq or ref.numel() != (1 if ref_shared else B) * n_ref * n_levels * ref_dim:
        raise TairError("msda_fused: inconsistent shapes")
    out = torch.empty((B * Lq, M * D), device=value.device, dtype=BF16)
    stride = 0 if ref_shared else n_ref * n_levels * ref_dim
    with _timed("msda", 2.0 * out.numel() + 2.0 * value.numel() + 4.0 * p2.shape[0] * M * n_levels * n_points * 3,
                (B, Lq, M, n_levels, n_points)):
        rc = _lib.lib().tair_msda_fused(value.data_ptr(), spatial_shapes.data_ptr(), level_start_index.data_ptr(),
                                        p2.data_ptr(), ldp, int(proj.dtype == BF16), ref.data_ptr(), ref_dim, stride,
                                        q_per_ref, out.data_ptr(),
                                        B, S, M, D, n_levels, Lq, n_points, _stream())
    _lib.check(rc, "tair_msda_fused")
    return out


def attention_seq(qkv: torch.Tensor, *, n_heads: int, L: int, n_outer: int, n_inner: int, outer_stride: int,
                  inner_stride: int, tok_stride: int, scale: float, out: Optional[torch.Tensor] = None,
                  real_head_dim: int = 64) -> torch.Tensor:
    """Self-attention over many short strided sequences on the tcgen05 flash kernel.  qkv bf16 [rows, 3*H*64]
    (q | k | v, 64-column head slots, narrower heads zero-padded); returns [rows, H*64] in the same row order."""
    _cuda(qkv, "qkv", BF16)
    q2, ld = _rows(qkv, "qkv")
    E = n_heads * 64
    if q2.shape[1] != 3 * E:
        raise TairError(f"attention_seq: expected {3 * E} columns, got {q2.shape[1]}")
    if out is None:
        out = torch.empty((q2.shape[0], E), device=qkv.device, dtype=BF16)
    o2, ldo = _rows(out, "out")
    base = q2.data_ptr()
    # algorithmic FLOPs count the real head width, not the zero-padded 64-column slot
    with _timed("attention_seq", 4.0 * n_outer * n_inner * n_heads * L * L * real_head_dim, (n_outer, n_inner, n_heads, L)):
        rc = _lib.lib().tair_attention_seq_bf16(base, base + 2 * E, base + 4 * E, ld, o2.data_ptr(), ldo, n_heads, L,
                                                n_outer, n_inner, outer_stride, inner_stride, tok_stride, float(scale),
                                                _stream())
    _lib.check(rc, "tair_attention_seq_bf16")
    return out


def attention_seq32(qkv: torch.Tensor, *, n_heads: int, L: int, n_outer: int, n_inner: int, outer_stride: int,
                    inner_stride: int, tok_stride: int, scale: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Self-attention over many short (L <= 128) strided sequences with 32-wide heads on UNPADDED projections: qkv bf16
    [rows, 3*H*32] (q | k | v); returns [rows, H*32] in the same row order (csrc/attn_small.cu)."""
    _cuda(qkv, "qkv", BF16)
    q2, ld = _rows(qkv, "qkv")
    E = n_heads * 32
    if q2.shape[1] != 3 * E:
        raise TairError(f"attention_seq32: expected {3 * E} columns, got {q2.shape[1]}")
    last = (n_outer - 1) * outer_stride + (n_inner - 1) * inner_stride + (L - 1) * tok_stride
    if min(n_outer, n_inner, L, tok_stride) < 1 or min(outer_stride, inner_stride) < 0 or last >= q2.shape[0]:
        raise TairError("attention_seq32: the sequence addressing leaves the qkv rows")
    if out is None:
        out = torch.empty((q2.shape[0], E), device=qkv.device, dtype=BF16)
    _cuda(out, "out", BF16)
    o2, ldo = _rows(out, "out")
    if o2.shape[0] != q2.shape[0] or o2.shape[1] != E:
        raise TairError(f"attention_seq32: out must be [{q2.shape[0]}, {E}]")
    base = q2.data_ptr()
    with _timed("attention_seq", 4.0 * n_outer * n_inner * n_heads * L * L * 32, (n_outer, n_inner, n_heads, L)):
        rc = _lib.lib().tair_attention_seq32_bf16(base, base + 2 * E, base + 4 * E, ld, o2.data_ptr(), ldo, n_heads, L,
                                                  n_outer, n_inner, outer_stride, inner_stride, tok_stride, float(scale),
                                                  _stream())
    _lib.check(rc, "tair_attention_seq32_bf16")
    return out


def tiles_bicubic(image_u8: torch.Tensor, origins: torch.Tensor, bounds: torch.Tensor, coeffs: torch.Tensor,
                  tile: int, out_size: int) -> torch.Tensor:
    """image_u8 [Hp,Wp,3] uint8 (zero-padded LQ), origins [P,2] int32 (y,x) -> [P,3,out,out] fp32 in [0,1],
    bit-identical to PIL BICUBIC + ToTensor per tile."""
    _cuda(image_u8, "image", torch.uint8), _cuda(origins, "origins", torch.int32)
    _cuda(bounds, "bounds", torch.int32), _cuda(coeffs, "coeffs", torch.int32)
    if image_u8.dim() != 3 or image_u8.shape[2] != 3 or not image_u8.is_contiguous():
        raise TairError("tiles_bicubic: image must be a contiguous [H,W,3] uint8 tensor")
    P = origins.shape[0]
    Hp, Wp = image_u8.shape[:2]
    tmp = torch.empty((P, tile, out_size, 3), device=image_u8.device, dtype=torch.uint8)
    dst = torch.empty((P, 3, out_size, out_size), device=image_u8.device, dtype=torch.float32)
    rc = _lib.lib().tair_tiles_bicubic_u8(image_u8.data_ptr(), Hp, Wp, origins.contiguous().data_ptr(), P, tile, out_size,
                                          bounds.contiguous().data_ptr(), coeffs.contiguous().data_ptr(), coeffs.shape[1],
                                          tmp.data_ptr(), dst.data_ptr(), _stream())
    _lib.check(rc, "tair_tiles_bicubic_u8")
    return dst


def attention_windows(qkv: torch.Tensor, *, n_heads: int, L: int, n_windows: int, scale: float,
                      bias: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
                      real_head_dim: int = 64) -> torch.Tensor:
    """Swin window attention: qkv bf16 [n_windows*L, 3*H*64] (q | k | v, 64-column head slots); bias fp32
    [nw, H, L(key), L(query)] = (relative-position bias + mask) / scale, window w uses table w % nw."""
    _cuda(qkv, "qkv", BF16)
    q2, ld = _rows(qkv, "qkv")
    E = n_heads * 64
    if q2.shape[1] != 3 * E or q2.shape[0] != n_windows * L:
        raise TairError(f"attention_windows: expected [{n_windows * L}, {3 * E}], got {tuple(q2.shape)}")
    nw = 1
    if bias is not None:
        _cuda(bias, "bias", torch.float32)
        if bias.dim() != 4 or tuple(bias.shape[1:]) != (n_heads, L, L) or not bias.is_contiguous():
            raise TairError("attention_windows: bias must be contiguous [nw, H, L, L] fp32")
        nw = bias.shape[0]
    if out is None:
        out = torch.empty((q2.shape[0], E), device=qkv.device, dtype=BF16)
    o2, ldo = _rows(out, "out")
    base = q2.data_ptr()
    with _timed("attention_windows", 4.0 * n_windows * n_heads * L * L * real_head_dim, (n_windows, n_heads, L)):
        rc = _lib.lib().tair_attention_windows_bf16(base, base + 2 * E, base + 4 * E, ld, o2.data_ptr(), ldo, n_heads, L,
                                                    n_windows, None if bias is None else bias.data_ptr(), nw, float(scale),
                                                    _stream())
    _lib.check(rc, "tair_attention_windows_bf16")
    return out


def layernorm_ragged(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, c_valid: int, *, eps: float = 1e-5) -> torch.Tensor:
    _cuda(x, "x", BF16), _cuda(gamma, "gamma", torch.float32), _cuda(beta, "beta", torch.float32)
    x2, ldx = _rows(x, "x")
    out = torch.empty_like(x2)
    rc = _lib.lib().tair_layernorm_ragged(x2.data_ptr(), ldx, out.data_ptr(), out.stride(0), gamma.data_ptr(), beta.data_ptr(),
                                          x2.shape[0], x2.shape[1], int(c_valid), float(eps), _stream())
    _lib.check(rc, "tair_layernorm_ragged")
    return out


def gather_rows(x: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    _cuda(x, "x", BF16), _cuda(idx, "idx", torch.int32)
    x2, ldx = _rows(x, "x")
    out = torch.empty((idx.numel(), x2.shape[1]), device=x.device, dtype=BF16)
    rc = _lib.lib().tair_gather_rows_bf16(x2.data_ptr(), ldx, idx.data_ptr(), out.data_ptr(), out.stride(0), idx.numel(),
                                          x2.shape[1], _stream())
    _lib.check(rc, "tair_gather_rows_bf16")
    return out


def leaky_relu(x: torch.Tensor, slope: float) -> torch.Tensor:
    _cuda(x, "x", BF16)
    if not x.is_contiguous():
        raise TairError("leaky_relu: x must be contiguous")
    out = torch.empty_like(x)
    rc = _lib.lib().tair_leaky_relu_bf16(x.data_ptr(), out.data_ptr(), x.numel(), float(slope), _stream())
    _lib.check(rc, "tair_leaky_relu_bf16")
    return out


def softmax_rows(x: torch.Tensor, scale: float = 1.0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _cuda(x, "x", BF16)
    x2, ldx = _rows(x, "x")
    if out is None:
        out = torch.empty_like(x2)
    o2, ldy = _rows(out, "out")
    rc = _lib.lib().tair_softmax_rows_bf16(x2.data_ptr(), ldx, o2.data_ptr(), ldy, x2.shape[0], x2.shape[1], float(scale), _stream())
    _lib.check(rc, "tair_softmax_rows_bf16")
    return out


def transpose(x: torch.Tensor) -> torch.Tensor:
    """bf16 [batch, R, C] (or [R, C]) contiguous -> [batch, C, R]."""
    _cuda(x, "x", BF16)
    if not x.is_contiguous():
        raise TairError("transpose: x must be contiguous")
    x3 = x if x.dim() == 3 else x[None]
    Bn, R, Cc = x3.shape
    out = torch.empty((Bn, Cc, R), device=x.device, dtype=BF16)
    rc = _lib.lib().tair_transpose_bf16(x3.data_ptr(), Cc, R * Cc, out.data_ptr(), R, R * Cc, Bn, R, Cc, _stream())
    _lib.check(rc, "tair_transpose_bf16")
    return out if x.dim() == 3 else out[0]


def testr_postprocess(pred_logits: torch.Tensor, pred_ctrl_points: torch.Tensor, pred_texts: torch.Tensor,
                      image_w: float, image_h: float):
    """Dense TESTR outputs (B,Q,P,1) / (B,Q,P,2) / (B,Q,L,V) fp32 -> (scores fp32 [B,Q], polygons fp32 [B,Q,2P] in pixels,
    recs uint8 [B,Q,L], the packed uint8 buffer the three are views of) in one kernel; see tair_testr_postprocess."""
    for t, n in ((pred_logits, "pred_logits"), (pred_ctrl_points, "pred_ctrl_points"), (pred_texts, "pred_texts")):
        _cuda(t, n, torch.float32)
        if not t.is_contiguous():
            raise TairError(f"testr_postprocess: {n} must be contiguous")
    B, Q, P = pred_ctrl_points.shape[:3]
    L, V = pred_texts.shape[2:]
    if pred_logits.numel() != B * Q * P or pred_ctrl_points.shape[3] != 2 or tuple(pred_texts.shape[:2]) != (B, Q):
        raise TairError("testr_postprocess: inconsistent shapes (one class per control point expected)")
    dev = pred_logits.device
    # one packed buffer (scores | polygons | recs) so that the caller brings everything to the host in a single copy
    n_s, n_p = B * Q * 4, B * Q * 2 * P * 4
    pack = torch.empty((n_s + n_p + B * Q * L,), device=dev, dtype=torch.uint8)
    scores = pack[:n_s].view(torch.float32).view(B, Q)
    polys = pack[n_s:n_s + n_p].view(torch.float32).view(B, Q, 2 * P)
    recs = pack[n_s + n_p:].view(B, Q, L)
    rc = _lib.lib().tair_testr_postprocess(pred_logits.data_ptr(), pred_ctrl_points.data_ptr(), pred_texts.data_ptr(),
                                           scores.data_ptr(), polys.data_ptr(), recs.data_ptr(), B * Q, P, L, V,
                                           float(image_w), float(image_h), _stream())
    _lib.check(rc, "tair_testr_postprocess")
    return scores, polys, recs, pack
