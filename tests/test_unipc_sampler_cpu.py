"""UniPC without a GPU: the product's float64 packed tables against the float64 paper-form restatement
(oracle/unipc_sampler.py) on the analytic Gaussian model, identities with DPM-Solver++(2M) and DDIM, zero-terminal-SNR
handling, convergence, and argument validation of the fused update's C entry point."""
import os

import numpy as np
import pytest

from oracle import multistep_sampler as OM, sampler as OS, unipc_sampler as OU
from tair_b200.sampler import DDIMSampler, DPMSolverSampler, SpacedSampler, UniPCSampler
from tair_b200.sampler.unipc_sampler import COL_A, COL_B, COL_C, COL_E, COL_F, COL_G, COL_U

BETAS = OS.diffusion_betas()                           # zero terminal SNR, as the val config
BETAS_SNR = OS.diffusion_betas(zero_snr=False)


def apply_tables(tabs, betas, model, x_T, parameterization="v"):
    """The kernel's update in float64, with NaN-filled state: row t = N-1-i at step i, each term added only where its
    coefficient is non-zero, then x_corr <- xc and the history shifts."""
    T = tabs["table"]
    N = len(T)
    abar_train = np.cumprod(1.0 - betas)
    x, xc, hist, out = x_T.copy(), np.full_like(x_T, np.nan), [np.full_like(x_T, np.nan)] * 3, []
    for i, tau in enumerate(tabs["timesteps"][::-1]):
        r, ab = T[N - 1 - i], abar_train[tau]
        if parameterization == "v":
            mo = model.v(x, ab)
        else:
            mo = (x - np.sqrt(ab) * model.x0_hat(x, ab)) / np.sqrt(1.0 - ab)
        x0 = r[0] * x - r[1] * mo
        c = 0.0
        for co, term in [(r[COL_U], x), (r[COL_E], xc), (r[COL_F], x0)] + [(r[COL_G + k], hist[k]) for k in range(3)]:
            if co != 0.0:
                c = c + co * term
        nx = 0.0
        for co, term in [(r[COL_A], c), (r[COL_B], x0)] + [(r[COL_C + k], hist[k]) for k in range(3)]:
            if co != 0.0:
                nx = nx + co * term
        x, xc, hist = nx, c, [x0, hist[0], hist[1]]
        out.append(x)
    return out


@pytest.mark.parametrize("betas,param", [(BETAS, "v"), (BETAS_SNR, "v"), (BETAS_SNR, "eps")],
                         ids=["v-zero-snr", "v", "eps"])
@pytest.mark.parametrize("corrector", [True, False])
@pytest.mark.parametrize("order", [1, 2, 3])
@pytest.mark.parametrize("N", [1, 2, 3, 5, 10, 20, 50])
def test_host_tables_match_paper_oracle(betas, param, corrector, order, N):
    model = OM.GaussianData(0.3, 0.7)
    x_T = np.random.default_rng(N).standard_normal(4096)
    s = UniPCSampler(betas, param, order=order, corrector=corrector)
    got = apply_tables(s.host_tables(N), betas, model, x_T, param)
    ref = []
    OU.sample_loop(model.x0_hat, betas, N, x_T, "unipc", order=order, corrector=corrector, trace=ref)
    assert len(got) == len(ref) == N
    for i, (g, r) in enumerate(zip(got, ref)):
        err = np.abs(g - r).max() / np.abs(r).max()
        assert err < 1e-12, (i, err)
    # the last step returns x0_hat(tau = 0)
    x_last = ref[-2] if N > 1 else x_T
    assert np.allclose(got[-1], model.x0_hat(x_last, np.cumprod(1.0 - betas)[0]), rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("betas", [BETAS, BETAS_SNR], ids=["zero-snr", "snr"])
@pytest.mark.parametrize("N", [2, 3, 10, 20, 50])
def test_unip2_is_dpm_solver_2m_and_unip1_is_ddim(betas, N):
    cols = {"ms_a": COL_A, "ms_b": COL_B, "ms_c": COL_C}
    for uni, ref in ((UniPCSampler(betas, order=2, corrector=False), DPMSolverSampler(betas)),
                     (UniPCSampler(betas, order=1, corrector=False), DDIMSampler(betas))):
        got, want = uni.host_tables(N)["table"], ref.host_tables(N)
        for k, col in cols.items():
            assert np.allclose(got[:, col], want[k], rtol=1e-13, atol=1e-15), (k, uni.order)
        assert not got[:, COL_C + 1:COL_C + 3].any()
        assert (got[:, COL_U] == 1.0).all() and not got[:, COL_E:COL_G + 3].any()


@pytest.mark.parametrize("order", [1, 2, 3])
@pytest.mark.parametrize("corrector", [True, False])
def test_zero_snr_tables(order, corrector):
    """Finite for every N; the first step is first order and uncorrected; no coefficient on a state slot this run has
    not written yet (slot k of the history holds x0 of step i-1-k, x_corr is written from step 0 on)."""
    spaced = SpacedSampler(BETAS)
    for N in range(1, 61):
        s = UniPCSampler(BETAS, order=order, corrector=corrector)
        tabs = s.host_tables(N)
        T = tabs["table"][::-1]                        # visiting order
        assert T.shape == (N, 16) and np.isfinite(T).all() and not T[:, 13:].any()
        spaced.make_schedule(N)
        assert np.array_equal(tabs["timesteps"], spaced.timesteps)
        orders = tabs["orders"]
        assert orders[0] == 1 and orders[-1] == 1 and orders.max() <= order
        if N > 2:
            assert orders[1] == 1                      # lambda(999) = -inf: no second-order step from point 1 either
        assert T[0, COL_U] == 1.0 and not T[0, COL_E:COL_G + 3].any() and not T[0, COL_C:COL_C + 3].any()
        for i in range(N):
            written = i                                # history slots 0 .. i-1 hold x0 of this run
            assert not T[i, COL_G + written:COL_G + 3].any(), (N, i)
            assert not T[i, COL_C + written:COL_C + 3].any(), (N, i)
            assert (T[i, COL_C:COL_C + 3] != 0).sum() == orders[i] - 1
            if corrector and i >= 1:
                assert T[i, COL_U] == 0.0 and T[i, COL_E] != 0.0 and T[i, COL_F] != 0.0
                assert (T[i, COL_G:COL_G + 3] != 0).sum() == orders[i - 1]
            else:
                assert T[i, COL_U] == 1.0 and not T[i, COL_E:COL_G + 3].any()
        # the last step targets the clean sample at first order: x_next = x0_hat(tau = 0)
        assert (T[-1, COL_A], T[-1, COL_B]) == (0.0, 1.0)
        s.make_schedule(N)
        assert s.unipc_table.numpy().tolist() == tabs["table"].astype(np.float32).tolist()


def test_argument_validation():
    with pytest.raises(ValueError):
        UniPCSampler(BETAS, order=4)
    with pytest.raises(ValueError):
        UniPCSampler(BETAS, order=0)
    s = UniPCSampler(BETAS)
    s.order = 5
    with pytest.raises(ValueError):
        s.make_schedule(10)
    with pytest.raises(ValueError):
        UniPCSampler(BETAS, "x0")
    for order in (1, 2, 3):
        with pytest.raises(ValueError):
            UniPCSampler(BETAS, "eps", order=order).make_schedule(20)
        tabs = UniPCSampler(BETAS_SNR, "eps", order=order).host_tables(20)
        assert np.isfinite(tabs["table"]).all()


def test_analytic_convergence_orders():
    """Relative RMS error of the endpoint against the exact probability-flow ODE solution mu + s x_T, 100 000 samples,
    float64 oracle loop, trailing zero-terminal-SNR schedule.  Values when this test was written:

      | (mu, s)    | sampler        | N=10    | 20      | 40      | 80      | err(40)/err(80) |
      |------------|----------------|---------|---------|---------|---------|-----------------|
      | (0.0, 2.0) | DPM-Solver++2M | 4.69e-2 | 1.42e-2 | 4.66e-3 | 1.52e-3 | 3.07            |
      | (0.0, 2.0) | UniPC-2        | 6.98e-2 | 1.86e-2 | 5.54e-3 | 1.65e-3 | 3.35            |
      | (0.0, 2.0) | UniPC-3        | 3.96e-2 | 1.24e-2 | 3.95e-3 | 1.20e-3 | 3.28            |
      | (0.5, 1.0) | DPM-Solver++2M | 1.48e-1 | 5.65e-2 | 1.95e-2 | 6.37e-3 | 3.06            |
      | (0.5, 1.0) | UniPC-2        | 1.64e-1 | 5.55e-2 | 1.82e-2 | 5.64e-3 | 3.22            |
      | (0.5, 1.0) | UniPC-3        | 1.52e-1 | 4.34e-2 | 1.38e-2 | 4.23e-3 | 3.27            |
      | (0.3, 0.5) | DPM-Solver++2M | 1.90e-1 | 1.21e-1 | 5.45e-2 | 2.02e-2 | 2.70            |
      | (0.3, 0.5) | UniPC-2        | 2.03e-1 | 1.22e-1 | 5.24e-2 | 1.85e-2 | 2.83            |
      | (0.3, 0.5) | UniPC-3        | 2.19e-1 | 1.17e-1 | 4.55e-2 | 1.50e-2 | 3.04            |

    UniP-2 without the corrector gives the DPM-Solver++(2M) row exactly.  The corrector raises the observed order of
    UniPC-2 over DPM-Solver++(2M) in every case (err(40)/err(80) 3.35 / 3.22 / 2.83 against 3.07 / 3.06 / 2.70), but only
    a little: neither reaches the third order (ratio 8) on this schedule.  UniPC-2 is not uniformly more accurate: for
    (0, 2) it is behind DPM-Solver++(2M) at every N, and for the other two cases it leads from N = 40 (N = 20 for
    (0.5, 1)).  UniPC-3 is the most accurate of the three at N = 80 in every case.  The test asserts the ratios and the
    N = 80 ordering of UniPC-3."""
    x_T = np.random.default_rng(0).standard_normal(100_000)
    kinds = {"dpmpp2m": dict(kind="dpmpp2m"), "unipc2": dict(order=2), "unipc3": dict(order=3),
             "unip2": dict(order=2, corrector=False)}
    for mu, s in ((0.0, 2.0), (0.5, 1.0), (0.3, 0.5)):
        model = OM.GaussianData(mu, s)
        exact = model.ode_endpoint(x_T)
        err = {}
        for name, kw in kinds.items():
            for N in (40, 80):
                x = OU.sample_loop(model.x0_hat, BETAS, N, x_T, **kw)
                err[name, N] = np.sqrt(np.mean((x - exact) ** 2) / np.mean(exact ** 2))
        ratio = {k: err[k, 40] / err[k, 80] for k in kinds}
        assert abs(err["unip2", 80] / err["dpmpp2m", 80] - 1.0) < 1e-9, (mu, s, err)
        assert ratio["unipc2"] > ratio["dpmpp2m"] + 0.1, (mu, s, ratio)
        assert ratio["unipc2"] < 4.0 and ratio["unipc3"] >= 3.0, (mu, s, ratio)
        assert err["unipc3", 80] < min(err["unipc2", 80], err["dpmpp2m", 80]), (mu, s, err)


def test_unipc_update_argument_validation_without_gpu():
    from tair_b200 import _lib, build
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    lib = _lib.lib()
    f = lib.tair_sampler_unipc_update
    # x, v, v_uncond, scale, scale_dev, x_next, x_corr, x0_hist, t, table, K, B, per_sample, stream
    ok = dict(x=16, v=1 << 20, xn=2 << 20, xc=3 << 20, h=4 << 20, t=5 << 20, tab=6 << 20)

    def call(K=2, per=4, **kw):
        a = dict(ok, **kw)
        return f(a["x"], a["v"], None, 1.0, None, a["xn"], a["xc"], a["h"], a["t"], a["tab"], K, 1, per, None)
    for name in ("x", "v", "xn", "xc", "h", "t", "tab"):
        assert call(**{name: None}) == -1 and b"NULL" in lib.tair_last_error(), name
    for K in (0, 4):
        assert call(K=K) == -1 and b"history depth" in lib.tair_last_error()
    assert call(per=6) == -1 and b"multiple of 4" in lib.tair_last_error()
    assert call(xc=ok["xc"] + 8) == -1 and b"aligned" in lib.tair_last_error()
    assert call(tab=ok["tab"] + 4) == -1 and b"aligned" in lib.tair_last_error()
    assert call(xn=ok["x"]) == -1 and b"x_next must not alias" in lib.tair_last_error()
    assert call(xn=ok["h"] + 16, per=4, K=2) == -1 and b"x_next must not alias" in lib.tair_last_error()
    assert call(xn=ok["xc"]) == -1 and b"x_next must not alias" in lib.tair_last_error()
    assert call(xc=ok["h"] + 16) == -1 and b"x_corr and x0_hist" in lib.tair_last_error()
    assert call(h=ok["v"]) == -1 and b"x_corr and x0_hist" in lib.tair_last_error()
