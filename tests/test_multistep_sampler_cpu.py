"""DDIM and DPM-Solver++(2M) without a GPU: the product's float64 host tables against the float64 textbook restatement
(oracle/multistep_sampler.py) on an analytic Gaussian model, table identities, and argument validation of the fused
update's C entry point."""
import os

import numpy as np
import pytest

from oracle import multistep_sampler as OM, sampler as OS
from tair_b200.sampler import DDIMSampler, DPMSolverSampler, SpacedSampler
from tair_b200.sampler.multistep_sampler import dpm_solver_2m_coefficients, schedule_points

BETAS = OS.diffusion_betas()          # zero terminal SNR, as the val config
KINDS = {"ddim": DDIMSampler, "dpmpp2m": DPMSolverSampler}


def apply_tables(tabs, model, x_T, noises=None):
    """The product's update in float64: row t = N-1-i at step i, x0 = P x - Q v, x_next = b x0 + a x + c hist + d z."""
    N = len(tabs["timesteps"])
    abar_train = np.cumprod(1.0 - BETAS)
    x, hist, out = x_T.copy(), np.zeros_like(x_T), []
    for i, tau in enumerate(tabs["timesteps"][::-1]):
        r = N - 1 - i
        v = model.v(x, abar_train[tau])
        x0 = tabs["ms_P"][r] * x - tabs["ms_Q"][r] * v
        z = np.zeros_like(x) if noises is None else noises[i]
        x = ((tabs["ms_b"][r] * x0 + tabs["ms_a"][r] * x) + tabs["ms_c"][r] * hist) + tabs["ms_d"][r] * z
        hist = x0
        out.append(x)
    return out


@pytest.mark.parametrize("kind", ["ddim", "dpmpp2m"])
@pytest.mark.parametrize("N", [5, 20, 50])
def test_host_tables_match_textbook_oracle(kind, N):
    model = OM.GaussianData(0.3, 0.7)
    x_T = np.random.default_rng(N).standard_normal(4096)
    got = apply_tables(KINDS[kind](BETAS).host_tables(N), model, x_T)
    ref = []
    OM.sample_loop(model.x0_hat, BETAS, N, x_T, kind, trace=ref)
    assert len(got) == len(ref) == N
    for i, (g, r) in enumerate(zip(got, ref)):
        err = np.abs(g - r).max() / np.abs(r).max()
        assert err < 1e-12, (i, err)


@pytest.mark.parametrize("N", [5, 20])
def test_stochastic_ddim_tables_match_textbook_oracle(N):
    model = OM.GaussianData(0.0, 1.0)
    rng = np.random.default_rng(100 + N)
    x_T = rng.standard_normal(4096)
    noises = [rng.standard_normal(4096) for _ in range(N)]
    got = apply_tables(DDIMSampler(BETAS, eta=1.0).host_tables(N), model, x_T, noises)
    ref = []
    OM.sample_loop(model.x0_hat, BETAS, N, x_T, "ddim", eta=1.0, noises=noises, trace=ref)
    # the textbook form takes sqrt(1 - abar_n - s^2) of a difference that is exactly 0 on the first step under zero
    # terminal SNR: its rounding residue enters as sqrt(1e-16) ~ 1e-8
    for i, (g, r) in enumerate(zip(got, ref)):
        assert np.abs(g - r).max() / np.abs(r).max() < 1e-7, i


@pytest.mark.parametrize("N", [1, 2, 3, 10, 20, 25, 50, 100])
def test_tables_are_finite_and_follow_the_spaced_timesteps(N):
    spaced = SpacedSampler(BETAS)
    spaced.make_schedule(N)
    for s in (DDIMSampler(BETAS), DDIMSampler(BETAS, eta=1.0), DPMSolverSampler(BETAS)):
        tabs = s.host_tables(N)
        assert np.array_equal(tabs["timesteps"], spaced.timesteps)
        for k in ("ms_P", "ms_Q", "ms_a", "ms_b", "ms_c", "ms_d"):
            assert tabs[k].shape == (N,) and np.isfinite(tabs[k]).all(), k
        # the last step (row 0) returns x0_hat(tau=0): a = c = d = 0, b = 1
        assert (tabs["ms_a"][0], tabs["ms_b"][0], tabs["ms_c"][0], tabs["ms_d"][0]) == (0.0, 1.0, 0.0, 0.0)
        s.make_schedule(N)
        assert np.array_equal(s.timesteps, spaced.timesteps)
        assert s.ms_b.dtype.is_floating_point and s.ms_b.numpy().tolist() == tabs["ms_b"].astype(np.float32).tolist()


@pytest.mark.parametrize("N", [3, 20, 50])
def test_ddim_eta0_equals_first_order_dpm_solver(N):
    ddim = DDIMSampler(BETAS).host_tables(N)
    _, alpha, sigma = schedule_points(np.cumprod(1.0 - BETAS), N)
    first = [np.ascontiguousarray(v[::-1]) for v in dpm_solver_2m_coefficients(alpha, sigma, second_order=False)]
    for k, ref in zip(("ms_a", "ms_b", "ms_c", "ms_d"), first):
        assert np.allclose(ddim[k], ref, rtol=1e-12, atol=0.0), k


def test_second_order_starts_on_the_third_step_under_zero_snr():
    tabs = DPMSolverSampler(BETAS).host_tables(20)
    c = tabs["ms_c"][::-1]                          # visiting order
    assert c[0] == 0.0 and c[1] == 0.0 and c[-1] == 0.0
    assert (c[2:-1] != 0.0).all()


def test_eta_changes_a_b_d_only():
    t0, t1 = DDIMSampler(BETAS).host_tables(20), DDIMSampler(BETAS, eta=1.0).host_tables(20)
    assert not (t0["ms_d"] != 0).any() and (t1["ms_d"][1:] > 0).all()
    assert (t1["ms_a"][1:] != t0["ms_a"][1:]).all() and (t1["ms_b"][1:-1] != t0["ms_b"][1:-1]).all()   # step 0 (last row) has alpha_i = 0: b = alpha_n for any eta
    assert not t1["ms_c"].any() and np.array_equal(t0["ms_P"], t1["ms_P"]) and np.array_equal(t0["ms_Q"], t1["ms_Q"])


def test_eps_parameterisation_needs_nonzero_terminal_snr():
    for cls in (DDIMSampler, DPMSolverSampler):
        with pytest.raises(ValueError):
            cls(BETAS, "eps").make_schedule(20)
        tabs = cls(OS.diffusion_betas(zero_snr=False), "eps").host_tables(20)
        assert all(np.isfinite(v).all() for v in tabs.values())


def test_analytic_convergence_orders():
    """Relative RMS error of the endpoint against the exact probability-flow ODE solution mu + s x_T, 100 000 samples,
    float64 oracle loop.  Values when this test was written:

      | (mu, s)    | sampler | N=10    | 20      | 40      | 50      | 80      |
      |------------|---------|---------|---------|---------|---------|---------|
      | (0.0, 2.0) | DDIM    | 1.31e-1 | 6.49e-2 | 3.24e-2 | 2.59e-2 | 1.63e-2 |
      | (0.0, 2.0) | DPM++2M | 4.69e-2 | 1.42e-2 | 4.66e-3 | 3.27e-3 | 1.52e-3 |
      | (0.5, 1.0) | DDIM    | 1.32e-1 | 6.68e-2 | 3.42e-2 | 2.74e-2 | 1.76e-2 |
      | (0.5, 1.0) | DPM++2M | 1.48e-1 | 5.65e-2 | 1.95e-2 | 1.37e-2 | 6.37e-3 |
      | (0.3, 0.5) | DDIM    | 2.00e-1 | 1.08e-1 | 5.82e-2 | 4.72e-2 | 3.12e-2 |
      | (0.3, 0.5) | DPM++2M | 1.90e-1 | 1.21e-1 | 5.45e-2 | 4.03e-2 | 2.02e-2 |

    The test asserts the orders: DDIM is first order (error halves when N doubles), DPM-Solver++(2M) falls faster and is
    below DDIM from N = 40 on."""
    x_T = np.random.default_rng(0).standard_normal(100_000)
    for mu, s in ((0.0, 2.0), (0.5, 1.0), (0.3, 0.5)):
        model = OM.GaussianData(mu, s)
        exact = model.ode_endpoint(x_T)
        err = {}
        for kind in ("ddim", "dpmpp2m"):
            for N in (20, 40, 80):
                x = OM.sample_loop(model.x0_hat, BETAS, N, x_T, kind)
                err[kind, N] = np.sqrt(np.mean((x - exact) ** 2) / np.mean(exact ** 2))
        for a, b in ((20, 40), (40, 80)):
            assert 1.8 <= err["ddim", a] / err["ddim", b] <= 2.1, (mu, s, a, err)
        assert err["dpmpp2m", 40] / err["dpmpp2m", 80] >= 2.5, (mu, s, err)
        for N in (40, 80):
            assert err["dpmpp2m", N] < err["ddim", N], (mu, s, N, err)


def test_multistep_update_argument_validation_without_gpu():
    from tair_b200 import _lib, build
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    lib = _lib.lib()
    f = lib.tair_sampler_multistep_update
    tabs = [16] * 6
    rc = f(None, 16, None, 1.0, None, 16, 32, None, 16, *tabs, 1, 4, None)
    assert rc == -1 and b"NULL" in lib.tair_last_error()
    rc = f(16, 16, None, 1.0, None, 16, 32, None, 16, 16, None, 16, 16, 16, 16, 1, 4, None)
    assert rc == -1 and b"NULL" in lib.tair_last_error()
    rc = f(16, 16, None, 1.0, None, 16, 32, None, 16, *tabs, 1, 6, None)
    assert rc == -1 and b"multiple of 4" in lib.tair_last_error()
    rc = f(16, 16, None, 1.0, None, 16, 40, 8, 16, *tabs, 1, 4, None)
    assert rc == -1 and b"aligned" in lib.tair_last_error()
    rc = f(16, 16, None, 1.0, None, 16, 16, None, 16, *tabs, 1, 4, None)
    assert rc == -1 and b"alias" in lib.tair_last_error()
