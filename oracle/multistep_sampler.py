"""TEST INFRASTRUCTURE — float64 restatement of the DDIM and DPM-Solver++(2M) samplers, and an analytic model.

Written from the textbook forms, not from the product's (a, b, c, d) tables:

* DDIM (Song et al. 2021, eq. 12):  x_n = sqrt(abar_n) x0 + sqrt(1 - abar_n - s^2) eps + s z,
  eps = (x - sqrt(abar_i) x0) / sqrt(1 - abar_i),  s = eta sqrt((1 - abar_n)/(1 - abar_i)) sqrt(1 - abar_i/abar_n).
* DPM-Solver++(2M) (Lu et al. 2022, Algorithm 2):  x_n = (sigma_n/sigma_i) x - alpha_n (exp(-h) - 1) (D0 + D1/2),
  D0 = m0, D1 = (m0 - m1)/r, r = h_prev/h; first order (D1 = 0) with no history, on the final step (sigma_n = 0)
  and when h_prev is infinite.

Timesteps: ``oracle.sampler.space_timesteps(1000, N)`` visited in descending order, the final step targeting the
clean sample (abar = 1).

The analytic model: data x0 ~ N(mu, s^2) per element.  Its exact denoiser is
x0_hat = mu + alpha s^2/(alpha^2 s^2 + sigma^2) (x - alpha mu), its v-prediction v = (alpha x - x0_hat)/sigma, and the
probability-flow ODE maps a pure-noise x_T exactly to mu + s x_T.
"""
from __future__ import annotations

import numpy as np

from .sampler import space_timesteps


def schedule(betas: np.ndarray, num_steps: int):
    """-> (timesteps in visiting order, abar per step, abar of each step's target), float64."""
    abar_train = np.cumprod(1.0 - np.asarray(betas, dtype=np.float64))
    taus = np.array(space_timesteps(len(betas), num_steps)[::-1], dtype=np.int64)
    abar = abar_train[taus]
    return taus, abar, np.append(abar[1:], 1.0)


class GaussianData:
    """x0 ~ N(mu, s^2) per element: exact denoiser, v-prediction and probability-flow ODE endpoint."""

    def __init__(self, mu: float, s: float):
        self.mu, self.s = float(mu), float(s)

    def x0_hat(self, x, abar):
        alpha, sigma2 = np.sqrt(abar), 1.0 - abar
        return self.mu + alpha * self.s ** 2 / (abar * self.s ** 2 + sigma2) * (x - alpha * self.mu)

    def v(self, x, abar):
        return (np.sqrt(abar) * x - self.x0_hat(x, abar)) / np.sqrt(1.0 - abar)

    def ode_endpoint(self, x_T):
        return self.mu + self.s * x_T


def ddim_step(x, x0, abar_i, abar_n, eta=0.0, z=None):
    eps = (x - np.sqrt(abar_i) * x0) / np.sqrt(1.0 - abar_i)
    s = eta * np.sqrt((1.0 - abar_n) / (1.0 - abar_i)) * np.sqrt(1.0 - abar_i / abar_n)
    out = np.sqrt(abar_n) * x0 + np.sqrt(max(1.0 - abar_n - s * s, 0.0)) * eps
    return out + s * z if s != 0.0 else out


def _lam(abar):
    with np.errstate(divide="ignore"):
        return 0.5 * np.log(abar) - 0.5 * np.log1p(-abar) if abar < 1.0 else np.inf


def dpmpp2m_step(x, m0, abar_i, abar_n, m_prev=None, abar_prev=None):
    """One DPM-Solver++(2M) step from abar_i to abar_n; m_prev is the data prediction of the previous step at
    abar_prev (None on the first step)."""
    lam_i, lam_n = _lam(abar_i), _lam(abar_n)
    h = lam_n - lam_i
    sig_i, sig_n, alpha_n = np.sqrt(1.0 - abar_i), np.sqrt(1.0 - abar_n), np.sqrt(abar_n)
    D = m0
    if m_prev is not None and sig_n != 0.0:
        h_prev = lam_i - _lam(abar_prev)
        if np.isfinite(h_prev):
            r = h_prev / h
            D = m0 + 0.5 * ((m0 - m_prev) / r)
    return (sig_n / sig_i) * x - alpha_n * np.expm1(-h) * D


def sample_loop(x0_fn, betas, num_steps, x_T, kind="dpmpp2m", eta=0.0, noises=None, trace=None):
    """x0_fn(x, abar) -> x0_hat.  kind: 'ddim' or 'dpmpp2m'.  ``noises[i]`` is the z of DDIM step i (eta > 0).
    ``trace`` (a list) receives the latent after every step."""
    _, abar, abar_next = schedule(betas, num_steps)
    x = np.asarray(x_T, dtype=np.float64)
    m_prev = None
    for i in range(num_steps):
        m0 = x0_fn(x, abar[i])
        if kind == "ddim":
            x = ddim_step(x, m0, abar[i], abar_next[i], eta, None if noises is None else noises[i])
        else:
            x = dpmpp2m_step(x, m0, abar[i], abar_next[i], m_prev, abar[i - 1] if i else None)
            m_prev = m0
        if trace is not None:
            trace.append(x)
    return x
