"""TEST INFRASTRUCTURE — float64 restatement of the UniPC sampler (bh2, data prediction, multistep).

Written from the paper's algorithm (Zhao et al., NeurIPS 2023, "UniPC: A Unified Predictor-Corrector Framework for Fast
Sampling of Diffusion Models", UniP-p / UniC-p with B(h) = e^h - 1 and h -> -h for data prediction), not from the
product's packed table: every step forms the D1 differences of the data predictions and solves R rho = b explicitly.

With s0 the newest point of the history, t the target, h = lambda_t - lambda_s0, hh = -h, B = expm1(hh)::

    r_k  = (lambda_{s0-k} - lambda_s0)/h,   D1_k = (m_{s0-k} - m_s0)/r_k,   k = 1 .. p-1
    R_jk = r_k^j,   b_j = j! hh phi_{j+1}(hh)/B,   phi_j(z) = (e^z - sum_{k<j} z^k/k!)/z^j
    UniP-p:  x_t  = (sigma_t/sigma_s0) x_s0 - alpha_t expm1(hh) m_s0 - alpha_t B sum_k rho_k D1_k
             rho solves the (p-1) x (p-1) system; rho = 1/2 at p = 2
    UniC-p:  xc_t = (sigma_t/sigma_s0) xc_s0 - alpha_t expm1(hh) m_s0
                    - alpha_t B (sum_k rho_k D1_k + rho_p (m_t - m_s0))
             rho solves the p x p system with r_p = 1 appended; rho = 1/2 at p = 1

Step i evaluates the model at x_i (the previous predictor output), corrects x_i with the order of the predictor that
produced it (i >= 1, if enabled), then predicts x_{i+1} at order min(order, i + 1, N - i, 1 + #history points with
finite lambda).  Timesteps, the clean-sample target of the last step and the analytic ``GaussianData`` model are those
of ``oracle/multistep_sampler.py``.
"""
from __future__ import annotations

import math

import numpy as np

from . import multistep_sampler as OM
from .multistep_sampler import GaussianData, schedule  # noqa: F401


def _phi(j: int, z: float) -> float:
    return (math.expm1(z) - sum(z ** k / math.factorial(k) for k in range(1, j))) / z ** j


def _b(hh: float, n: int) -> np.ndarray:
    B = math.expm1(hh)
    return np.array([math.factorial(j) * hh * _phi(j + 1, hh) / B for j in range(1, n + 1)])


def _solve(r, hh):
    R = np.array([[rk ** j for rk in r] for j in range(len(r))])
    return np.linalg.solve(R, _b(hh, len(r)))


def unip_update(x_s0, ms, lams, lam_t, alpha_t, sigma_t, sigma_s0, p):
    """UniP-p from s0 = the last entry of ``ms`` / ``lams`` (data predictions, lambdas; oldest first) to t."""
    h = lam_t - lams[-1]
    hh = -h
    x_t = (sigma_t / sigma_s0) * x_s0 - alpha_t * math.expm1(hh) * ms[-1]
    if p == 1:
        return x_t
    r = [(lams[-1 - k] - lams[-1]) / h for k in range(1, p)]
    D1 = [(ms[-1 - k] - ms[-1]) / r[k - 1] for k in range(1, p)]
    rho = np.array([0.5]) if p == 2 else _solve(r, hh)
    return x_t - alpha_t * math.expm1(hh) * sum(rk * d for rk, d in zip(rho, D1))


def unic_update(xc_s0, m_t, ms, lams, lam_t, alpha_t, sigma_t, sigma_s0, p):
    """UniC-p: the corrected latent at t from the corrected latent at s0 and the new data prediction m_t."""
    h = lam_t - lams[-1]
    hh = -h
    r = [(lams[-1 - k] - lams[-1]) / h for k in range(1, p)]
    D1 = [(ms[-1 - k] - ms[-1]) / r[k - 1] for k in range(1, p)]
    rho = np.array([0.5]) if p == 1 else _solve(r + [1.0], hh)
    res = sum(rk * d for rk, d in zip(rho[:-1], D1)) + rho[-1] * (m_t - ms[-1])
    return (sigma_t / sigma_s0) * xc_s0 - alpha_t * math.expm1(hh) * ms[-1] - alpha_t * math.expm1(hh) * res


def unipc_step(x, xc_prev, m, ms, lams, abar_i, abar_prev, abar_next, order, prev_order, step, num_steps,
               corrector=True):
    """One step i: correct x_i (given m_i = ``m`` and the history ``ms`` / ``lams`` of steps < i), then predict.
    Appends m_i and lambda_i to the history and returns (x_{i+1}, xc_i, predictor order)."""
    lam_i = OM._lam(abar_i)
    sig_i, al_n, sig_n = math.sqrt(1.0 - abar_i), math.sqrt(abar_next), math.sqrt(1.0 - abar_next)
    if corrector and step >= 1:
        xc = unic_update(xc_prev, m, ms, lams, lam_i, math.sqrt(abar_i), sig_i, math.sqrt(1.0 - abar_prev), prev_order)
    else:
        xc = x
    ms.append(m)
    lams.append(lam_i)
    p = min(order, step + 1, num_steps - step, 1 + sum(1 for lam in lams[:-1] if np.isfinite(lam)))
    return unip_update(xc, ms, lams, OM._lam(abar_next), al_n, sig_n, sig_i, p), xc, p


def sample_loop(x0_fn, betas, num_steps, x_T, kind="unipc", order=2, corrector=True, trace=None, **kw):
    """x0_fn(x, abar) -> x0_hat.  kind 'unipc' here; 'ddim' / 'dpmpp2m' go to ``oracle.multistep_sampler``.
    ``trace`` (a list) receives the latent after every step (the predictor output; x0_hat(tau=0) after the last)."""
    if kind != "unipc":
        return OM.sample_loop(x0_fn, betas, num_steps, x_T, kind, trace=trace, **kw)
    _, abar, abar_next = schedule(betas, num_steps)
    x = np.asarray(x_T, dtype=np.float64)
    xc, ms, lams, p = None, [], [], None
    for i in range(num_steps):
        m = x0_fn(x, abar[i])
        x, xc, p = unipc_step(x, xc, m, ms, lams, abar[i], abar[i - 1] if i else None, abar_next[i], order, p, i,
                              num_steps, corrector)
        if trace is not None:
            trace.append(x)
    return x
