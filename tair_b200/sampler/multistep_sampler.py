"""DDIM and DPM-Solver++(2M) samplers on the fused multistep update (``tair_sampler_multistep_update``).

Both reuse the loops of ``SpacedSampler`` (``sample``, ``val_sample`` with text-spotting feedback, CUDA-graph replay,
``rescale_cfg`` with a device guidance scale, ``noise_fn``, ``trace``) and differ from it only in the schedule tables
and the per-step update.  They visit the same ``space_timesteps(1000, N)`` set in descending order
tau_0 = 999 > ... > tau_{N-1} = 0 with one network evaluation per step.  This "trailing" spacing starts from pure noise
under the zero-terminal-SNR schedule; LDM's leading spacing (1 ... 981) never does.

Every step is one kernel::

    x0     = P[t] x - Q[t] v                       v: P = alpha_i, Q = sigma_i;  eps: P = 1/alpha_i, Q = sqrt(1/abar - 1)
    x_next = ((b[t] x0 + a[t] x) + c[t] x0_hist) + d[t] noise,   x0_hist <- x0

with alpha_i = sqrt(abar(tau_i)), sigma_i = sqrt(1 - abar(tau_i)), lambda_i = log alpha_i - log sigma_i.  The target of
step i is (alpha_n, sigma_n) = step i+1, or the clean sample (alpha = 1, sigma = 0, lambda = +inf) after the last step;
h = lambda_n - lambda_i.

* DDIM(eta):  s = eta sqrt(sigma_n^2/sigma_i^2 (1 - alpha_i^2/alpha_n^2)), a = sqrt(sigma_n^2 - s^2)/sigma_i,
  b = alpha_n - a alpha_i, c = 0, d = s.
* DPM-Solver++(2M), data prediction:  a = sigma_n/sigma_i, b0 = alpha_n (1 - exp(-h)), k = h / (2 h_prev) with
  h_prev = lambda_i - lambda_{i-1};  b = b0 (1 + k), c = -b0 k, d = 0.  k = 0 on the first step, on the last step
  (sigma_n = 0) and wherever h_prev is infinite.

Consequences:

* DPM-Solver++ at first order (k = 0) is DDIM(eta=0) algebraically; the two tables differ only by float64 rounding.
* Every sampler's last step returns x0_hat(tau=0), as the spaced sampler does.
* Under zero terminal SNR lambda_0 = -inf, so h_prev is infinite on step 1 and the first two steps of 2M are first order.
* Karras sigma spacing is not offered: sigma_max is infinite under zero terminal SNR.

The tables are built in float64 and cast to fp32 once.  For DDIM(eta=0) and DPM-Solver++ d is all zeros: the loops
still draw the step noise, and 0 * z adds +0, so the result does not depend on it.
"""
from __future__ import annotations

from typing import Dict, Tuple

import numpy as np
import torch

from .. import ops
from .spaced_sampler import SpacedSampler, space_timesteps

_MS_TABLES = ("ms_P", "ms_Q", "ms_a", "ms_b", "ms_c", "ms_d")


def schedule_points(alphas_cumprod: np.ndarray, num_steps: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """-> (timesteps in visiting order, alpha, sigma), float64.  alpha and sigma have num_steps + 1 entries: the last is
    the clean-sample target (1, 0) of the final step."""
    taus = np.array(sorted(space_timesteps(len(alphas_cumprod), str(num_steps)), reverse=True), dtype=np.int64)
    abar = alphas_cumprod[taus].astype(np.float64)
    alpha = np.append(np.sqrt(abar), 1.0)
    sigma = np.append(np.sqrt(1.0 - abar), 0.0)
    return taus, alpha, sigma


def _lambda(alpha: np.ndarray, sigma: np.ndarray) -> np.ndarray:
    with np.errstate(divide="ignore"):
        return np.log(alpha) - np.log(sigma)


def ddim_coefficients(alpha: np.ndarray, sigma: np.ndarray, eta: float = 0.0):
    """(a, b, c, d) per step, in visiting order, of DDIM(eta) for the points of ``schedule_points``."""
    ai, si, an, sn = alpha[:-1], sigma[:-1], alpha[1:], sigma[1:]
    s = eta * np.sqrt(sn ** 2 / si ** 2 * (1.0 - ai ** 2 / an ** 2))
    # sqrt(sn^2 - s^2)/si rewritten without the cancellation: at eta = 1 and alpha_i = 0 (the first step under zero
    # terminal SNR) sn^2 - s^2 is exactly 0, and the difference could round to a negative number
    a = sn / si * np.sqrt((1.0 - eta ** 2) + eta ** 2 * (sn * ai / (si * an)) ** 2)
    b = an - a * ai
    return a, b, np.zeros_like(a), s


def dpm_solver_2m_coefficients(alpha: np.ndarray, sigma: np.ndarray, second_order: bool = True):
    """(a, b, c, d) per step, in visiting order, of DPM-Solver++(2M) with data prediction.  ``second_order=False``
    forces k = 0 everywhere (DPM-Solver++ first order)."""
    lam = _lambda(alpha, sigma)
    ai, si, an, sn = alpha[:-1], sigma[:-1], alpha[1:], sigma[1:]
    with np.errstate(invalid="ignore"):
        h = lam[1:] - lam[:-1]
    e = np.exp(-h)                                    # 0 where h = +inf
    a = sn / si
    b0 = an * (1.0 - e)
    k = np.zeros_like(a)
    if second_order:
        for i in range(1, len(a)):
            h_prev = h[i - 1]
            if sn[i] != 0.0 and np.isfinite(h_prev):
                k[i] = h[i] / (2.0 * h_prev)
    return a, b0 * (1.0 + k), -b0 * k, np.zeros_like(a)


class _MultistepSampler(SpacedSampler):
    """Shared part of the DDIM and DPM-Solver++ samplers: float64 host tables and the x0 history buffer."""

    def __init__(self, betas: np.ndarray, parameterization: str = "v", rescale_cfg: bool = False):
        super().__init__(betas, parameterization, rescale_cfg)
        # one history buffer per (device, x.shape), kept at a stable address: captured step graphs read and write it
        self._x0_hist: Dict[tuple, torch.Tensor] = {}

    def _coefficients(self, alpha: np.ndarray, sigma: np.ndarray):
        raise NotImplementedError

    def host_tables(self, num_steps: int) -> Dict[str, np.ndarray]:
        """float64 tables before the fp32 cast.  Row r belongs to step N-1-r (the loops pass t = N-1-i at step i);
        ``timesteps`` are ascending, as in ``SpacedSampler``."""
        taus, alpha, sigma = schedule_points(self.training_alphas_cumprod, num_steps)
        if self.parameterization == "v":
            P, Q = alpha[:-1], sigma[:-1]
        else:
            abar = alpha[:-1] ** 2
            with np.errstate(divide="ignore"):
                P, Q = 1.0 / alpha[:-1], np.sqrt(1.0 / abar - 1.0)
        steps = dict(zip(_MS_TABLES, (P, Q) + tuple(self._coefficients(alpha, sigma))))
        bad = [k for k, v in steps.items() if not np.isfinite(v).all()]
        if bad:
            raise ValueError(f"{type(self).__name__}: non-finite schedule tables {bad} for {num_steps} steps with "
                             f"{self.parameterization!r} parameterisation (eps-prediction is undefined at zero terminal SNR)")
        out = {k: v[::-1].copy() for k, v in steps.items()}
        out["timesteps"] = taus[::-1].astype(np.int32)
        return out

    def make_schedule(self, num_steps: int) -> None:
        tabs = self.host_tables(num_steps)
        self.timesteps = tabs.pop("timesteps")
        for k, v in tabs.items():
            self.register(k, v)

    def _tables(self):
        return [getattr(self, n) for n in _MS_TABLES]

    def x0_history(self, x: torch.Tensor) -> torch.Tensor:
        """The x0 history buffer that the update for latents shaped like ``x`` reads and overwrites."""
        key = (x.device, tuple(x.shape))
        buf = self._x0_hist.get(key)
        if buf is None:
            buf = self._x0_hist[key] = torch.zeros(x.shape, device=x.device, dtype=torch.float32)
        return buf

    @torch.no_grad()
    def p_sample(self, model, x, model_t, t, cond, uncond, cfg_scale, noise=None, cfg_scale_dev=None):
        """One step: network evaluation(s), then the fused multistep update (which also stores this step's x0)."""
        v, v_u, feats = self.apply_model(model, x, model_t, cond, uncond, cfg_scale)
        if noise is None:
            noise = torch.randn_like(x)
        x_next = ops.sampler_multistep_update(x.contiguous(), v.contiguous(), noise.contiguous(), t, self._tables(),
                                              x0_hist=self.x0_history(x), v_uncond=v_u, cfg_scale=float(cfg_scale),
                                              cfg_scale_dev=cfg_scale_dev)
        return x_next, feats


class DDIMSampler(_MultistepSampler):
    """DDIM(eta) on the trailing timesteps; eta = 0 is deterministic, eta = 1 matches the ancestral step's variance."""

    def __init__(self, betas: np.ndarray, parameterization: str = "v", rescale_cfg: bool = False, eta: float = 0.0):
        super().__init__(betas, parameterization, rescale_cfg)
        self.eta = float(eta)

    def _coefficients(self, alpha, sigma):
        return ddim_coefficients(alpha, sigma, self.eta)


class DPMSolverSampler(_MultistepSampler):
    """DPM-Solver++(2M): second-order multistep solver of the probability-flow ODE in data prediction."""

    def _coefficients(self, alpha, sigma):
        return dpm_solver_2m_coefficients(alpha, sigma)
