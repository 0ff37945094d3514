"""UniPC predictor-corrector sampler on the fused update (``tair_sampler_unipc_update``).

UniPC (Zhao et al., NeurIPS 2023) in data prediction with B(h) = e^{-h} - 1 ("bh2"), multistep.  Like the DDIM and
DPM-Solver++ samplers it reuses the loops of ``SpacedSampler`` (``sample``, ``val_sample`` with text-spotting feedback,
CUDA-graph replay, ``rescale_cfg`` with a device guidance scale, ``trace``) and visits ``space_timesteps(1000, N)`` in
descending order, one network evaluation per step.  Points j = 0 .. N are the visited timesteps plus the clean-sample
target (alpha = 1, sigma = 0) of the last step; lambda_j = log alpha_j - log sigma_j, m_j = x0_hat at point j.

Step i (network evaluated at x_i, the predictor output of step i-1) is one kernel:

* UniC, i >= 1: correct x_i with m_i, using the order q of the predictor that produced x_i (s0 = i-1, t = i)::

      xc_i = (sigma_i/sigma_{i-1}) xc_{i-1} - alpha_i phi1 m_{i-1}
             - alpha_i B (sum_{k<q} rho_k D1_k + rho_q (m_i - m_{i-1}))

  On step 0, or with ``corrector=False``, xc_0 = x_0 (u = 1, every other corrector coefficient 0).
* UniP of order p (s0 = i, t = i+1)::

      x_{i+1} = (sigma_{i+1}/sigma_i) xc_i - alpha_{i+1} phi1 m_i - alpha_{i+1} B sum_{k<p} rho_k D1_k

with h = lambda_t - lambda_s0, hh = -h, phi1 = B = expm1(hh), r_k = (lambda_{s0-k} - lambda_s0)/h,
D1_k = (m_{s0-k} - m_s0)/r_k, and rho from R rho = b with R_jk = r_k^j (r_p = 1 appended for the corrector) and
b_j = j! hh phi_{j+1}(hh)/B.  The predictor's rho is 1/2 at order 2 (UniP-2 is then DPM-Solver++(2M) exactly), and the
order-1 corrector's rho is 1/2, as in the authors' implementation.

The predictor order of step i is min(order, 1 + i, N - i, 1 + #{j < i : lambda_j finite}): a warm-up, lower order on
the final steps, and no history point with lambda = -inf (tau = 999 under zero terminal SNR), so no r_k is ever
infinite.  The last step targets sigma = 0 at first order and returns x0_hat(tau = 0), as every sampler here does.

Everything is collapsed into per-step coefficients on x, xc_{i-1}, m_i and the history h_k = m_{i-1-k}
(k < K = order), built in float64 and cast to fp32 once, in one packed [N, 16] table.  The loops still draw step
noise; UniPC is an ODE solver and ignores it.
"""
from __future__ import annotations

import math
from typing import Dict

import numpy as np
import torch

from .. import ops
from .multistep_sampler import _lambda, schedule_points
from .spaced_sampler import SpacedSampler

# columns of the packed table (include/tair_b200.h, tair_sampler_unipc_update)
COL_P, COL_Q, COL_U, COL_E, COL_F, COL_G, COL_A, COL_B, COL_C = 0, 1, 2, 3, 4, 5, 8, 9, 10
TABLE_WIDTH = 16


def _b_vector(hh: float, n: int) -> np.ndarray:
    """b_j = j! hh phi_{j+1}(hh) / B(hh), j = 1 .. n, B = expm1(hh), through phi_{j+1}(z) = (phi_j(z) - 1/j!)/z."""
    Bh = math.expm1(hh)
    g, out = Bh / hh - 1.0, []                       # hh phi_2(hh)
    for j in range(1, n + 1):
        out.append(g * math.factorial(j) / Bh)
        g = g / hh - 1.0 / math.factorial(j + 1)
    return np.array(out)


def _rho(rks, hh: float, corrector: bool) -> np.ndarray:
    """UniP (corrector=False, rks = r_1 .. r_{p-1}) or UniC (rks = r_1 .. r_{q-1}) weights; the corrector's last weight
    belongs to m_t - m_s0."""
    if corrector:
        if not rks:
            return np.array([0.5])
        r = np.append(np.asarray(rks, dtype=np.float64), 1.0)
    else:
        if len(rks) == 1:
            return np.array([0.5])
        r = np.asarray(rks, dtype=np.float64)
    R = np.vander(r, len(r), increasing=True).T      # R_jk = r_k^j
    return np.linalg.solve(R, _b_vector(hh, len(r)))


def predictor_orders(lam: np.ndarray, order: int) -> np.ndarray:
    """Predictor order of every step (visiting order) for the N + 1 points' lambda."""
    N = len(lam) - 1
    finite = np.cumsum(np.concatenate([[0], np.isfinite(lam[:-1])]))    # finite[i] = #{j < i: lambda_j finite}
    return np.array([min(order, 1 + i, N - i, 1 + int(finite[i])) for i in range(N)])


def unipc_coefficients(alpha: np.ndarray, sigma: np.ndarray, order: int = 2, corrector: bool = True):
    """float64 [N, 13] coefficients (u, e, f, g0..g2, a, b, c0..c2 at columns 2..12; P, Q left 0) in visiting order,
    and the predictor orders."""
    lam = _lambda(alpha, sigma)
    N = len(alpha) - 1
    orders = predictor_orders(lam, order)
    tab = np.zeros((N, TABLE_WIDTH))
    for i in range(N):
        # corrector of x_i: the predictor of step i-1 (order q) refined with m_i
        if corrector and i >= 1:
            q, s0 = int(orders[i - 1]), i - 1
            h = lam[i] - lam[s0]
            hh = -h
            phi1 = math.expm1(hh)
            rks = [(lam[s0 - k] - lam[s0]) / h for k in range(1, q)]
            rho = _rho(rks, hh, corrector=True)
            scale = alpha[i] * phi1                  # alpha_t B (bh2: B = phi1)
            tab[i, COL_E] = sigma[i] / sigma[s0]
            tab[i, COL_F] = -scale * rho[-1]
            tab[i, COL_G] = -alpha[i] * phi1 + scale * rho[-1]
            for k in range(1, q):
                tab[i, COL_G] += scale * rho[k - 1] / rks[k - 1]
                tab[i, COL_G + k] = -scale * rho[k - 1] / rks[k - 1]
        else:
            tab[i, COL_U] = 1.0
        # predictor x_i -> x_{i+1}
        p = int(orders[i])
        h = lam[i + 1] - lam[i]                      # +inf on the first zero-SNR step and on the last step (p = 1)
        hh = -h
        phi1 = math.expm1(hh)
        tab[i, COL_A] = sigma[i + 1] / sigma[i]
        tab[i, COL_B] = -alpha[i + 1] * phi1
        if p > 1:
            rks = [(lam[i - k] - lam[i]) / h for k in range(1, p)]
            rho = _rho(rks, hh, corrector=False)
            scale = alpha[i + 1] * phi1
            for k in range(1, p):
                tab[i, COL_B] += scale * rho[k - 1] / rks[k - 1]
                tab[i, COL_C + k - 1] = -scale * rho[k - 1] / rks[k - 1]
    return tab, orders


class UniPCSampler(SpacedSampler):
    """UniPC-p (bh2, data prediction) with the UniC corrector; ``corrector=False`` gives UniP-p alone."""

    def __init__(self, betas: np.ndarray, parameterization: str = "v", rescale_cfg: bool = False, order: int = 2,
                 corrector: bool = True):
        super().__init__(betas, parameterization, rescale_cfg)
        self.order, self.corrector = order, bool(corrector)
        self._check_order()
        # one (x_corr, x0_hist) pair per (device, x.shape, K), at a stable address: captured step graphs read and
        # write them
        self._state: Dict[tuple, tuple] = {}

    def _check_order(self) -> None:
        if self.order not in (1, 2, 3):
            raise ValueError(f"UniPCSampler: order must be 1, 2 or 3, got {self.order!r}")

    def host_tables(self, num_steps: int) -> Dict[str, np.ndarray]:
        """float64 tables before the fp32 cast: ``table`` [N, 16], row r for step N-1-r (the loops pass t = N-1-i at
        step i); ``orders`` the predictor order per step in visiting order; ``timesteps`` ascending, as in
        ``SpacedSampler``."""
        self._check_order()
        taus, alpha, sigma = schedule_points(self.training_alphas_cumprod, num_steps)
        tab, orders = unipc_coefficients(alpha, sigma, self.order, self.corrector)
        if self.parameterization == "v":
            tab[:, COL_P], tab[:, COL_Q] = alpha[:-1], sigma[:-1]
        else:
            with np.errstate(divide="ignore"):
                tab[:, COL_P], tab[:, COL_Q] = 1.0 / alpha[:-1], np.sqrt(1.0 / alpha[:-1] ** 2 - 1.0)
        if not np.isfinite(tab).all():
            bad = sorted({int(c) for c in np.argwhere(~np.isfinite(tab))[:, 1]})
            raise ValueError(f"UniPCSampler: non-finite schedule table columns {bad} for {num_steps} steps with "
                             f"{self.parameterization!r} parameterisation (eps-prediction is undefined at zero terminal SNR)")
        return dict(table=tab[::-1].copy(), orders=orders, timesteps=taus[::-1].astype(np.int32))

    def make_schedule(self, num_steps: int) -> None:
        tabs = self.host_tables(num_steps)
        self.timesteps = tabs["timesteps"]
        self.register("unipc_table", tabs["table"])

    def _tables(self):
        return [self.unipc_table]

    def _graph_key(self, *parts) -> tuple:
        # the history depth K = order is a kernel argument and selects the state buffers: a captured graph holds both
        return super()._graph_key(*parts) + (self.order,)

    def state_buffers(self, x: torch.Tensor):
        """(x_corr, x0_hist) that the update for latents shaped like ``x`` reads and overwrites; x0_hist is
        [K, *x.shape] with K = order (the order-q corrector reads m_{i-1} .. m_{i-q})."""
        K = self.order
        key = (x.device, tuple(x.shape), K)
        st = self._state.get(key)
        if st is None:
            st = self._state[key] = (torch.zeros(x.shape, device=x.device, dtype=torch.float32),
                                     torch.zeros((K,) + tuple(x.shape), device=x.device, dtype=torch.float32))
        return st

    @torch.no_grad()
    def p_sample(self, model, x, model_t, t, cond, uncond, cfg_scale, noise=None, cfg_scale_dev=None):
        """One step: network evaluation(s), then the fused UniPC update.  ``noise`` is accepted for the loops' sake and
        ignored."""
        v, v_u, feats = self.apply_model(model, x, model_t, cond, uncond, cfg_scale)
        x_corr, x0_hist = self.state_buffers(x)
        x_next = ops.sampler_unipc_update(x.contiguous(), v.contiguous(), t, self.unipc_table, x_corr=x_corr,
                                          x0_hist=x0_hist, v_uncond=v_u, cfg_scale=float(cfg_scale),
                                          cfg_scale_dev=cfg_scale_dev)
        return x_next, feats
