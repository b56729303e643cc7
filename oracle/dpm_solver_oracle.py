"""
ORACLE — TEST INFRASTRUCTURE ONLY.  Not product code.

A plain numpy restatement of the DPM-Solver++(2M) sampler, an addition beyond the reference (which samples with DDPM /
DDIM only): Lu et al., "DPM-Solver++: Fast Solver for Guided Sampling of Diffusion Probabilistic Models" (2022),
Algorithm 2 (multistep, second order, data prediction).  It runs on the schedule tables, the denoiser and the x0
post-processing of `musediff_oracle` (rounding to the nearest embedding, then clip, as the DDIM loop forms it).  Only
`tests/` imports this module; the product package never does.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np

import musediff_oracle as O

F32 = np.float32


def _log_snr(s: O.Schedule) -> np.ndarray:
    """lambda_i = log alpha_i - log sigma_i, alpha_i = sqrt(abar_i), sigma_i = sqrt(1 - abar_i)."""
    ab = np.asarray(s.alphas_cumprod, dtype=np.float64)
    return 0.5 * np.log(ab) - 0.5 * np.log1p(-ab)


def dpm_solver_indices(s: O.Schedule, t_start: int, steps: int) -> List[int]:
    """Evaluation indices, uniform in lambda (Lu et al. 2022, Sec. 3: time steps uniform in lambda), rounded to the table and
    kept distinct: s_0 = t_start, s_k = clip(round(g_k), N-1-k, s_{k-1}-1), g_k the fractional index whose interpolated
    lambda is the k-th of N evenly spaced values from lambda[t_start] to lambda[0]."""
    T = s.num_timesteps
    if not (0 <= t_start < T) or not (1 <= steps <= t_start + 1):
        raise ValueError("need 0 <= t_start < %d and 1 <= steps <= t_start + 1 (t_start=%r, steps=%r)" % (T, t_start, steps))
    lam = _log_snr(s)
    lam_inc, idx_inc = lam[t_start::-1], np.arange(t_start, -1, -1, dtype=np.float64)   # lambda increasing
    targets = np.linspace(lam[t_start], lam[0], steps)
    out = [int(t_start)]
    for k in range(1, steps):
        g = np.interp(targets[k], lam_inc, idx_inc)
        out.append(int(min(max(np.rint(g), steps - 1 - k), out[-1] - 1)))
    return out


def dpm_solver_coefficients(s: O.Schedule, indices: Sequence[int], order: int = 2) -> np.ndarray:
    """float64 [N, 4] = (a, b, c0, c1) per evaluation: x_{k+1} = a x_k + b (c0 x0_k + c1 x0_{k-1}).
    Algorithm 2 (data prediction): with h = lambda_{s_{k+1}} - lambda_{s_k},
    x_{k+1} = sigma_{k+1}/sigma_k x_k - alpha_{k+1} (e^{-h} - 1) D_k, D_0 = x0_0, and for k >= 1 with r = h_{k-1} / h:
    D_k = (1 + 1/(2r)) x0_k - 1/(2r) x0_{k-1}.  order 1 keeps D_k = x0_k (DDIM at eta = 0).  The last evaluation returns its
    x0: row (0, 1, 1, 0)."""
    if order not in (1, 2):
        raise ValueError("order must be 1 or 2")
    ab = np.asarray(s.alphas_cumprod, dtype=np.float64)
    lam = _log_snr(s)
    alpha, sigma = np.sqrt(ab), np.sqrt(1.0 - ab)
    N = len(indices)
    coef = np.zeros((N, 4), dtype=np.float64)
    coef[N - 1] = (0.0, 1.0, 1.0, 0.0)
    for k in range(N - 1):
        cur, nxt = indices[k], indices[k + 1]
        h = lam[nxt] - lam[cur]
        coef[k, 0] = sigma[nxt] / sigma[cur]
        coef[k, 1] = -alpha[nxt] * np.expm1(-h)
        if order == 2 and k > 0:
            r = (lam[cur] - lam[indices[k - 1]]) / h
            coef[k, 2], coef[k, 3] = 1.0 + 1.0 / (2.0 * r), -1.0 / (2.0 * r)
        else:
            coef[k, 2], coef[k, 3] = 1.0, 0.0
    return coef


def dpm_solver_sample_loop(s: O.Schedule, p: Dict[str, np.ndarray], x_noised: np.ndarray, steps: int, t_start: int,
                           order: int = 2, clip_denoised=True, round_to_emb=True, mask=None, x_start=None,
                           record: Optional[list] = None, model_fn=None) -> np.ndarray:
    """DPM-Solver++(2M) from x_noised at t_start in `steps` evaluations; x0 processed as in O.ddim_sample_loop (rounded,
    then clipped), coefficients cast to float32 once, the update in float32.  Returns the last x0.  `record` receives
    {"t", "x_t", "model_output", "sample"} per evaluation, as the oracle loops record them."""
    idx = dpm_solver_indices(s, t_start, steps)
    coef = dpm_solver_coefficients(s, idx, order).astype(F32)
    E = p["word_embedding.weight"]
    x = x_noised.astype(F32)
    B = x.shape[0]
    prev = None
    for k, i in enumerate(idx):
        t = np.full((B,), i, dtype=np.int64)
        mo = (model_fn or O.denoiser_forward)(p, x, s.model_timestep(t))
        x0 = O.predict_xstart(s, mo, x, t, E if round_to_emb else None, clip_denoised)
        a, b, c0, c1 = coef[k]
        d = c0 * x0 + c1 * prev if c1 != 0 else c0 * x0
        sample = (a * x + b * d) if a != 0 else b * d
        if mask is not None:
            sample = np.where(mask == 0, x_start, sample)
        if record is not None:
            record.append({"t": i, "x_t": x, "model_output": mo, "sample": sample.astype(F32)})
        x, prev = sample.astype(F32), x0
    return x
