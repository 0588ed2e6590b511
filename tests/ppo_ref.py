"""References for ``rover_b200::ppo_gae`` (skrl 1.1.0 ``PPO._update.compute_gae``, restated in DESIGN.md section 2).

* ``skrl_gae_loop`` / ``skrl_compute_gae``: skrl's function transcribed literally in torch (any device).  The loop is split
  from the final normalisation line only so that the raw advantages can be compared too.
* ``gae_np`` / ``normalise_np``: the same loop in numpy fp32 with one rounding per operation, and the normalisation contract
  of the kernel in float64: mean_f = fl32(sum / n), std_f = fl32(sqrt(M2 / (n - 1))),
  out = fl32(fl32(a - mean_f) / fl32(std_f + 1e-8f)).
"""
from __future__ import annotations

import numpy as np
import torch


def skrl_gae_loop(rewards, dones, values, next_values, discount_factor=0.99, lambda_coefficient=0.95):
    """skrl's loop up to ``returns = advantages + values``: ``(returns, raw advantages)``."""
    advantage = 0
    advantages = torch.zeros_like(rewards)
    not_dones = dones.logical_not()
    memory_size = rewards.shape[0]
    for i in reversed(range(memory_size)):
        next_values = values[i + 1] if i < memory_size - 1 else next_values
        advantage = rewards[i] - values[i] + discount_factor * not_dones[i] * (next_values + lambda_coefficient * advantage)
        advantages[i] = advantage
    returns = advantages + values
    return returns, advantages


def skrl_compute_gae(rewards, dones, values, next_values, discount_factor=0.99, lambda_coefficient=0.95):
    returns, advantages = skrl_gae_loop(rewards, dones, values, next_values, discount_factor, lambda_coefficient)
    advantages = (advantages - advantages.mean()) / (advantages.std() + 1e-8)
    return returns, advantages


def gae_np(rewards, dones, values, next_values, discount_factor=0.99, lambda_coefficient=0.95):
    """numpy fp32, one rounding per operation: ``(returns, raw advantages)``; arrays ``[T, ...]``."""
    r = np.asarray(rewards, np.float32)
    v = np.asarray(values, np.float32)
    nd = np.logical_not(np.asarray(dones, bool)).astype(np.float32)
    last = np.asarray(next_values, np.float32).reshape(r.shape[1:])
    g, lam = np.float32(discount_factor), np.float32(lambda_coefficient)
    adv = np.zeros(r.shape[1:], np.float32)
    out = np.empty_like(r)
    with np.errstate(invalid="ignore", over="ignore"):
        for i in reversed(range(r.shape[0])):
            nv = v[i + 1] if i < r.shape[0] - 1 else last
            adv = np.float32(r[i] - v[i]) + np.float32(np.float32(g * nd[i]) * np.float32(nv + np.float32(lam * adv)))
            out[i] = adv
        returns = (out + v).astype(np.float32)
    return returns, out


def normalise_np(adv):
    """The kernel's normalisation contract: float64 mean and two-pass unbiased variance, fp32 roundings as stated."""
    a = np.asarray(adv, np.float32)
    a64 = a.astype(np.float64)
    n = a.size
    with np.errstate(invalid="ignore", divide="ignore"):
        mean64 = a64.sum() / n
        m2 = ((a64 - mean64) ** 2).sum()
        mean_f = np.float32(mean64)
        std_f = np.float32(np.sqrt(m2 / (n - 1)) if n > 1 else np.nan)
        out = np.float32(a - mean_f) / np.float32(std_f + np.float32(1e-8))
    return out.astype(np.float32), mean_f, std_f


def exact_case(T, N, seed, scale=1.0, p_done=0.1):
    """Inputs on which every sum of the normalisation is exact in float64 (and the recurrence exact in fp32) for
    gamma = lambda = 1 and T * N <= 4096: rewards in {-1, 0, 1} / 4, values in [-4, 4] in steps of 1 / 4, times a power
    of two ``scale``.  |advantage| < 2^5 with 2 fractional bits, so (a - mean)^2 and its sum over 2^12 entries fit 53 bits."""
    rng = np.random.default_rng(seed)
    r = rng.integers(-1, 2, (T, N)).astype(np.float32) * np.float32(0.25 * scale)
    v = rng.integers(-16, 17, (T, N)).astype(np.float32) * np.float32(0.25 * scale)
    last = rng.integers(-16, 17, N).astype(np.float32) * np.float32(0.25 * scale)
    d = rng.random((T, N)) < p_done
    return r, d, v, last
