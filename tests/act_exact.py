"""An exact fp32 model of the policy's action sampling: ``normal2`` (``csrc/rng.cuh``) and ``gaussian_sample``
(``csrc/policy_common.cuh``), which ``gaussian_act_kernel`` and the ``kSample`` epilogue of ``policy_forward_ws_kernel``
run.

Contract: every operation is ONE fp32 rounding in the kernel's order (numpy float32; ``fma32`` of ``tests/scan_exact.py``
for the one ``fmaf``).  The three functions CUDA does not round correctly -- ``logf``, ``expf``, ``sincospif`` -- come
from a pluggable provider: ``DeviceMath`` evaluates them with the library's device code (``rover_policy_math``),
``Float64Math`` in float64 rounded to fp32, ``RecordedMath`` is ``Float64Math`` with the device's values at the points
of ``tests/golden/act_math.npz`` where ``logf`` is not the correctly rounded log (CPU-only tests).

* ``box_muller(w0, w1)``: ``u1 = fl((w0 >> 8) + 1) * 2^-24``, ``u2 = fl(w1 >> 8) * 2^-24``, ``r = sqrt_rn(fl(-2 logf(u1)))``,
  ``(s, c) = sincospif(fl(2 u2))``, ``(fl(r c), fl(r s))``; ``normal2`` feeds it the first two words of Philox4x32-10 with
  counter ``(env_offset + row, step_lo, step_hi, 0x80000000)`` and key ``(seed_lo, seed_hi)``.
* ``gaussian_sample``: ``ls = clamp(log_std, -20, 2)``, ``sd = expf(ls)``, ``a = clamp(fma(sd, eps, mean), -1, 1)``,
  ``d = a - m``, ``term = fl(fl(-fl(d d)) / fl(fl(2 sd) sd)) - ls - 0.9189385f`` (each step rounded),
  ``log_prob = fl(0 + term0) + term1``.  Both clamps keep NaN, as ``torch.clamp`` does.

``mut`` (a set of names, see ``MUTANTS``) plants one deliberate defect: tests/test_act_exact_cpu.py checks that each
changes at least one output bit on the fixtures tests/test_gpu_act_exact.py uses.
"""
from __future__ import annotations

import os

import numpy as np

from action_noise_ref import action_counters
from oracle import philox as PH
from scan_exact import fma32, mul_add32

F = np.float32
TWO_M24 = F(2.0 ** -24)
LOG_SQRT_2PI = F(0.91893853320467274178)
GOLDEN_MATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "act_math.npz")

MUTANTS = {
    "u1_no_plus1": "u1 = (w0 >> 8) * 2^-24, without the + 1",
    "u2_from_w2": "u2 from the third Philox word",
    "sincos_swap": "sin and cos swapped",
    "rc_fused": "r * c carried unrounded into the sample's fma",
    "log_f64": "float64 log rounded to fp32 instead of logf",
    "mul_add": "fl(fl(sd * eps) + mean) instead of fmaf(sd, eps, mean)",
    "neg_log_exp": "-logf(expf(ls)) instead of -ls in the log-prob",
    "lp_unclipped": "the log-prob of the unclipped sample",
    "ls_bound_ulp": "log_std clamped to [-20, 2 + 1 ulp]",
    "clip_bound_ulp": "the action clipped to [-1, 1 + 1 ulp]",
    "nan_drop": "fminf / fmaxf clamps: a NaN log_std becomes -20, a NaN sample -1",
}
NOISE_MUTANTS = ("u1_no_plus1", "u2_from_w2", "sincos_swap", "log_f64")


def f32(x):
    return np.asarray(x, dtype=F)


def bits_equal(a, b):
    """Same fp32 bits, or both NaN (the payload of a NaN is not part of the contract)."""
    a, b = f32(a), f32(b)
    return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


# ----------------------------------------------------------------------------------------------------------------------
# providers of logf, expf, sincospif
# ----------------------------------------------------------------------------------------------------------------------
class Float64Math:
    """float64 evaluated, rounded to fp32 (correctly rounded but for double rounding); sincospi exact at multiples of
    1/2 (IEEE 754 sinPi / cosPi: sinPi(n) = +-0 with the sign of n, cosPi(n + 1/2) = +0)."""

    name = "float64"

    def log(self, x):
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.log(f32(x).astype(np.float64)).astype(F)

    def exp(self, x):
        with np.errstate(over="ignore"):
            return np.exp(f32(x).astype(np.float64)).astype(F)

    def sincospi(self, x):
        x64 = f32(x).astype(np.float64)
        with np.errstate(invalid="ignore"):
            s, c = np.sin(np.pi * x64), np.cos(np.pi * x64)
            h = 2.0 * x64
            on = np.isfinite(h) & (h == np.floor(h))
            q = np.where(on, np.mod(h, 4.0), 0).astype(np.int64)
        s = np.where(on, np.choose(q, [np.copysign(0.0, x64), np.ones_like(x64), np.copysign(0.0, x64), -np.ones_like(x64)]), s)
        c = np.where(on, np.choose(q, [np.ones_like(x64), np.zeros_like(x64), -np.ones_like(x64), np.zeros_like(x64)]), c)
        return s.astype(F), c.astype(F)


class RecordedMath(Float64Math):
    """``Float64Math`` with the device's ``logf`` at the recorded points where it is not the correctly rounded log
    (``tests/golden/act_math.npz``, written by ``tests/golden/make_act_math.py``)."""

    name = "recorded"

    def __init__(self, path=GOLDEN_MATH):
        z = np.load(path)
        order = np.argsort(z["log_x"])
        self.log_x, self.log_y = f32(z["log_x"])[order], f32(z["log_y"])[order]

    def log(self, x):
        x = f32(x)
        y = super().log(x)
        k = np.clip(np.searchsorted(self.log_x, x), 0, len(self.log_x) - 1)
        hit = self.log_x[k] == x
        return np.where(hit, self.log_y[k], y).astype(F)


class DeviceMath:
    """``logf`` / ``expf`` / ``sincospif`` of the policy kernels (``rover_policy_math``) on a CUDA device."""

    name = "device"

    def __init__(self, device):
        self.device = device

    def _run(self, op, x):
        import torch

        from isaac_rover_orbit_b200 import _lib

        x = np.ascontiguousarray(f32(x))
        if x.size == 0:
            return (x.copy(), x.copy()) if op == 2 else x.copy()
        out = _lib.policy_math(op, torch.from_numpy(x.reshape(-1)).to(self.device))
        if op == 2:
            return tuple(o.cpu().numpy().reshape(x.shape) for o in out)
        return out.cpu().numpy().reshape(x.shape)

    def log(self, x):
        return self._run(0, x)

    def exp(self, x):
        return self._run(1, x)

    def sincospi(self, x):
        return self._run(2, x)


# ----------------------------------------------------------------------------------------------------------------------
# normal2
# ----------------------------------------------------------------------------------------------------------------------
def box_muller_parts(w0, w1, math, mut=frozenset(), w2=None):
    """``(r, s, c)`` of two Philox words (``w2``: the third word, read only by the ``u2_from_w2`` mutant)."""
    w0, w1 = np.asarray(w0, np.uint32), np.asarray(w1, np.uint32)
    k1 = (w0 >> np.uint32(8)).astype(np.int64) + (0 if "u1_no_plus1" in mut else 1)
    u1 = (k1.astype(F) * TWO_M24).astype(F)  # the int -> float conversion is exact (k1 <= 2^24)
    wu = np.asarray(w2, np.uint32) if "u2_from_w2" in mut else w1
    u2 = ((wu >> np.uint32(8)).astype(F) * TWO_M24).astype(F)
    lg = Float64Math.log(None, u1) if "log_f64" in mut else math.log(u1)
    with np.errstate(invalid="ignore"):
        r = np.sqrt((F(-2.0) * lg).astype(F)).astype(F)  # numpy's fp32 sqrt is correctly rounded (= __fsqrt_rn)
    s, c = math.sincospi((F(2.0) * u2).astype(F))
    if "sincos_swap" in mut:
        s, c = c, s
    return r, s, c


def box_muller(w0, w1, math, mut=frozenset(), w2=None):
    """``[..., 2]`` fp32: the two N(0, 1) values ``normal2`` makes of the Philox words ``w0``, ``w1``."""
    r, s, c = box_muller_parts(w0, w1, math, mut, w2)
    with np.errstate(invalid="ignore"):
        return np.stack([(r * c).astype(F), (r * s).astype(F)], axis=-1)


def philox_words(seed: int, step: int, n: int, env_offset: int = 0) -> np.ndarray:
    """``[n, 4]`` uint32: the Philox block of the action stream for rows ``env_offset .. env_offset + n - 1``."""
    return PH.philox4x32_10(action_counters(step, env_offset, n), (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))


def normal2(seed: int, step: int, n: int, math, env_offset: int = 0, mut=frozenset()) -> np.ndarray:
    w = philox_words(seed, step, n, env_offset)
    return box_muller(w[:, 0], w[:, 1], math, mut, w[:, 2])


# ----------------------------------------------------------------------------------------------------------------------
# gaussian_sample
# ----------------------------------------------------------------------------------------------------------------------
def clamp(x, lo, hi, mut=frozenset()):
    x = f32(x)
    if "nan_drop" in mut:
        return np.fmin(np.fmax(x, F(lo)), F(hi)).astype(F)  # fmaxf / fminf: the non-NaN operand wins
    return np.minimum(np.maximum(x, F(lo)), F(hi)).astype(F)


def gaussian_sample(mean, log_std, eps, math, mut=frozenset(), rc=None):
    """``(actions [N, 2], log_prob [N])``; ``log_std`` [2] (one pair per launch, as the kernels read it) or [N, 2].
    ``rc = (r, s, c)`` of the noise: the ``rc_fused`` mutant needs the unrounded products."""
    mean, eps = f32(mean), f32(eps)
    log_std = np.broadcast_to(f32(log_std), mean.shape)
    hi_ls = np.nextafter(F(2), F(3)) if "ls_bound_ulp" in mut else F(2)
    hi_a = np.nextafter(F(1), F(2)) if "clip_bound_ulp" in mut else F(1)
    ls = clamp(log_std, -20.0, hi_ls, mut)
    sd = math.exp(ls)
    with np.errstate(invalid="ignore", over="ignore"):
        if "mul_add" in mut:
            x = mul_add32(sd, eps, mean)
        elif "rc_fused" in mut and rc is not None:  # (the mutant lives in the fused epilogue only)
            r, s, c = (f32(v).astype(np.float64) for v in rc)
            p = np.stack([r * c, r * s], axis=-1)  # exact (24 + 24 bits)
            x = (sd.astype(np.float64) * p + mean.astype(np.float64)).astype(F)
        else:
            x = fma32(sd, eps, mean)
        a = clamp(x, -1.0, hi_a, mut)
        d = ((x if "lp_unclipped" in mut else a) - mean).astype(F)
        q = ((F(2) * sd).astype(F) * sd).astype(F)
        t = ((-(d * d).astype(F)) / q).astype(F)
        t = (t - (math.log(sd) if "neg_log_exp" in mut else ls)).astype(F)
        t = (t - LOG_SQRT_2PI).astype(F)
        lp = ((F(0) + t[..., 0]).astype(F) + t[..., 1]).astype(F)
    return a, lp


def sample_from_words(w, mean, log_std, math, mut=frozenset()):
    """The sampling epilogue for one launch: ``eps = box_muller(w)``, then ``gaussian_sample``.  ``(eps, actions, log_prob)``."""
    r, s, c = box_muller_parts(w[:, 0], w[:, 1], math, mut, w[:, 2])
    with np.errstate(invalid="ignore"):
        eps = np.stack([(r * c).astype(F), (r * s).astype(F)], axis=-1)
    a, lp = gaussian_sample(mean, log_std, eps, math, mut, rc=(r, s, c))
    return eps, a, lp


# ----------------------------------------------------------------------------------------------------------------------
# fixtures with constructed edges
# ----------------------------------------------------------------------------------------------------------------------
def _up(x, k=1):
    x = F(x)
    for _ in range(abs(k)):
        x = np.nextafter(x, F(np.inf) if k > 0 else F(-np.inf))
    return F(x)


NAN = F(np.nan)
SUB = F(np.float32(1e-45))              # the smallest subnormal
LS_EDGES = [F(-20), _up(-20, -1), _up(-20, 1), F(2), _up(2, -1), _up(2, 1), F(-25), F(3), F(0), F(-0.0), NAN,
            F(-np.inf), F(np.inf), F(-0.5), F(0.7), F(1e-3), F(-0.03)]
MEAN_EDGES = [F(1), F(-1), F(0), F(-0.0), SUB, -SUB, F(np.finfo(F).tiny), _up(1, -1), _up(-1, 1), F(0.5), F(-0.25),
              F(0.999), NAN]


def crafted_words():
    """Philox words random counters never reach: ``w >> 8`` at 0 and 2^24 - 1 for u1, and ``w1 >> 8`` at 0, 2^22, 2^23,
    3 * 2^22 (the quadrant points of the angle), each with low bytes 0x00 and 0xff (dropped by the shift)."""
    hi0 = [0, 1, 2, (1 << 23), (1 << 24) - 2, (1 << 24) - 1]
    hi1 = [0, 1 << 22, 1 << 23, 3 << 22, 1, (1 << 24) - 1]
    w0 = np.array([(h << 8) | lo for h in hi0 for lo in (0, 0xFF)], dtype=np.uint32)
    w1 = np.array([(h << 8) | lo for h in hi1 for lo in (0, 0xFF)], dtype=np.uint32)
    W0, W1 = np.meshgrid(w0, w1, indexing="ij")
    return W0.reshape(-1), W1.reshape(-1)


def log_words():
    """Words whose u1 is a recorded point where ``logf`` is not the correctly rounded log (``act_math.npz``)."""
    z = np.load(GOLDEN_MATH)
    k = np.round(f32(z["log_x"]).astype(np.float64) * 2.0 ** 24).astype(np.int64) - 1  # u1 = (k + 1) 2^-24
    return (k.astype(np.uint32) << np.uint32(8)) | np.uint32(0x5A)


def _landing_eps(sd, m, target, fma=fma32):
    """An fp32 ``eps`` with ``fma(sd, eps, m) == target`` (searched around ``(target - m) / sd``), or NaN if none."""
    e0 = F((np.float64(target) - np.float64(m)) / np.float64(sd))
    cands = [e0]
    lo = hi = e0
    for _ in range(256):
        lo, hi = np.nextafter(lo, F(-np.inf)), np.nextafter(hi, F(np.inf))
        cands += [lo, hi]
    c = f32(cands)
    ok = fma(np.full_like(c, sd), c, np.full_like(c, m)) == F(target)
    return c[np.argmax(ok)] if ok.any() else NAN


def gaussian_fixture(math, seed=0):
    """``[(log_std [2], mean [N, 2], eps [N, 2])]``: one case per log_std pair (the kernels read one pair per launch)."""
    rng = np.random.default_rng(seed)
    pairs = [(LS_EDGES[i], LS_EDGES[(i + 1) % len(LS_EDGES)]) for i in range(len(LS_EDGES))] + [(NAN, NAN), (F(-0.5), NAN)]
    W0, W1 = crafted_words()
    extreme = box_muller(W0, W1, math).reshape(-1)  # +-r_max = sqrt(-2 ln 2^-24), +-0, the quadrant points
    eps_edges = np.unique(np.concatenate([f32([0.0, -0.0, 1.0, -1.0, 0.5, -3.0]), extreme[np.isfinite(extreme)]]))
    eps_edges = np.concatenate([eps_edges, f32([-0.0])])  # np.unique merges -0 into +0
    cases = []
    for ls in pairs:
        ls = f32(ls)
        sd = math.exp(clamp(ls, -20.0, 2.0))
        rows = []
        # every mean edge against every noise edge, the other component rolled
        me, ee = np.meshgrid(f32(MEAN_EDGES), eps_edges, indexing="ij")
        me, ee = me.reshape(-1), ee.reshape(-1)
        rows.append((np.stack([me, np.roll(me, 7)], 1), np.stack([ee, np.roll(ee, 3)], 1)))
        # the sample lands exactly on +-1 and one ulp either side
        for m in f32([0.3, -0.7, 0.0, 0.999, -1e-45, 0.5]):
            for t in (F(1), _up(1, -1), _up(1, 1), F(-1), _up(-1, -1), _up(-1, 1)):
                e = [_landing_eps(sd[j], m, t) if np.isfinite(sd[j]) and sd[j] > 0 else F(0) for j in range(2)]
                rows.append((f32([[m, m]]), f32([e])))
        # fma and mul + add round differently: found by search
        m = rng.uniform(-1, 1, size=(4096, 2)).astype(F)
        e = rng.standard_normal((4096, 2)).astype(F)
        with np.errstate(invalid="ignore"):
            differ = (fma32(sd, e, m) != mul_add32(sd, e, m)).all(axis=1)
        rows.append((m[differ][:24], e[differ][:24]))
        # ordinary draws
        rows.append((rng.uniform(-1, 1, size=(16, 2)).astype(F), rng.standard_normal((16, 2)).astype(F)))
        mean = np.concatenate([r[0] for r in rows]).astype(F)
        eps = np.concatenate([r[1] for r in rows]).astype(F)
        eps = np.where(np.isnan(eps), F(0), eps)  # (no landing eps: keep the row with eps 0)
        cases.append((ls, mean, eps))
    return cases
