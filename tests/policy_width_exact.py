"""``policy_exact`` for any encoder input width R: lattice cases on which the policy / value kernels are exact, and the
float64 reference at the kernels' rounding points, for observations ``[N, 4 + R]`` whose encoder reads ``s[:, 3:-1]``
= columns ``[3, 3 + R)`` (no tests in this module).

The number formats, the layer arithmetic and the exactness certificate are ``policy_exact``'s (``bf16``, ``leaky``,
``matmul64``, ``certify``, ``linear``); only the width of layer 0 and of the observation is general here.  At R = 961
``build_net`` draws the same weights as ``policy_exact.build_net`` from the same generator, and ``forward`` gives the same
bits as ``policy_exact.forward``.

Defects (``DEFECTS``) are the layer-0 mistakes a run-time chunk count can make, each computed as a wrong reference so
that the tests can show it changes an output bit:
  * ``shift``: the window shifted by one column (columns [4, 4 + R));
  * ``last_col``: the dropped last column (3 + R) fed in, with its neighbour's weights;
  * ``tail_k``: the tail chunk (the last 64-column chunk, where the chunk count steps) read one column further along K;
  * ``chunk_short``: one chunk too few (the tail chunk's columns never reach the MMA).
"""
from __future__ import annotations

import numpy as np

import policy_exact as PE

ENC0 = PE.ENC0
DEFECTS = ("shift", "last_col", "tail_k", "chunk_short")


def in_dims(r: int) -> tuple:
    return (r,) + PE.IN_DIMS[1:]


def tail_start(r: int) -> int:
    """First encoder input index of the last 64-column observation chunk (the bf16 pass's chunk; the fp32 pass's 32-column
    chunks end on the same column)."""
    n_chunks = (ENC0 + r + 63) // 64
    return max(64 * (n_chunks - 1) - ENC0, 0)


def encoder_input(obs, r: int, defect: str | None = None):
    """Layer 0's operand ``bf16(obs[:, 3:3 + R])`` and the column count its weights need (R, or R + 1 for ``last_col``)."""
    obs = np.asarray(obs, np.float32)
    x = PE.bf16(obs[:, ENC0 + (defect == "shift"):ENC0 + r + (defect == "shift")])
    if defect == "last_col":
        x = np.concatenate([x, PE.bf16(obs[:, ENC0 + r:ENC0 + r + 1])], axis=1)
    elif defect == "tail_k":
        k0 = tail_start(r)
        x = x.copy()
        x[:, k0:] = PE.bf16(obs[:, ENC0 + k0 + 1:ENC0 + r + 1])
    elif defect == "chunk_short":
        x = x.copy()
        x[:, tail_start(r):] = 0.0
    return x


def forward(obs, net: PE.Net, r: int, defect: str | None = None, check: bool = True) -> dict:
    """Reference forward pass of a width-R network (``policy_exact.forward`` with layer 0 over [3, 3 + R)): ``pre``
    (s0..s5, fp32), ``act`` (a0..a4), ``out`` (= s5).  ``defect``: one of ``DEFECTS``; only the true reference is
    certified."""
    obs = np.asarray(obs, np.float32)
    if obs.shape[1] != 4 + r or net.w[0].shape[1] != r:
        raise ValueError(f"observations [N, {4 + r}] and W0 [80, {r}] expected")
    check = check and defect is None
    x = encoder_input(obs, r, defect)
    w0 = net.w[0] if defect != "last_col" else np.concatenate([net.w[0], net.w[0][:, r - 1:r]], axis=1)
    head = PE.bf16(obs[:, 0:4])
    pre, act = [], []
    for l in range(6):
        s = PE.linear(x, w0 if l == 0 else net.w[l], net.b[l], check, name=f"layer {l}")
        pre.append(s)
        if l < 5:
            a = PE.leaky(s)
            act.append(a)
            x = np.concatenate([head, a], axis=1) if l == 1 else a
    return {"pre": pre, "act": act, "out": pre[5]}


def make_obs(n: int, r: int, rng: np.random.Generator, tie_fraction: float = 0.125) -> np.ndarray:
    """``policy_exact.make_obs`` for observations ``[n, 4 + r]`` (at r = 961 the same values from the same generator)."""
    cols = 4 + r
    obs = (rng.integers(-255, 256, size=(n, cols)) * 2.0 ** -4).astype(np.float32)
    sel = rng.random((n, cols)) < tie_fraction
    k = int(sel.sum())
    m = rng.integers(128, 256, size=k)
    tie = (2 * m + 1) * 2.0 ** -5 + rng.integers(-1, 2, size=k) * 2.0 ** -20
    obs[sel] = (tie * rng.choice([-1.0, 1.0], size=k)).astype(np.float32)
    return obs


def build_net(obs, r: int, family: str, rng: np.random.Generator, n_out: int):
    """``policy_exact.build_net`` for a width-R encoder: weights certified on these observations, and the reference
    pass.  Raises ``policy_exact.CertificateError`` where the family cannot be made exact at this width."""
    obs = np.asarray(obs, np.float32)
    x = PE.bf16(obs[:, ENC0:ENC0 + r])
    head = PE.bf16(obs[:, 0:4])
    dims = in_dims(r)
    ws, bs, pre, act = [], [], [], []
    for l in range(6):
        k_in, n_units, last = dims[l], (n_out if l == 5 else PE.HIDDEN[l]), l == 5
        if family == "dense":
            wi = rng.integers(-7, 8, size=(n_units, k_in)).astype(np.float64)
        elif family == "sparse":
            wi = np.zeros((n_units, k_in))
            for i in range(n_units):
                c = int(rng.integers(1, min(4, k_in) + 1)) if k_in < 4 else int(rng.integers(1, 5))
                wi[i, rng.choice(k_in, size=c, replace=False)] = rng.choice([-3.0, -2.0, -1.0, 1.0, 2.0, 3.0], size=c)
        else:
            raise ValueError(family)
        raw = PE.matmul64(x, wi)
        lo, hi = raw.min(axis=0), raw.max(axis=0)
        span = max(float((hi - lo).max()), float(np.abs(raw).max()) / 8, 2.0 ** -60)
        if last:
            e = np.round(np.log2(4.0 / span))
            bias = -np.floor((lo + hi) * 2.0 ** e / 2) + rng.integers(-2 ** 11, 2 ** 11, size=n_units) * 2.0 ** -12
        elif family == "dense":
            e = np.round(np.log2(PE.ACT_SCALE / span))
            bias = -lo * 2.0 ** e + PE._p2(max(span * 2.0 ** e, PE.ACT_SCALE / 2))
        else:
            e = np.round(np.log2(PE.ACT_SCALE / 2 / span))
            p = PE._p2(span * 2.0 ** e)
            sign = np.where(np.arange(n_units) % 2 == 0, 1.0, -1.0)
            rng.shuffle(sign)
            bias = sign * p - (lo + hi) * 2.0 ** e / 2 + rng.integers(0, 2 ** 11, size=n_units) * p * 2.0 ** -12 * sign
        wi = wi * 2.0 ** e
        PE.certify(x, wi, bias, name=f"layer {l}")
        s = (raw * 2.0 ** e + bias).astype(np.float32)
        if family == "dense" and not last and not (s > 0).all():
            raise PE.CertificateError(f"dense layer {l}: a pre-activation is not positive")
        ws.append(wi)
        bs.append(bias)
        pre.append(s)
        if not last:
            a = PE.leaky(s)
            act.append(a)
            x = np.concatenate([head, a], axis=1) if l == 1 else a
    return PE.Net(ws, bs), {"pre": pre, "act": act, "out": pre[5]}


class Case:
    """``policy_exact.Case`` at width R: observations ``[N, 4 + R]``, a policy (2 outputs) and a value network (1 output,
    other weights), and their references."""

    def __init__(self, obs, r: int, family: str, seed: int):
        rng = np.random.default_rng(seed)
        self.obs, self.r, self.family = np.asarray(obs, np.float32), r, family
        self.policy, self.ref_policy = build_net(self.obs, r, family, rng, 2)
        self.value, self.ref_value = build_net(self.obs, r, family, rng, 1)

    @property
    def n(self) -> int:
        return self.obs.shape[0]


def make_case(n: int, r: int, family: str, seed: int, obs=None) -> Case:
    """``policy_exact.make_case`` at width R (the same generator calls: at R = 961 the same case)."""
    rng = np.random.default_rng(seed)
    if obs is None:
        obs = make_obs(n, r, rng)
    return Case(obs, r, family, seed + 1)
