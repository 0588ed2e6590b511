"""Lattice cases on which the policy / value kernels' arithmetic is EXACT, the float64 reference that follows the kernels'
rounding points, and the certificate that proves the exactness (no tests in this module).

Why.  The tensor-core kernels accumulate bf16 products in fp32 in an order of their own, so on general inputs they can
only be compared with a reference to a tolerance (4e-3 on the means), and a one-line numeric defect -- a bf16 slope, a
bf16-rounded bias, a tanh approximation -- hides inside it.  On the cases built here every product and every partial sum
of every layer is a multiple of a power of two ``g`` and smaller than ``2^24 g``, so it is exact in fp32 in ANY order: the
kernels must then equal the float64 reference bit for bit, and any wrong index, padding, rounding mode or constant shows.

Reference (both networks of models.py:24-36, 89-102, 151-162, at the kernels' rounding points):
    x0 = bf16(obs[:, 3:964])                       (obs columns 0..2 and 964 do not reach the encoder)
    s_l = sum_k x_l[k] W_l[:, k] + b_l              exact (certificate), then fp32
    a_l = bf16_rne(s_l > 0 ? s_l : 0.01f * s_l)     (fp32 multiply)
    x2 = [bf16(obs[:, 0:4]), a1]                    (reference order; column 3 reaches the encoder AND the MLP)
    value = s5 (fp32),  mean = tanh(s5)

Cases.  Weights are small integers times a power of two (exact in bf16); observations are bf16-exact lattice values plus
fp32 values that are not: exact bf16 rounding ties and their fp32 neighbours one ulp either side.  Biases are chosen from
the case's own pre-activations and need more than 8 significant bits.  Two families:
  * ``dense``: every weight drawn, every hidden pre-activation positive (LeakyReLU is the identity) -- pins the MMA operand
    indexing, the K tail, the N padding, the inject of obs[:, 0:4] and the row / tile mapping;
  * ``sparse``: each unit reads 1..4 inputs and about half the units are negative (a bias that dominates the unit's
    inputs fixes its sign, which keeps the magnitudes of a row within a bounded ratio) -- pins the 0.01f branch and the
    RNE rounding of the activations.
The policy and the value network get different weights.
"""
from __future__ import annotations

import numpy as np
import torch

IN_DIMS = (961, 80, 64, 256, 160, 128)
HIDDEN = (80, 60, 256, 160, 128)
ENC0 = 3  # first observation column of the encoder input
SLOPE = np.float32(0.01)
SLOPE_BF16 = np.float32(0.010009765625)  # bf16(0.01): a defect the tests must see
ROWS = 4096  # row chunk of the float64 products
ACT_SCALE = 16.0  # hidden activations sit in [16, 32) (dense) or +-[8, 32) / 0.01 x that (sparse)
DEFECTS = ("slope_bf16", "bias_bf16", "act_rz", "window0", "window1", "window2", "col964", "inject_fp32",
           "transpose0", "transpose1", "transpose2", "transpose3", "transpose4", "transpose5", "tanh_approx")


class CertificateError(AssertionError):
    pass


# ------------------------------------------------------------------------------------------------ number formats
def bf16(x, rz: bool = False) -> np.ndarray:
    """fp32 -> bf16 (round to nearest even, or toward zero with ``rz``), returned as float32."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    if not rz:
        u = u + np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))
    return (u & np.uint32(0xFFFF0000)).view(np.float32)


def lowbit_exp(x) -> np.ndarray:
    """Exponent of the largest power of two dividing each value (+inf for 0)."""
    x = np.abs(np.asarray(x, np.float64))
    m, e = np.frexp(x)
    q = (m * 2.0 ** 53).astype(np.int64)
    with np.errstate(divide="ignore"):
        tz = np.log2((q & -q).astype(np.float64))
    return np.where(x == 0, np.inf, e - 53 + tz)


def row_lowbit_exp32(x) -> np.ndarray:
    """``lowbit_exp(x).min(axis=1)`` for normal fp32 values, on their bits (+inf for an all-zero row)."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.int32)
    ex = (u >> 23) & 0xFF
    m = (u & 0x7FFFFF) | 0x800000
    low = (m & -m).astype(np.float32).view(np.int32) >> 23  # 127 + trailing zeros of the significand
    lb = np.where(ex == 0, 1 << 20, ex + low - 277).min(axis=1)
    return np.where(lb == 1 << 20, np.inf, lb.astype(np.float64))


def ulp_distance(a, b) -> np.ndarray:
    """Distance of two fp32 arrays in units in the last place (0 for equal bits, +0 == -0)."""
    def ordered(v):
        i = np.ascontiguousarray(v, dtype=np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(ordered(a) - ordered(b))


def leaky(s, slope=SLOPE, rz: bool = False) -> np.ndarray:
    s = np.asarray(s, np.float32)
    return bf16(np.where(s > 0, s, s * slope), rz)


# ------------------------------------------------------------------------------------------------ one layer
def matmul64(x, w) -> np.ndarray:
    """``x [N,K] @ w.T`` in float64 (row chunks): exact whenever the certificate below holds."""
    x = np.asarray(x, np.float32)
    wt = np.asarray(w, np.float64).T.copy()
    out = np.empty((x.shape[0], wt.shape[1]), np.float64)
    for r in range(0, x.shape[0], ROWS):
        out[r:r + ROWS] = x[r:r + ROWS].astype(np.float64) @ wt
    return out


def certify(x, w, b, name: str = "") -> None:
    """The exactness certificate of ``x [N,K] @ w.T + b`` (x: normal fp32 values): for every (row, unit), g = a power of
    two dividing every term and the bias -- the largest dividing all of the row's inputs times the largest dividing all of
    the unit's weights, or the bias's if smaller -- and B = sum |terms| + |bias| must satisfy B < 2^24 g.  Then every
    partial sum, in every order and blocking, is a multiple of g below 2^24 g: exact in fp32, equal to the float64 sum.
    Raises ``CertificateError`` naming the first (row, unit) that fails."""
    x = np.asarray(x, np.float32)
    w = np.asarray(w, np.float64)
    b = np.asarray(b, np.float64)
    wa = np.abs(w).T.copy()
    lb_w = lowbit_exp(w).min(axis=1)
    lb_b = lowbit_exp(b)
    for r in range(0, x.shape[0], ROWS):
        xc = x[r:r + ROWS]
        big = np.abs(xc).astype(np.float64) @ wa + np.abs(b)
        g = np.minimum(row_lowbit_exp32(xc)[:, None] + lb_w[None, :], lb_b[None, :])
        live = big > 0  # (a live row / unit has a nonzero term or bias, so its g is finite)
        gl = np.where(live, g, 0.0)
        ok = ~live | ((big < np.ldexp(1.0, (24 + gl).astype(np.int64))) & (gl >= -120) & (big < 2.0 ** 100))
        if not ok.all():
            n, i = np.argwhere(~ok)[0]
            raise CertificateError(f"{name}: env {r + n} unit {i}: sum |terms| + |bias| = {big[n, i]!r} is not below "
                                   f"2^24 g, g = 2^{g[n, i]:.0f}: its fp32 sums are not exact")


def linear(x, w, b, check: bool = True, name: str = "") -> np.ndarray:
    """``x @ w.T + b`` rounded to fp32 (certified exact with ``check``)."""
    if check:
        certify(x, w, b, name)
    return (matmul64(x, w) + np.asarray(b, np.float64)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ networks
class Net:
    """Six nn.Linear layers (W [out, in] float64, b [out] float64) in the reference's order: encoder 961->80->60, MLP
    [x(4), e(60)] -> 256 -> 160 -> 128 -> out."""

    def __init__(self, w, b):
        self.w, self.b = [np.asarray(t, np.float64) for t in w], [np.asarray(t, np.float64) for t in b]

    def state_dict(self) -> dict:
        from isaac_rover_orbit_b200.policy import WEIGHT_KEYS

        sd = {}
        for k, w, b in zip(WEIGHT_KEYS, self.w, self.b):
            sd[k + ".weight"] = torch.from_numpy(w.astype(np.float32))
            sd[k + ".bias"] = torch.from_numpy(b.astype(np.float32))
        return sd

    def with_outputs(self, rows) -> "Net":
        """The same network with the last layer cut to ``rows`` (e.g. ``[0]``: the first pre-activation as a value)."""
        return Net(self.w[:5] + [self.w[5][rows]], self.b[:5] + [self.b[5][rows]])

    def probe(self, layer: int, unit: int, sign: float) -> "Net":
        """Value network whose output is ``sign * a_layer[unit]`` carried through the layers after ``layer`` by selection
        weights (+1, no bias): a positive activation passes LeakyReLU and bf16 unchanged, so any difference of that unit
        reaches the output (``sign`` is chosen so that the reference value is the positive one)."""
        w, b = [t.copy() for t in self.w[:layer + 1]], [t.copy() for t in self.b[:layer + 1]]
        src = unit
        for l in range(layer + 1, 6):
            n_out = 1 if l == 5 else HIDDEN[l]
            wl = np.zeros((n_out, IN_DIMS[l]))
            wl[0, src + (4 if l == 2 else 0)] = sign if l == layer + 1 else 1.0
            w.append(wl)
            b.append(np.zeros(n_out))
            src = 0
        return Net(w, b)


def _apply_defect_weights(net: Net, defect: str | None):
    w, b = list(net.w), list(net.b)
    if defect == "bias_bf16":
        b = [bf16(t).astype(np.float64) for t in b]
    if defect and defect.startswith("transpose"):
        # one transposed weight pair: W[i, j] <-> W[j, i] for the first pair that differs (if there is none: W[0, j] <->
        # W[0, j + 1])
        l = int(defect[-1])
        wl = w[l].copy()
        m = min(wl.shape)
        pair = next(((i, j) for i in range(m) for j in range(i + 1, m) if wl[i, j] != wl[j, i]), None)
        if pair is not None:
            i, j = pair
            wl[i, j], wl[j, i] = wl[j, i], wl[i, j]
        else:
            j = next(j for j in range(wl.shape[1] - 1) if wl[0, j] != wl[0, j + 1])
            wl[0, j], wl[0, j + 1] = wl[0, j + 1], wl[0, j]
        w[l] = wl
    return w, b


def forward(obs, net: Net, defect: str | None = None, check: bool = True) -> dict:
    """Reference forward pass.  Returns ``pre`` (s0..s5, fp32), ``act`` (a0..a4, bf16 values), ``out`` (= s5).  ``defect``
    (one of ``DEFECTS``) computes a deliberately wrong variant, to show that the comparisons would catch it; only the
    true reference is certified."""
    obs = np.asarray(obs, np.float32)
    check = check and defect is None
    w, b = _apply_defect_weights(net, defect)
    c0 = int(defect[-1]) if defect and defect.startswith("window") else ENC0
    x = bf16(obs[:, c0:c0 + 961])
    w0 = w[0]
    if defect == "col964":  # the dropped column reaches the encoder with the weight of its neighbour
        x = np.concatenate([x, bf16(obs[:, 964:965])], axis=1)
        w0 = np.concatenate([w0, w0[:, 960:961]], axis=1)
    slope = SLOPE_BF16 if defect == "slope_bf16" else SLOPE
    rz = defect == "act_rz"
    head = obs[:, 0:4] if defect == "inject_fp32" else bf16(obs[:, 0:4])
    pre, act = [], []
    for l in range(6):
        s = linear(x, w0 if l == 0 else w[l], b[l], check, name=f"layer {l}")
        pre.append(s)
        if l < 5:
            a = leaky(s, slope, rz)
            act.append(a)
            x = np.concatenate([head, a], axis=1) if l == 1 else a
    return {"pre": pre, "act": act, "out": pre[5]}


def mean_of(out, defect: str | None = None) -> np.ndarray:
    """tanh of the exact pre-activation, rounded to fp32 (``tanh_approx``: with the 2^-11 relative error of
    ``tanh.approx.f32``)."""
    t = np.tanh(np.asarray(out, np.float64))
    if defect == "tanh_approx":
        t = t * (1.0 + 2.0 ** -11)
    return t.astype(np.float32)


# ------------------------------------------------------------------------------------------------ generator
def make_obs(n: int, rng: np.random.Generator, tie_fraction: float = 0.125) -> np.ndarray:
    """Observations ``[n, 965]`` fp32: multiples of 2^-4 below 16 in magnitude (bf16-exact), and a fraction of fp32 values
    that are not bf16: exact ties (2M+1) 2^-5 between two bf16 values M 2^-4, (M+1) 2^-4 (M in [128, 256), both parities:
    ties to even go both ways) and the fp32 values one ulp (2^-20) below and above each tie."""
    obs = (rng.integers(-255, 256, size=(n, 965)) * 2.0 ** -4).astype(np.float32)
    sel = rng.random((n, 965)) < tie_fraction
    k = int(sel.sum())
    m = rng.integers(128, 256, size=k)
    tie = (2 * m + 1) * 2.0 ** -5 + rng.integers(-1, 2, size=k) * 2.0 ** -20
    obs[sel] = (tie * rng.choice([-1.0, 1.0], size=k)).astype(np.float32)
    return obs


def _p2(x: float) -> float:
    return float(2.0 ** np.ceil(np.log2(x)))


def build_net(obs, family: str, rng: np.random.Generator, n_out: int):
    """Weights for one network on these observations -- biases chosen from the case's own pre-activations, every layer
    certified -- and the network's reference pass (what ``forward`` returns)."""
    obs = np.asarray(obs, np.float32)
    x = bf16(obs[:, ENC0:ENC0 + 961])
    head = bf16(obs[:, 0:4])
    ws, bs, pre, act = [], [], [], []
    for l in range(6):
        k_in, n_units, last = IN_DIMS[l], (n_out if l == 5 else HIDDEN[l]), l == 5
        if family == "dense":
            wi = rng.integers(-7, 8, size=(n_units, k_in)).astype(np.float64)
        elif family == "sparse":
            wi = np.zeros((n_units, k_in))
            for i in range(n_units):
                c = int(rng.integers(1, 5))
                wi[i, rng.choice(k_in, size=c, replace=False)] = rng.choice([-3.0, -2.0, -1.0, 1.0, 2.0, 3.0], size=c)
        else:
            raise ValueError(family)
        raw = matmul64(x, wi)
        lo, hi = raw.min(axis=0), raw.max(axis=0)
        span = max(float((hi - lo).max()), float(np.abs(raw).max()) / 8, 2.0 ** -60)
        if last:
            # outputs in about [-2.5, 2.5] (tanh far from saturation): each unit centred, plus a 12-bit offset below 0.5
            e = np.round(np.log2(4.0 / span))
            bias = -np.floor((lo + hi) * 2.0 ** e / 2) + rng.integers(-2 ** 11, 2 ** 11, size=n_units) * 2.0 ** -12
        elif family == "dense":
            # s in [R, R + span_i], R = the largest span rounded up to a power of two: positive, all within a factor 2
            e = np.round(np.log2(ACT_SCALE / span))
            bias = -lo * 2.0 ** e + _p2(max(span * 2.0 ** e, ACT_SCALE / 2))
        else:
            # s in sign * [P/2, 2P): each unit centred on +-P (P >= every unit's span) plus a 12-bit offset below P/2,
            # about half the units negative
            e = np.round(np.log2(ACT_SCALE / 2 / span))
            p = _p2(span * 2.0 ** e)
            sign = np.where(np.arange(n_units) % 2 == 0, 1.0, -1.0)
            rng.shuffle(sign)
            bias = sign * p - (lo + hi) * 2.0 ** e / 2 + rng.integers(0, 2 ** 11, size=n_units) * p * 2.0 ** -12 * sign
        wi = wi * 2.0 ** e
        certify(x, wi, bias, name=f"layer {l}")
        s = (raw * 2.0 ** e + bias).astype(np.float32)
        if family == "dense" and not last and not (s > 0).all():
            raise CertificateError(f"dense layer {l}: a pre-activation is not positive")
        ws.append(wi)
        bs.append(bias)
        pre.append(s)
        if not last:
            a = leaky(s)
            act.append(a)
            x = np.concatenate([head, a], axis=1) if l == 1 else a
    return Net(ws, bs), {"pre": pre, "act": act, "out": pre[5]}


class Case:
    """Observations + a policy network (2 outputs) + a value network (1 output, other weights) + their references."""

    def __init__(self, obs, family: str, seed: int):
        rng = np.random.default_rng(seed)
        self.obs, self.family = np.asarray(obs, np.float32), family
        self.policy, self.ref_policy = build_net(self.obs, family, rng, 2)
        self.value, self.ref_value = build_net(self.obs, family, rng, 1)

    @property
    def n(self) -> int:
        return self.obs.shape[0]

    def encoder_rows(self, ref: dict) -> np.ndarray:
        """The MLP's input as the fused encoder writes it: ``[e(60), bf16(obs[:, 0:4])]`` (bf16 values as float32)."""
        return np.concatenate([ref["act"][1], bf16(self.obs[:, 0:4])], axis=1)


def make_case(n: int, family: str, seed: int, obs=None) -> Case:
    rng = np.random.default_rng(seed)
    if obs is None:
        obs = make_obs(n, rng)
    return Case(obs, family, seed + 1)
