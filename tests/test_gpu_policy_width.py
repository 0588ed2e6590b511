"""GPU: the policy and value networks for any encoder input width R (``encoder_input_size``; observations ``[N, 4 + R]``,
encoder over columns ``[3, 3 + R)``), through ``rover_policy_pass`` / ``rover_b200::policy_pass``.

Every form -- fp32 and bf16 observations; policy, value and both networks in one pass; forward and act -- must equal the
exact float64 model of ``policy_width_exact`` bit for bit on its lattice cases, and the forms must agree with each other
bit for bit on general weights.  At R = 961 the new entry point equals the fixed-width ones and the blob is unchanged."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

import act_exact as AX  # noqa: E402
import policy_exact as PE  # noqa: E402
import policy_width_exact as PW  # noqa: E402
from isaac_rover_orbit_b200 import _lib, ops, torch_ops  # noqa: E402
from isaac_rover_orbit_b200 import terrain as TR  # noqa: E402
from isaac_rover_orbit_b200.config import RoverEnvCfg  # noqa: E402
from isaac_rover_orbit_b200.env import RoverEnv  # noqa: E402
from isaac_rover_orbit_b200.policy import (DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs,  # noqa: E402
                                           alloc_obs_bf16, policy_value_act, policy_value_forward)
from isaac_rover_orbit_b200.trainer import (PPORolloutAgent, RolloutMemory, SkrlSequentialLogTrainer,  # noqa: E402
                                            compute_gae)

pytestmark = pytest.mark.gpu
OPS = torch.ops.rover_b200
# the chunk-count steps of both stage sizes (61 / 62, 125 / 126, 1021 / 1022), ORBIT's grids (81 .. 3721) and the ends
WIDTHS = [1, 61, 62, 81, 125, 126, 256, 441, 651, 961, 1021, 1022, 1681, 3721, 4092]
SIZES = [1, 127, 128, 129, 16384]
BIG = [81, 961, 3721]  # + N = 65536


def _bits(t):
    return t.contiguous().view(torch.int32)


def _same(got, want, what):
    """Bit for bit, NaN positions included (NaN payloads aside)."""
    got, want = got.reshape(want.shape), want
    gn, wn = torch.isnan(got), torch.isnan(want)
    assert torch.equal(gn, wn), f"{what}: NaN positions differ"
    assert torch.equal(_bits(got.masked_fill(gn, 0.0)), _bits(want.masked_fill(wn, 0.0))), f"{what} differs"


def _nets(dev, r, pol_sd, val_sd, log_std=0.3):
    pol = GaussianNeuralNetwork(device=dev, encoder_input_size=r)
    val = DeterministicNeuralNetwork(device=dev, encoder_input_size=r)
    pol.load_state_dict({**pol_sd, "log_std_parameter": torch.full((2,), log_std)})
    val.load_state_dict(val_sd)
    return pol, val


def _random_sd(r, n_out, seed, last_bias=0.0):
    """Golden-shaped random weights (the scale of the shipped checkpoint's layers) for width R."""
    g = torch.Generator().manual_seed(seed)
    dims = [(80, r), (60, 80), (256, 64), (160, 256), (128, 160), (n_out, 128)]
    from isaac_rover_orbit_b200.policy import WEIGHT_KEYS

    sd = {}
    for k, (o, i) in zip(WEIGHT_KEYS, dims):
        sd[k + ".weight"] = torch.randn(o, i, generator=g) * (1.5 / i ** 0.5)
        sd[k + ".bias"] = torch.randn(o, generator=g) * 0.01
    if last_bias:  # means near +-1 (the action clip fires)
        sd["mlp.6.bias"] = torch.tensor([last_bias, -last_bias])[:n_out]
    return sd


def _states(obs, dev, r, bf16):
    n = obs.shape[0]
    s = alloc_obs_bf16(n, dev, 4 + r) if bf16 else alloc_obs(n, dev, 4 + r)
    s.copy_(torch.as_tensor(obs, device=dev))
    return s


def _all_forms(pol, val, s, seed=5):
    """Every form on states ``s``: the single passes, the one-pass pair, and the sampling forms with their noise."""
    out = {"policy": pol.compute({"states": s})[0], "value": val.compute({"states": s})[0]}
    out["dual_mean"], out["dual_value"] = policy_value_forward(pol, val, s)
    rng = ops.ActionRng(seed, s.device)
    out["eps"] = rng.noise(s.shape[0])
    a, lp, o = pol.act({"states": s}, rng=rng)
    out["act_actions"], out["act_log_prob"], out["act_mean"] = a, lp, o["mean_actions"]
    rng = ops.ActionRng(seed, s.device)
    a, lp, v, m = policy_value_act(pol, val, s, rng)
    out["dact_actions"], out["dact_log_prob"], out["dact_value"], out["dact_mean"] = a, lp, v, m
    return out


def _check_consistent(out, log_std, what):
    """Dual = the two single passes; act = forward + gaussian_act fed the previewed noise."""
    for k in ("dual_mean", "act_mean", "dact_mean"):
        _same(out[k], out["policy"], f"{what}: {k}")
    for k in ("dual_value", "dact_value"):
        _same(out[k], out["value"], f"{what}: {k}")
    a, lp = OPS.gaussian_act(out["policy"], log_std, out["eps"])
    for p in ("act", "dact"):
        _same(out[p + "_actions"], a, f"{what}: {p} actions")
        _same(out[p + "_log_prob"], lp.unsqueeze(-1), f"{what}: {p} log_prob")


def _act_equals_model(out, mean, log_std, n, math, what, seed=5):
    """The sampling forms against the exact fp32 model of tests/act_exact.py: the noise ``normal2(seed, step 0, env)``
    and ``gaussian_sample`` of the launch's own means (which are held to the float64 model above), bit for bit."""
    eps = AX.normal2(seed, 0, n, math)
    a, lp = AX.gaussian_sample(mean, log_std.cpu().numpy(), eps, math)
    for p in ("act", "dact"):
        assert AX.bits_equal(out[p + "_actions"].cpu().numpy(), a).all(), f"{what}: {p} actions vs the sampling model"
        assert AX.bits_equal(out[p + "_log_prob"].cpu().numpy().reshape(-1), lp).all(), f"{what}: {p} log_prob vs the model"


# ------------------------------------------------------------------------------------------------ exact lattice cases
_CASES = {}


def _case(r, family, n):
    key = (r, family, n)
    if key not in _CASES:
        _CASES[key] = PW.make_case(n, r, family, seed=7 * r + n % 1000 + (3 if family == "sparse" else 0))
    return _CASES[key]


# the dense family certifies at every width and size used here (checked when the case is built: build_net raises
# policy_exact.CertificateError otherwise, and the test then fails rather than skips)
@pytest.mark.parametrize("family", ["sparse", "dense"])
@pytest.mark.parametrize("r", WIDTHS)
def test_exact_lattice_cases(cuda_device, r, family):
    dev = cuda_device
    math = AX.DeviceMath(dev)
    case = _case(r, family, max(SIZES))
    pol, val = _nets(dev, r, case.policy.state_dict(), case.value.state_dict())
    want_v = torch.from_numpy(case.ref_value["out"][:, 0]).to(dev)
    for bf16 in (False, True):
        for n in SIZES:
            what = f"R={r} {family} N={n} {'bf16' if bf16 else 'fp32'}"
            s = _states(case.obs[:n], dev, r, bf16)
            out = _all_forms(pol, val, s)
            _same(out["value"], want_v[:n], what + " value")
            # the means: tanhf of the exact pre-activation, within 2 ulp of the float64 tanh (test_gpu_policy_exact's
            # rule); the sampling forms: gaussian_act of those means with the previewed noise, bit for bit
            got = out["policy"].cpu().numpy()
            assert PE.ulp_distance(got, PE.mean_of(case.ref_policy["out"][:n])).max() <= 2, what
            _check_consistent(out, pol.log_std_parameter, what)
            _act_equals_model(out, got, pol.log_std_parameter, n, math, what)


@pytest.mark.parametrize("r", BIG)
def test_exact_lattice_cases_65536(cuda_device, r):
    dev = cuda_device
    case = PW.make_case(65536, r, "dense", seed=r)
    pol, val = _nets(dev, r, case.policy.state_dict(), case.value.state_dict())
    want_v = torch.from_numpy(case.ref_value["out"][:, 0]).to(dev)
    for bf16 in (False, True):
        out = _all_forms(pol, val, _states(case.obs, dev, r, bf16))
        _same(out["value"], want_v, f"R={r} value")
        assert PE.ulp_distance(out["policy"].cpu().numpy(), PE.mean_of(case.ref_policy["out"])).max() <= 2
        _check_consistent(out, pol.log_std_parameter, f"R={r} N=65536")


# ------------------------------------------------------------------------------------------------ general weights
@pytest.mark.parametrize("weights", ["random", "saturated"])
@pytest.mark.parametrize("r", WIDTHS)
def test_forms_agree_bitwise(cuda_device, r, weights):
    dev = cuda_device
    pol, val = _nets(dev, r, _random_sd(r, 2, 11, last_bias=6.0 if weights == "saturated" else 0.0), _random_sd(r, 1, 12))
    for n in (129, 16384):
        g = torch.Generator(device=dev).manual_seed(r + n)
        obs = alloc_obs(n, dev, 4 + r)
        obs.copy_(torch.randn(n, 4 + r, device=dev, generator=g))
        ob = alloc_obs_bf16(n, dev, 4 + r)
        ob.copy_(obs)
        rounded = alloc_obs(n, dev, 4 + r)
        rounded.copy_(ob.float())
        o32 = _all_forms(pol, val, rounded)
        o16 = _all_forms(pol, val, ob)
        _check_consistent(o32, pol.log_std_parameter, f"R={r} N={n} fp32")
        _check_consistent(o16, pol.log_std_parameter, f"R={r} N={n} bf16")
        for k in o32:
            _same(o16[k], o32[k], f"R={r} N={n} bf16 vs fp32 on rounded observations: {k}")
        if weights == "saturated":
            assert (o32["act_actions"].abs() == 1.0).any()
        # against a float64 torch forward of the reference network: the tolerance test_gpu_policy.py uses (4e-3 on
        # the means; 4e-3 of the output range on the values)
        ref_m, ref_v = _torch64(obs, pol, r, False), _torch64(obs, val, r, True)
        m, v = pol.compute({"states": obs})[0], val.compute({"states": obs})[0]
        assert (m.double() - ref_m).abs().max() <= 4e-3 + _bf16_noise(obs, pol, r, False, ref_m)
        assert (v.double() - ref_v).abs().max() <= 4e-3 * max(float(ref_v.abs().max()), 1.0) + _bf16_noise(
            obs, val, r, True, ref_v)


def _torch64(obs, net, r, value_head, bf16_operands=False):
    """The reference network (models.py) in float64 torch: encoder over s[:, 3:-1], MLP over [s[:, 0:4], e]."""
    from isaac_rover_orbit_b200.policy import WEIGHT_KEYS

    sd = {k: t.double() for k, t in net.state_dict().items()}
    q = (lambda x: x.to(torch.bfloat16).double()) if bf16_operands else (lambda x: x)
    act = lambda x: torch.nn.functional.leaky_relu(x, 0.01)  # noqa: E731
    lin = lambda k, x: q(x) @ q(sd[k + ".weight"]).T + sd[k + ".bias"]  # noqa: E731
    s = obs.double()
    e = act(lin(WEIGHT_KEYS[1], act(lin(WEIGHT_KEYS[0], s[:, 3:3 + r]))))
    h = torch.cat([s[:, 0:4], e], dim=1)
    for k in WEIGHT_KEYS[2:5]:
        h = act(lin(k, h))
    y = lin(WEIGHT_KEYS[5], h)
    return y if value_head else torch.tanh(y)


def _bf16_noise(obs, net, r, value_head, ref):
    """How far bf16 operands alone move the float64 forward (test_gpu_policy.py holds the kernel to that + 4e-3)."""
    return float((_torch64(obs, net, r, value_head, bf16_operands=True) - ref).abs().max())


# ------------------------------------------------------------------------------------------------ R = 961: as before
def test_961_pass_equals_the_fixed_width_entry_points(cuda_device, golden_dir):
    from oracle import policy as OP

    dev = cuda_device
    pol = GaussianNeuralNetwork(device=dev)
    val = DeterministicNeuralNetwork(device=dev)
    pol.load_state_dict(OP.load_golden_weights(np.load(os.path.join(golden_dir, "policy.npz"))))
    val.load_state_dict(OP.load_golden_weights(np.load(os.path.join(golden_dir, "value.npz"))))
    # the blob of width 961 is today's blob, byte for byte
    n_bytes = torch_ops.policy_packed_bytes(961)
    assert n_bytes == torch_ops.policy_packed_bytes() == pol.packed().numel()
    for n in (1, 129, 16384, 65536):
        g = torch.Generator(device=dev).manual_seed(n)
        obs = alloc_obs(n, dev)
        obs.copy_(torch.randn(n, 965, device=dev, generator=g))
        ob = alloc_obs_bf16(n, dev)
        ob.copy_(obs)
        for s in (obs, ob):
            bf = s.dtype == torch.bfloat16
            for net, head in ((pol, False), (val, True)):
                out = torch.empty(n, 1 if head else 2, device=dev)
                OPS.policy_pass(s, 961, net.packed(), None, head, out, None, None, None, 0, None, None)
                _same(out, OPS.policy_forward(s, net.packed(), head), f"N={n} single")
            mean, value = torch.empty(n, 2, device=dev), torch.empty(n, 1, device=dev)
            OPS.policy_pass(s, 961, pol.packed(), val.packed(), False, mean, value, None, None, 0, None, None)
            fixed = (OPS.policy_value_forward_bf16 if bf else OPS.policy_value_forward)(s, pol.packed(), val.packed())
            _same(mean, fixed[0], "dual mean")
            _same(value, fixed[1], "dual value")
            for dual in (False, True):
                res = []
                for which in ("pass", "fixed"):
                    st = torch.tensor([77, 3], dtype=torch.int64, device=dev)
                    m, a, lp = (torch.empty(n, 2, device=dev), torch.empty(n, 2, device=dev), torch.empty(n, 1, device=dev))
                    v = torch.empty(n, 1, device=dev)
                    if which == "pass":
                        OPS.policy_pass(s, 961, pol.packed(), val.packed() if dual else None, False, m, v if dual else None,
                                        pol.log_std_parameter, st, 5, a, lp)
                    elif dual:
                        (OPS.policy_value_act_bf16 if bf else OPS.policy_value_act)(
                            s, pol.packed(), val.packed(), pol.log_std_parameter, st, 5, m, v, a, lp)
                    else:
                        OPS.policy_act(s, pol.packed(), pol.log_std_parameter, st, 5, m, a, lp)
                    res.append((m, a, lp, v if dual else m, st))
                for x, y in zip(*res):
                    _same(x.float(), y.float(), f"N={n} act dual={dual}")


def _fixed_width_blob(sd) -> np.ndarray:
    """The packed blob of a 961-wide network by the fixed-width layout rover_policy_pack had before the width became a
    run-time value, restated in numpy: W0 in 16 chunks of [8 planes][80 rows][8] bf16 over observation columns [0, 1024)
    (column c carries W0[:, c - 3], zero outside [3, 964)), then W1..W5 as [K/8 planes][N rows][8] bf16 (W2's columns
    in the operand order [e(60), obs[:, 0:4]]), then every layer's bias as fp32, all padded to the kernels' shapes."""
    from isaac_rover_orbit_b200.policy import WEIGHT_KEYS

    k_pad, n_pad = (1024, 80, 64, 256, 160, 128), (80, 64, 256, 160, 128, 16)
    parts, biases = [], []
    for l, key in enumerate(WEIGHT_KEYS):
        w = sd[key + ".weight"].numpy().astype(np.float32)
        b = sd[key + ".bias"].numpy().astype(np.float32)
        k = np.arange(k_pad[l])
        src = k - 3 if l == 0 else ((np.where(k < 60, k + 4, k - 60)) if l == 2 else k)
        ok = (src >= 0) & (src < w.shape[1])
        full = np.zeros((n_pad[l], k_pad[l]), np.float32)
        full[: w.shape[0], ok] = w[:, src[ok]]
        img = full.reshape(n_pad[l], k_pad[l] // 8, 8).transpose(1, 0, 2)  # [plane][n][8]
        parts.append((PE.bf16(img).view(np.uint32) >> 16).astype(np.uint16).tobytes())
        bb = np.zeros(n_pad[l], np.float32)
        bb[: b.shape[0]] = b
        biases.append(bb.tobytes())
    return np.frombuffer(b"".join(parts + biases), np.uint8)


@pytest.mark.parametrize("n_out", [2, 1])
def test_961_blob_equals_the_fixed_width_layout(cuda_device, n_out):
    sd = _random_sd(961, n_out, 3 + n_out)
    net = (GaussianNeuralNetwork if n_out == 2 else DeterministicNeuralNetwork)(device=cuda_device, encoder_input_size=961)
    net.load_state_dict({**sd, "log_std_parameter": torch.zeros(2)} if n_out == 2 else sd)
    want = _fixed_width_blob(sd)
    assert want.size == torch_ops.policy_packed_bytes() == torch_ops.policy_packed_bytes(961)
    assert np.array_equal(net.packed().cpu().numpy(), want)


def test_961_blob_is_byte_identical(cuda_device):
    dev = cuda_device
    sd = _random_sd(961, 2, 3)
    pol = GaussianNeuralNetwork(device=dev, encoder_input_size=961)
    pol.load_state_dict({**sd, "log_std_parameter": torch.zeros(2)})
    blob = pol.packed().clone()
    # the blob packed through the new width rule at 1022 starts with the same W0 chunks' layout and moves the rest
    wide = GaussianNeuralNetwork(device=dev, encoder_input_size=1022)
    sd2 = dict(sd)
    sd2["dense_encoder.encoder_layers.0.weight"] = torch.cat([sd["dense_encoder.encoder_layers.0.weight"],
                                                              torch.zeros(80, 61)], dim=1)
    wide.load_state_dict({**sd2, "log_std_parameter": torch.zeros(2)})
    wb = wide.packed()
    assert wb.numel() == blob.numel() + 10240
    assert torch.equal(wb[:16 * 10240], blob[:16 * 10240]) and not wb[16 * 10240:17 * 10240].any()
    assert torch.equal(wb[17 * 10240:], blob[16 * 10240:])


# ------------------------------------------------------------------------------------------------ NaN / inf
@pytest.mark.parametrize("r", [61, 256, 3721])
def test_nonfinite_observations_propagate(cuda_device, r):
    dev = cuda_device
    pol, val = _nets(dev, r, _random_sd(r, 2, 21), _random_sd(r, 1, 22))
    n = 300
    obs = alloc_obs(n, dev, 4 + r)
    obs.copy_(torch.randn(n, 4 + r, device=dev))
    obs[1, 5] = float("nan")
    obs[2, 3 + r - 1] = float("inf")
    obs[3, 10 % (3 + r)] = -float("inf")
    obs[4, 1] = float("nan")       # head column: reaches the MLP through the inject
    obs[5, 3 + r] = float("nan")   # the dropped last ray: must not reach the encoder
    ob = alloc_obs_bf16(n, dev, 4 + r)
    ob.copy_(obs)
    for s in (obs, ob):
        out = _all_forms(pol, val, s)
        _check_consistent(out, pol.log_std_parameter, f"R={r} nonfinite")
        m = out["policy"]
        assert torch.isnan(m[1]).all() and torch.isnan(m[4]).all()
        assert not torch.isnan(m[5]).any() and not torch.isnan(m[0]).any()
        assert torch.isnan(out["act_actions"][1]).all()
        ref = alloc_obs(n, dev, 4 + r)
        ref.copy_(obs)
        ref[5, 3 + r] = 0.0
        _same(m[5], pol.compute({"states": ref})[0][5], "dropped column ignored")


# ------------------------------------------------------------------------------------------------ errors, graphs, opcheck
def test_blob_sizes_are_checked(cuda_device):
    """A blob packed for another width is refused by the fixed-width operators (they would read the 961 layout past its
    end), and packing refuses a buffer shorter than the weights' width needs."""
    dev = cuda_device
    n = 64
    pol256, val256 = _nets(dev, 256, _random_sd(256, 2, 1), _random_sd(256, 1, 2))
    p961, v961 = _nets(dev, 961, _random_sd(961, 2, 1), _random_sd(961, 1, 2))
    obs, ob = alloc_obs(n, dev), alloc_obs_bf16(n, dev)
    ls, st = p961.log_std_parameter, torch.tensor([1, 0], dtype=torch.int64, device=dev)
    m, a, lp, v = (torch.empty(n, 2, device=dev), torch.empty(n, 2, device=dev), torch.empty(n, 1, device=dev),
                   torch.empty(n, 1, device=dev))
    for s in (obs, ob):
        bf = s.dtype == torch.bfloat16
        calls = [lambda: OPS.policy_forward(s, pol256.packed(), False),
                 lambda: OPS.policy_forward(s, val256.packed(), True),
                 lambda: OPS.policy_act(s, pol256.packed(), ls, st, 0, m, a, lp),
                 lambda: (OPS.policy_value_forward_bf16 if bf else OPS.policy_value_forward)(s, p961.packed(),
                                                                                             val256.packed()),
                 lambda: (OPS.policy_value_forward_bf16 if bf else OPS.policy_value_forward)(s, pol256.packed(),
                                                                                             v961.packed()),
                 lambda: (OPS.policy_value_act_bf16 if bf else OPS.policy_value_act)(s, pol256.packed(), v961.packed(), ls,
                                                                                     st, 0, m, v, a, lp)]
        for k, call in enumerate(calls):
            with pytest.raises(RuntimeError, match="961"):
                call()
                pytest.fail(f"case {k} was accepted")
    torch.cuda.synchronize()
    assert st.cpu().tolist() == [1, 0]  # nothing launched
    # packing: a 1681-wide W0 needs policy_packed_bytes(1681) bytes, more than the 961 default
    net = GaussianNeuralNetwork(device=dev, encoder_input_size=1681)
    net.load_state_dict({**_random_sd(1681, 2, 7), "log_std_parameter": torch.zeros(2)})
    keys = [k for k in net.state_dict() if k.endswith(".weight")]
    ws = [net.state_dict()[k] for k in keys]
    bs = [net.state_dict()[k[:-len("weight")] + "bias"] for k in keys]
    short = torch.zeros(torch_ops.policy_packed_bytes() + 64, dtype=torch.uint8, device=dev)
    short = short[(-short.data_ptr()) % 128:][: torch_ops.policy_packed_bytes()]
    with pytest.raises(RuntimeError, match="at least"):
        OPS.policy_pack(ws, bs, short)
    torch.cuda.synchronize()
    assert not short.any()  # nothing written
    size = torch_ops.policy_packed_bytes(1681)
    buf = torch.zeros(size + 128, dtype=torch.uint8, device=dev)
    buf = buf[(-buf.data_ptr()) % 128:][:size]
    OPS.policy_pack(ws, bs, buf)
    assert torch.equal(buf, net.packed())


def test_mean_output_must_be_8_byte_aligned(cuda_device):
    """The kernel stores each row's mean as one float2: a 4-byte-offset output is refused by the operator and by the C
    export, before any launch."""
    dev = cuda_device
    r, n = 256, 40
    pol, val = _nets(dev, r, _random_sd(r, 2, 1), _random_sd(r, 1, 2))
    obs = alloc_obs(n, dev, 4 + r)
    raw = torch.full((2 * n + 2,), 7.0, device=dev)
    odd = raw[1:1 + 2 * n].view(n, 2)  # contiguous, 4 bytes off an 8-byte boundary
    assert odd.data_ptr() % 8 == 4
    for pv, v in ((None, None), (val.packed(), torch.empty(n, 1, device=dev))):
        with pytest.raises(RuntimeError, match="8-byte"):
            OPS.policy_pass(obs, r, pol.packed(), pv, False, odd, v, None, None, 0, None, None)
    p = _lib.PolicyPass(obs=obs.data_ptr(), packed=pol.packed().data_ptr(), out=odd.data_ptr(), obs_dtype=_lib.OBS_FP32,
                        stride=int(obs.stride(0)), n_envs=n, enc_in=r)
    assert _lib.load().rover_policy_pass(ctypes.byref(p), _lib.current_stream(dev)) != 0
    assert b"8-byte aligned" in _lib.load().rover_last_error()
    torch.cuda.synchronize()
    assert bool((raw == 7.0).all())
    # a value output has no such requirement: [N] floats at any 4-byte offset
    vout = raw[1:1 + n].view(n, 1)
    OPS.policy_pass(obs, r, val.packed(), None, True, vout, None, None, None, 0, None, None)
    _same(vout, val.compute({"states": obs})[0], "value at a 4-byte offset")


def test_bad_widths_and_layouts_raise(cuda_device):
    dev = cuda_device
    for bad in (0, 4093):
        with pytest.raises(ValueError):
            GaussianNeuralNetwork(device=dev, encoder_input_size=bad)
    pol, val = _nets(dev, 256, _random_sd(256, 2, 1), _random_sd(256, 1, 2))
    with pytest.raises(RuntimeError, match=r"\[N,260\]"):
        pol.compute({"states": alloc_obs(8, dev, 261)})
    with pytest.raises(RuntimeError, match=r"\[N,260\]"):
        pol.compute({"states": alloc_obs_bf16(8, dev, 965)})
    with pytest.raises(RuntimeError, match=r"\[N,260\]"):
        val.compute({"states": alloc_obs(8, dev)})
    # a misaligned row stride: re-homed for the network API (fp32), rejected by the operator and for bf16 states
    raw = torch.randn(8, 261, device=dev)[:, :260]
    m = pol.compute({"states": raw})[0]
    s = alloc_obs(8, dev, 260)
    s.copy_(raw)
    _same(m, pol.compute({"states": s})[0], "re-homed")
    out = torch.empty(8, 2, device=dev)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        OPS.policy_pass(raw, 256, pol.packed(), None, False, out, None, None, None, 0, None, None)
    rb = torch.zeros(8, 261, dtype=torch.bfloat16, device=dev)[:, :260]
    with pytest.raises(RuntimeError, match=r"\[N,260\]"):
        pol.compute({"states": rb})
    with pytest.raises((RuntimeError, ValueError)):
        OPS.policy_pass(s, 0, pol.packed(), None, False, out, None, None, None, 0, None, None)
    with pytest.raises((RuntimeError, ValueError)):
        OPS.policy_pass(s, 4093, pol.packed(), None, False, out, None, None, None, 0, None, None)
    with pytest.raises(RuntimeError, match="packed for R = 255"):  # a blob of another chunk count
        OPS.policy_pass(alloc_obs(8, dev, 259), 255, _nets(dev, 62, _random_sd(62, 2, 1), _random_sd(62, 1, 2))[0].packed(),
                        None, False, out, None, None, None, 0, None, None)
    # mixing widths between the policy and the value network
    _, v81 = _nets(dev, 81, _random_sd(81, 2, 1), _random_sd(81, 1, 2))
    for fn in (lambda: policy_value_forward(pol, v81, s), lambda: policy_value_act(pol, v81, s, ops.ActionRng(1, dev))):
        with pytest.raises(ValueError, match="different observations"):
            fn()


def test_fused_encoder_and_mlp_reject_other_widths(cuda_device):
    dev = cuda_device
    pol, _ = _nets(dev, 256, _random_sd(256, 2, 1), _random_sd(256, 1, 2))
    with pytest.raises(ValueError, match="961"):
        pol.packed_fused()
    v, f = TR.make_synthetic_terrain(24.0, 0.2, seed=3)
    grid = ops.ScanGridHandle.from_mesh(v, f, dev)
    rays = ops.RayPattern.grid(dev)
    pos, quat = torch.zeros(4, 3, device=dev), torch.tensor([[1.0, 0, 0, 0]] * 4, device=dev)
    for fn in (ops.height_scan_encoder, ops.height_scan_policy):
        with pytest.raises(ValueError, match="961"):
            fn(pos, quat, rays, grid, alloc_obs(4, dev), pol)
    enc = torch.zeros(8 * 64 + 64, dtype=torch.bfloat16, device=dev)
    enc = enc[((-enc.data_ptr()) % 128) // 2:][: 8 * 64].view(8, 64)
    with pytest.raises(RuntimeError, match="961"):
        OPS.policy_mlp_forward(enc, pol.packed(), False)


@pytest.mark.parametrize("r", [62, 1681])
def test_graph_replay_equals_eager_and_opcheck(cuda_device, r):
    dev = cuda_device
    pol, val = _nets(dev, r, _random_sd(r, 2, 31), _random_sd(r, 1, 32))
    n = 333
    for bf16 in (False, True):
        obs = _states(torch.randn(n, 4 + r).numpy(), dev, r, bf16)
        eager = _all_forms(pol, val, obs, seed=9)
        st = torch.tensor([9, 0], dtype=torch.int64, device=dev)
        mean, value, actions, log_prob = (torch.empty(n, 2, device=dev), torch.empty(n, 1, device=dev),
                                          torch.empty(n, 2, device=dev), torch.empty(n, 1, device=dev))

        def call():
            OPS.policy_pass(obs, r, pol.packed(), val.packed(), False, mean, value, pol.log_std_parameter, st, 0, actions,
                            log_prob)

        call()
        torch.cuda.synchronize()
        st.copy_(torch.tensor([9, 0]))
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            call()
        st.copy_(torch.tensor([9, 0]))
        g.replay()
        torch.cuda.synchronize()
        _same(mean, eager["policy"], "graph mean")
        _same(value, eager["value"], "graph value")
        _same(actions, eager["dact_actions"], "graph actions")
        _same(log_prob, eager["dact_log_prob"], "graph log_prob")
        assert st.cpu().tolist() == [9, 1]
        args = (obs, r, pol.packed(), val.packed(), False, mean, value, pol.log_std_parameter, st, 0, actions, log_prob)
        for tests in ("test_schema", "test_faketensor"):
            torch.library.opcheck(OPS.policy_pass.default, args, test_utils=tests)
        args = (obs, r, pol.packed(), None, False, mean, None, None, None, 0, None, None)
        for tests in ("test_schema", "test_faketensor"):
            torch.library.opcheck(OPS.policy_pass.default, args, test_utils=tests)


# ------------------------------------------------------------------------------------------------ end to end
N_ENV = 160


@pytest.fixture(scope="module")
def terrain48():
    v, f = TR.make_synthetic_terrain(48.0, 0.2, seed=5)
    return TR.build_terrain_tables(v, f, N_ENV)


def _rollouts(dev, tables, resolution, dtype, rollout=12):
    cfg = RoverEnvCfg(num_envs=N_ENV)
    cfg.height_scanner.pattern_cfg.resolution = resolution
    env = RoverEnv(cfg, tables, dev, seed=2, observation_dtype=dtype)
    r = env.scene.sensors["height_scanner"].ray_pattern.n_rays
    pol, val = _nets(dev, r, _random_sd(r, 2, 4), _random_sd(r, 1, 5), log_std=0.5)
    rng = ops.ActionRng(2024, dev)
    mem = RolloutMemory(memory_size=rollout, num_envs=N_ENV, device=dev)
    agent = PPORolloutAgent(pol, val, mem, action_out=env.action_input, action_rng=rng)
    SkrlSequentialLogTrainer(env=env, agents=agent, cfg={"timesteps": 2 * rollout, "disable_progressbar": True}).train()
    torch.cuda.synchronize()
    assert rng.peek()[1] == 2 * rollout
    return r, mem, pol, val, agent


@pytest.mark.parametrize("resolution,rays", [(0.2, 256), (0.05, 3721)])
def test_ppo_rollouts_on_other_grids(cuda_device, terrain48, resolution, rays):
    dev = cuda_device
    res = {}
    for dtype in (torch.float32, torch.bfloat16):
        r, mem, pol, val, agent = _rollouts(dev, terrain48, resolution, dtype)
        assert r == rays
        st = mem.get_tensor_by_name("states")
        assert st.shape == (mem.memory_size, N_ENV, 4 + r)
        # values and log-probs are a separate forward on the recorded states
        t_, n_ = st.shape[:2]
        s = alloc_obs(t_ * n_, dev, 4 + r)
        s.copy_(st.reshape(-1, 4 + r))
        mean, value = policy_value_forward(pol, val, s)
        _same(mem.get_tensor_by_name("values").reshape(-1, 1), value, "values")
        # memory row i holds timestep rollout + i (the second rollout), whose act drew the noise of step rollout + i:
        # that forward's means through gaussian_act with the noise previewed for that step give the recorded actions and
        # log-probs bit for bit
        eps = torch.cat([ops.ActionRng(2024, dev, step=t_ + i).noise(n_) for i in range(t_)])
        a, lp = OPS.gaussian_act(mean, pol.log_std_parameter, eps)
        _same(mem.get_tensor_by_name("actions").reshape(-1, 2), a, "actions")
        _same(mem.get_tensor_by_name("log_prob").reshape(-1), lp, "log_prob")
        # returns and advantages: compute_gae of the memory (last values of the final next_states)
        last = val.act({"states": agent._current_next_states}, role="value")[0]
        ret, adv = compute_gae(mem.get_tensor_by_name("rewards"), mem.get_tensor_by_name("terminated"),
                               mem.get_tensor_by_name("values"), last)
        _same(mem.get_tensor_by_name("returns"), ret, "returns")
        _same(mem.get_tensor_by_name("advantages"), adv, "advantages")
        res[dtype] = mem
    m32, m16 = res[torch.float32], res[torch.bfloat16]
    for k in ("actions", "log_prob", "values", "rewards", "terminated", "returns", "advantages"):
        x, y = m16.get_tensor_by_name(k), m32.get_tensor_by_name(k)
        assert torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                           y.view(torch.int32) if y.dtype == torch.float32 else y), k
    _same(m16.get_tensor_by_name("states"), m32.get_tensor_by_name("states").to(torch.bfloat16).float(), "states")
