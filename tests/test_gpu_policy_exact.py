"""GPU: every tensor-core policy / value entry point against the float64 reference on lattice cases where the kernels'
arithmetic is exact (policy_exact.py): values and pre-activations bit for bit, means within 2 ulp of tanh of the exact
pre-activation (CUDA's documented bound for tanhf).  Entry points: ``compute`` (warp-specialised kernel and v1),
``compute_bf16``, ``policy_value_forward``, ``rover_policy_mlp_forward`` on encoder rows written directly, and the height
scan fused with the encoder followed by the MLP.  Shapes walk the tiling of ``launch_policy_forward_ws`` (tile height
ceil(N / (rounds * SMs)) rounded up to 8, at most 128).  A mismatch is reported with the first differing environment and
output, and localised to a layer and unit by re-running the case with the layers after each unit replaced by selection
weights."""
import numpy as np
import pytest
import torch

import policy_exact as PE
from isaac_rover_orbit_b200 import ops
from isaac_rover_orbit_b200.policy import (DeterministicNeuralNetwork, GaussianNeuralNetwork, alloc_obs, alloc_obs_bf16,
                                            policy_value_forward)

pytestmark = pytest.mark.gpu

# environment counts; "s" = the device's SM count (148 on a B200)
SMALL = ["1", "7", "8", "9", "127", "128", "129", "8s-1", "8s", "8s+1"]
CASES = [(n, fam) for n in SMALL for fam in ("dense", "sparse")] + [
    ("128s-1", "sparse"), ("128s", "dense"), ("128s+1", "sparse"), ("256s+77", "dense"), ("65536", "dense")]
_CACHE: dict = {}


def _size(spec: str, n_sms: int) -> int:
    if "s" not in spec:
        return int(spec)
    k, _, off = spec.partition("s")
    return int(k) * n_sms + (int(off) if off else 0)


def _case(spec, family, n_sms) -> PE.Case:
    n = _size(spec, n_sms)
    key = (n, family)
    if key not in _CACHE:
        _CACHE[key] = PE.make_case(n, family, seed=1000 + n + (7 if family == "sparse" else 0))
    return _CACHE[key]


@pytest.fixture(scope="module")
def n_sms(cuda_device):
    return torch.cuda.get_device_properties(cuda_device).multi_processor_count


class Nets:
    """One network object per role, re-loaded per case (each load re-packs the weights)."""

    def __init__(self, dev):
        self.dev = dev
        self.pol = GaussianNeuralNetwork(device=dev)
        self.val, self.pre0, self.pre1, self.probe = (DeterministicNeuralNetwork(device=dev) for _ in range(4))

    def load(self, case: PE.Case):
        sd = case.policy.state_dict()
        sd["log_std_parameter"] = torch.zeros(2)
        self.pol.load_state_dict(sd)
        self.val.load_state_dict(case.value.state_dict())
        self.pre0.load_state_dict(case.policy.with_outputs([0]).state_dict())
        self.pre1.load_state_dict(case.policy.with_outputs([1]).state_dict())


@pytest.fixture(scope="module")
def nets(cuda_device):
    return Nets(cuda_device)


# ---------------------------------------------------------------------------------------------------- comparison
def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.int32)


def _localize(run, net: PE.Net, obs, n0: int, first_layer: int = 0) -> str:
    """Re-run with probe networks (``Net.probe``): the first (layer, unit) whose value differs at env ``n0``."""
    row = obs[n0:n0 + 1]
    ref = PE.forward(row, net)
    for l in range(first_layer, 5):
        a = ref["act"][l][0]
        for u in range(a.shape[0]):
            probe = net.probe(l, u, -1.0 if a[u] < 0 else 1.0)
            want = PE.forward(row, probe)["out"][0, 0]
            got = np.float32(run(probe)[n0])
            if _bits(got) != _bits(want):
                return (f"first differing layer: {l}, unit {u} (reference activation {float(a[u])!r}, pre-activation "
                        f"{float(ref['pre'][l][0, u])!r}; through the probe: kernel {float(got)!r}, reference {float(want)!r})")
    return "layers 0..4 agree on every unit at this env: the difference is in layer 5 (or its epilogue)"


def _check(entry, what, got, want, obs, net=None, run=None, first_layer=0, mean=False):
    """``got`` vs ``want`` ([N, k] fp32): bit for bit, or (``mean``) within 2 ulp.  On a mismatch, fail naming the first
    differing env and output, localised through ``run`` (value-head runner of this entry point) when given."""
    got = np.asarray(got, np.float32).reshape(want.shape)
    bad = PE.ulp_distance(got, want) > 2 if mean else _bits(got) != _bits(want)
    if not bad.any():
        return
    n0, j = (int(v) for v in np.argwhere(bad)[0])
    msg = (f"{entry}: {what} differs from the exact reference in {int(bad.any(axis=1).sum())} of {want.shape[0]} envs; "
           f"first: env {n0}, output {j}: kernel {float(got[n0, j])!r}, reference {float(want[n0, j])!r}")
    if run is not None:
        try:
            msg += "; " + _localize(run, net, obs, n0, first_layer)
        except Exception as exc:  # the report must not hide the mismatch
            msg += f"; localisation failed: {exc!r}"
    pytest.fail(msg)


def _check_case(entry, case, mean, value, pre0, pre1, run):
    """The four outputs of one entry point.  ``run(net) -> value [N]`` runs a value network through the same entry point."""
    rp, rv = case.ref_policy, case.ref_value
    obs = case.obs
    _check(entry, "value", value, rv["out"], obs, case.value, run)
    _check(entry, "policy pre-activation 0", pre0, rp["out"][:, :1], obs, case.policy, run)
    _check(entry, "policy pre-activation 1", pre1, rp["out"][:, 1:], obs, case.policy, run)
    _check(entry, "mean", mean, PE.mean_of(rp["out"]), obs, case.policy, run, mean=True)


def _np(t):
    return t.detach().float().cpu().numpy()


def _compute_runner(nets, states, bf16: bool):
    def run(net):
        nets.probe.load_state_dict(net.state_dict())
        return _np((nets.probe.compute_bf16 if bf16 else nets.probe.compute)({"states": states})[0]).reshape(-1)
    return run


def _run_compute(entry, nets, case, states, bf16=False):
    f = (lambda m: m.compute_bf16({"states": states})[0]) if bf16 else (lambda m: m.compute({"states": states})[0])
    outs = [_np(f(m)) for m in (nets.pol, nets.val, nets.pre0, nets.pre1)]
    _check_case(entry, case, *outs, run=_compute_runner(nets, states, bf16))


def _run_dual(nets, case, states):
    mean, value = policy_value_forward(nets.pol, nets.val, states)
    m2, pre0 = policy_value_forward(nets.pol, nets.pre0, states)
    _, pre1 = policy_value_forward(nets.pol, nets.pre1, states)
    assert torch.equal(m2, mean)

    def run(net):
        nets.probe.load_state_dict(net.state_dict())
        return _np(policy_value_forward(nets.pol, nets.probe, states)[1]).reshape(-1)
    _check_case("policy_value_forward", case, _np(mean), _np(value), _np(pre0), _np(pre1), run)


# ---------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("spec,family", CASES)
def test_entry_points_equal_the_exact_reference(cuda_device, n_sms, nets, spec, family, monkeypatch):
    case = _case(spec, family, n_sms)
    nets.load(case)
    states = alloc_obs(case.n, cuda_device)
    states.copy_(torch.from_numpy(case.obs))
    monkeypatch.setenv("ROVER_POLICY_KERNEL", "ws")
    _run_compute("compute (ws)", nets, case, states)
    monkeypatch.setenv("ROVER_POLICY_KERNEL", "v1")
    _run_compute("compute (v1)", nets, case, states)
    monkeypatch.setenv("ROVER_POLICY_KERNEL", "ws")
    states_bf = alloc_obs_bf16(case.n, cuda_device)
    states_bf.copy_(states)  # RNE, like the kernels' conversion
    _run_compute("compute_bf16", nets, case, states_bf, bf16=True)
    _run_dual(nets, case, states)


@pytest.mark.parametrize("family", ["dense", "sparse"])
def test_unaligned_rows_and_nonfinite_dropped_column(cuda_device, n_sms, nets, family, monkeypatch):
    """A dense [N, 965] tensor (rows not 16-byte aligned: re-homed by compute / policy_value_forward), and +-inf / NaN in
    column 964, which the reference's slicing drops: the outputs stay those of the exact reference on every path."""
    case = _case("8s+1", family, n_sms)
    nets.load(case)
    obs = torch.from_numpy(case.obs).to(cuda_device)
    obs[0::3, 964] = float("inf")
    obs[1::3, 964] = float("nan")
    obs[2::3, 964] = float("-inf")
    assert obs.stride(0) == 965
    for kernel in ("ws", "v1"):
        monkeypatch.setenv("ROVER_POLICY_KERNEL", kernel)
        _run_compute(f"compute ({kernel}, unaligned rows, non-finite column 964)", nets, case, obs)
    monkeypatch.setenv("ROVER_POLICY_KERNEL", "ws")
    aligned = alloc_obs(case.n, cuda_device)
    aligned.copy_(obs)
    _run_compute("compute (ws, non-finite column 964)", nets, case, aligned)
    states_bf = alloc_obs_bf16(case.n, cuda_device)
    states_bf.copy_(aligned)
    _run_compute("compute_bf16 (non-finite column 964)", nets, case, states_bf, bf16=True)
    _run_dual(nets, case, obs)


def _enc_tensor(rows: np.ndarray, dev) -> torch.Tensor:
    n = rows.shape[0]
    raw = torch.empty(n + 1, 64, dtype=torch.bfloat16, device=dev)
    enc = raw.view(-1)[((-raw.data_ptr()) % 128) // 2:][: n * 64].view(n, 64)
    enc.copy_(torch.from_numpy(rows).to(torch.bfloat16))
    return enc


@pytest.mark.parametrize("spec,family", [("1", "dense"), ("129", "sparse"), ("8s+1", "dense"), ("128s+1", "sparse"),
                                         ("65536", "dense")])
def test_mlp_forward_on_encoder_rows(cuda_device, n_sms, nets, spec, family):
    """rover_policy_mlp_forward on ``[e(60), obs[:, 0:4]]`` bf16 rows written directly (the layout the fused encoder
    stores, fused_scan_policy.cu): layers 2..5 of the exact reference."""
    case = _case(spec, family, n_sms)
    nets.load(case)
    mlp = torch.ops.rover_b200.policy_mlp_forward
    enc_p = _enc_tensor(case.encoder_rows(case.ref_policy), cuda_device)
    enc_v = _enc_tensor(case.encoder_rows(case.ref_value), cuda_device)

    def run_with(enc):
        def run(net):
            nets.probe.load_state_dict(net.state_dict())
            return _np(mlp(enc, nets.probe.packed(), True)).reshape(-1)
        return run
    _check("policy_mlp_forward", "value", _np(mlp(enc_v, nets.val.packed(), True)), case.ref_value["out"], case.obs,
           case.value, run_with(enc_v), first_layer=2)
    outs = {"mean": _np(mlp(enc_p, nets.pol.packed(), False)), "pre0": _np(mlp(enc_p, nets.pre0.packed(), True)),
            "pre1": _np(mlp(enc_p, nets.pre1.packed(), True))}
    rp = case.ref_policy["out"]
    for what, got, want in (("policy pre-activation 0", outs["pre0"], rp[:, :1]),
                            ("policy pre-activation 1", outs["pre1"], rp[:, 1:])):
        _check("policy_mlp_forward", what, got, want, case.obs, case.policy, run_with(enc_p), first_layer=2)
    _check("policy_mlp_forward", "mean", outs["mean"], PE.mean_of(rp), case.obs, case.policy, run_with(enc_p),
           first_layer=2, mean=True)


@pytest.fixture(scope="module")
def tilted_plane(cuda_device):
    """The plane z = 0.1 x - 0.05 y + 1 (two triangles); body heights 3 m above it: all 961 heights in about [2.7, 3.3],
    bf16 multiples of 2^-6 -- inside the certified range of the dense family."""
    from isaac_rover_orbit_b200 import synthetic

    v = np.array([[-50, -50, 0], [50, -50, 0], [50, 50, 0], [-50, 50, 0]], dtype=np.float32)
    v[:, 2] = 0.1 * v[:, 0] - 0.05 * v[:, 1] + 1.0
    f = np.array([[0, 1, 2], [0, 2, 3]], dtype=np.int32)
    grid = ops.ScanGridHandle.from_mesh(v, f, cuda_device)

    def poses(n, seed):
        g = torch.Generator().manual_seed(seed)
        xy = torch.rand(n, 2, generator=g) * 60 - 30
        z = 0.1 * xy[:, 0:1] - 0.05 * xy[:, 1:2] + 1.0 + 3.0 + 0.26878
        yaw = (torch.rand(n, generator=g) * 2 - 1) * np.pi
        q = synthetic.quat_from_euler(torch.zeros(n), torch.zeros(n), yaw)
        return torch.cat([xy, z], 1).to(cuda_device), q.to(cuda_device)
    return grid, ops.RayPattern.grid(cuda_device), poses


@pytest.mark.parametrize("spec", ["1", "37", "16s+1", "5000"])
def test_scan_encoder_then_mlp_exact(cuda_device, n_sms, nets, tilted_plane, spec):
    """height_scan_encoder (scan fused with the encoder: transposed MMAs, W0 in tensor memory) + policy_mlp_forward: the
    heights it writes are those of rover_height_scan, the encoder rows and every output equal the exact reference."""
    grid, rays, poses = tilted_plane
    n = _size(spec, n_sms)
    p, q = poses(n, 40 + n)
    head = PE.make_obs(n, np.random.default_rng(n))[:, :4]
    obs_ref = alloc_obs(n, cuda_device)
    obs_ref[:, :4] = torch.from_numpy(head).to(cuda_device)
    ops.height_scan(p, q, rays, grid, out=obs_ref[:, 4:])
    obs_np = obs_ref.cpu().numpy()
    h = obs_np[:, 4:]
    assert np.isfinite(h).all() and h.min() > 2.0 and h.max() < 4.0
    case = PE.Case(obs_np, "dense", seed=77 + n)
    nets.load(case)
    mlp = torch.ops.rover_b200.policy_mlp_forward

    def fused(net, value_head, write_obs=False, obs=None):
        obs = alloc_obs(n, cuda_device) if obs is None else obs
        obs[:, :4] = obs_ref[:, :4]
        enc = ops.height_scan_encoder(p, q, rays, grid, obs, net, write_obs=write_obs)
        return enc, mlp(enc, net.packed(), value_head)

    obs_w = alloc_obs(n, cuda_device)
    obs_w[:, 4:] = 7.0
    enc_p, mean = fused(nets.pol, False, write_obs=True, obs=obs_w)
    assert torch.equal(obs_w, obs_ref), "heights written by the fused kernel are those of rover_height_scan"
    _check("scan_encoder_fused", "encoder rows (policy)", _np(enc_p), case.encoder_rows(case.ref_policy), case.obs)
    enc_v, value = fused(nets.val, True)
    _check("scan_encoder_fused", "encoder rows (value)", _np(enc_v), case.encoder_rows(case.ref_value), case.obs)
    pre0, pre1 = fused(nets.pre0, True)[1], fused(nets.pre1, True)[1]

    def run(net):
        nets.probe.load_state_dict(net.state_dict())
        return _np(fused(nets.probe, True)[1]).reshape(-1)
    _check_case("scan_encoder_fused + policy_mlp_forward", case, _np(mean), _np(value), _np(pre0), _np(pre1), run)
