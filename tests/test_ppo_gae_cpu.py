"""CPU: the references of ``rover_b200::ppo_gae`` (tests/ppo_ref.py) against skrl 1.1.0's ``compute_gae`` transcribed in
torch, and proof that the comparisons the GPU tests make would see the likely defects of a kernel."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))

import ppo_ref as R  # noqa: E402

from isaac_rover_orbit_b200 import _lib, torch_ops  # noqa: E402


def _random_case(T, N, seed, dones="random"):
    rng = np.random.default_rng(seed)
    r = rng.normal(0, 1, (T, N)).astype(np.float32)
    v = rng.normal(0, 3, (T, N)).astype(np.float32)
    last = rng.normal(0, 3, N).astype(np.float32)
    d = {"none": np.zeros((T, N), bool), "all": np.ones((T, N), bool), "random": rng.random((T, N)) < 0.2,
         "first": np.zeros((T, N), bool), "last": np.zeros((T, N), bool)}[dones]
    if dones == "first":
        d[0] = True
    if dones == "last":
        d[-1] = True
    return r, d, v, last


def _torch_loop(r, d, v, last, gamma, lam):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))  # noqa: E731
    ret, adv = R.skrl_gae_loop(t(r)[..., None], t(d)[..., None], t(v)[..., None], t(last)[:, None], gamma, lam)
    return ret[..., 0].numpy(), adv[..., 0].numpy()


def _same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


@pytest.mark.parametrize("T", [1, 2, 60, 257])
@pytest.mark.parametrize("dones", ["none", "all", "random", "first", "last"])
def test_numpy_loop_equals_skrl_torch_loop_bit_for_bit(T, dones):
    r, d, v, last = _random_case(T, 37, seed=T, dones=dones)
    for gamma, lam in ((0.99, 0.95), (1.0, 1.0), (0.5, 0.0)):
        want = _torch_loop(r, d, v, last, gamma, lam)
        got = R.gae_np(r, d, v, last, gamma, lam)
        assert _same_bits(got[0], want[0]) and _same_bits(got[1], want[1]), (gamma, lam)


def test_numpy_loop_keeps_signed_zeros_and_infinities():
    """A done step multiplies by 0: inf * 0 is NaN, and -0 survives where skrl's arithmetic leaves it."""
    T, N = 4, 8
    r = np.zeros((T, N), np.float32)
    v = np.zeros((T, N), np.float32)
    v[:, 1] = -0.0
    r[:, 2] = -0.0
    v[2, 3], v[1, 4], v[3, 5] = np.inf, -np.inf, np.inf
    r[0, 6] = np.inf
    last = np.zeros(N, np.float32)
    last[7], last[1], last[2] = np.inf, -0.0, -1.0
    d = np.zeros((T, N), bool)
    d[3, 2] = True  # -0 - 0 + (gamma * 0) * (-1 + lambda * 0) = -0 + -0
    d[:, 3:] = True
    d[:, 7] = False
    d[3, 7] = True  # the infinite last value meets a done step: inf * 0
    for gamma, lam in ((0.99, 0.95), (1.0, 1.0)):
        want = _torch_loop(r, d, v, last, gamma, lam)
        got = R.gae_np(r, d, v, last, gamma, lam)
        assert _same_bits(got[0], want[0]) and _same_bits(got[1], want[1])
    assert np.isnan(want[1]).any() and np.isinf(want[1]).any() and np.signbit(want[1][want[1] == 0]).any()


EXACT = [(64, 64), (16, 256), (1, 4096), (2, 2048), (4, 1024)]


@pytest.mark.parametrize("T,N", EXACT)
@pytest.mark.parametrize("scale", [1.0, 2.0 ** -10])
def test_normalisation_contract_equals_torch_on_exact_cases(T, N, scale):
    r, d, v, last = R.exact_case(T, N, seed=T * N + 1, scale=scale)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))[..., None]  # noqa: E731
    ret_t, adv_t = R.skrl_compute_gae(t(r), t(d), t(v), t(last), 1.0, 1.0)
    ret, raw = R.gae_np(r, d, v, last, 1.0, 1.0)
    adv, mean_f, std_f = R.normalise_np(raw)
    assert _same_bits(ret, ret_t[..., 0].numpy())
    assert _same_bits(adv, adv_t[..., 0].numpy())
    assert mean_f == np.float32(raw.astype(np.float64).mean()) and np.isfinite(std_f) and std_f > 0


def test_normalisation_of_one_entry_is_nan():
    out, mean_f, std_f = R.normalise_np(np.array([[1.5]], np.float32))
    assert np.isnan(std_f) and np.isnan(out).all() and mean_f == np.float32(1.5)
    with pytest.warns(UserWarning, match="degrees of freedom"):
        assert torch.isnan(torch.tensor([[1.5]]).std())  # torch agrees


# ---- the comparisons see the defects a kernel could have
def _fma_loop(r, d, v, last, gamma, lam):
    """The recurrence with (gamma * nd) * (nv + lambda * adv) + (r - v) contracted into one rounding."""
    nd = np.logical_not(d).astype(np.float32)
    adv = np.zeros(r.shape[1:], np.float32)
    out = np.empty_like(r)
    g, l_ = np.float32(gamma), np.float32(lam)
    for i in reversed(range(r.shape[0])):
        nv = v[i + 1] if i < r.shape[0] - 1 else last
        prod = np.float32(g * nd[i]).astype(np.float64) * np.float32(nv + np.float32(l_ * adv)).astype(np.float64)
        adv = (prod + np.float32(r[i] - v[i]).astype(np.float64)).astype(np.float32)
        out[i] = adv
    return out


def _shifted_dones_loop(r, d, v, last, gamma, lam):
    """not_dones[i + 1] instead of not_dones[i] (the last row reads 'not done')."""
    d2 = np.concatenate([d[1:], np.zeros_like(d[:1])])
    return R.gae_np(r, d2, v, last, gamma, lam)[1]


def test_comparisons_see_recurrence_defects():
    r, d, v, last = _random_case(60, 4103, seed=9)
    _, want = R.gae_np(r, d, v, last, 0.99, 0.95)
    assert not _same_bits(_fma_loop(r, d, v, last, 0.99, 0.95), want)
    assert not _same_bits(_shifted_dones_loop(r, d, v, last, 0.99, 0.95), want)
    # skrl 1.1.0 passes terminated only: a truncated step still bootstraps from the next row
    rng = np.random.default_rng(3)
    truncated = (rng.random(d.shape) < 0.05) & ~d
    assert not _same_bits(R.gae_np(r, d | truncated, v, last, 0.99, 0.95)[1], want)


@pytest.mark.parametrize("T,N", [(64, 64), (1, 4096)])
def test_comparisons_see_normalisation_defects(T, N):
    r, d, v, last = R.exact_case(T, N, seed=5, scale=2.0 ** -10)
    raw = R.gae_np(r, d, v, last, 1.0, 1.0)[1]
    want = R.normalise_np(raw)[0]
    a64 = raw.astype(np.float64)
    mean_f = np.float32(a64.mean())
    m2 = ((a64 - a64.mean()) ** 2).sum()
    biased = np.float32(raw - mean_f) / np.float32(np.float32(np.sqrt(m2 / a64.size)) + np.float32(1e-8))
    eps_inside = np.float32(raw - mean_f) / np.float32(np.sqrt(m2 / (a64.size - 1) + 1e-8))
    assert not _same_bits(biased, want)
    assert not _same_bits(eps_inside, want)


def test_operator_and_symbols_are_declared():
    assert "ppo_gae" in torch_ops.OPS
    assert {"rover_ppo_gae", "rover_ppo_gae_work_bytes"} <= set(_lib.SYMBOLS)
    assert _lib.ABI_VERSION == 5


def test_operator_has_no_cpu_implementation():
    z = torch.zeros(4, 3, 1)
    with pytest.raises(RuntimeError):
        torch.ops.rover_b200.ppo_gae(z, z.bool(), z, z[0], 0.99, 0.95, torch.empty_like(z), torch.empty_like(z))


def test_work_bytes():
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import __graft_entry__

    __graft_entry__.build()
    lib = _lib.load()
    assert lib.rover_ppo_gae_work_bytes(0, 5) == 0 and lib.rover_ppo_gae_work_bytes(-1, 5) == -1
    assert lib.rover_ppo_gae_work_bytes(60, 16384) == 8 * (128 + 592)
    assert lib.rover_ppo_gae_work_bytes(1, 1) == 16
