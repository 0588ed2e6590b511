"""CPU: the lattice cases of policy_exact.py are exact (certificate, fp32 sums in any order), the float64 reference equals
the torch emulation of the kernels' numerics bit for bit, and the comparisons the GPU tests make would see each of a list
of one-line numeric defects."""
import numpy as np
import pytest
import torch

import policy_exact as PE
from test_gpu_policy import emulate_bf16, emulate_value_bf16


@pytest.fixture(scope="module")
def cases():
    return {fam: PE.make_case(1500, fam, seed) for fam, seed in (("dense", 11), ("sparse", 12))}


def _layer_inputs(case, ref):
    x = [PE.bf16(case.obs[:, 3:964]), ref["act"][0], np.concatenate([PE.bf16(case.obs[:, 0:4]), ref["act"][1]], axis=1)]
    return x + ref["act"][2:5]


def test_bf16_rounding_is_round_to_nearest_even():
    g = np.random.default_rng(0)
    m = g.integers(128, 256, size=4096)
    x = ((2 * m + 1) * 2.0 ** -5 + g.integers(-1, 2, size=4096) * 2.0 ** -20) * g.choice([-1, 1], size=4096)
    x = np.concatenate([x, g.standard_normal(4096) * 100]).astype(np.float32)
    want = torch.from_numpy(x).to(torch.bfloat16).float().numpy()  # torch: RNE
    assert np.array_equal(PE.bf16(x).view(np.int32), want.view(np.int32))
    ties = PE.bf16(np.float32([257 * 2.0 ** -5, 259 * 2.0 ** -5]))  # 8.03125 -> 8.0 (even), 8.09375 -> 8.125 (even)
    assert ties.tolist() == [8.0, 8.125]
    assert PE.bf16(np.float32([8.09375]), rz=True).tolist() == [8.0625]


@pytest.mark.parametrize("family", ["dense", "sparse"])
def test_cases_are_certified_and_fp32_sums_are_order_free(cases, family):
    case = cases[family]
    for net, ref in ((case.policy, case.ref_policy), (case.value, case.ref_value)):
        again = PE.forward(case.obs, net)  # certifies every layer again
        assert all(np.array_equal(a.view(np.int32), b.view(np.int32)) for a, b in zip(again["pre"], ref["pre"]))
        if family == "dense":
            assert all(bool((s > 0).all()) for s in ref["pre"][:5])
        else:
            assert all(0.3 < float((s < 0).mean()) < 0.7 for s in ref["pre"][:5])
        g = np.random.default_rng(5)
        for l, x in enumerate(_layer_inputs(case, ref)):
            w32, b32 = net.w[l].astype(np.float32), net.b[l].astype(np.float32)
            assert np.array_equal(w32, net.w[l]) and np.array_equal(PE.bf16(w32), w32)  # weights are bf16 values
            for block in (1, 7, 16, 64, x.shape[1]):
                perm = g.permutation(x.shape[1])
                acc = np.zeros((x.shape[0], w32.shape[0]), np.float32)
                for k0 in range(0, x.shape[1], block):
                    k = perm[k0:k0 + block]
                    acc = acc + x[:, k] @ w32[:, k].T  # fp32 products and sums
                acc = acc + b32
                assert np.array_equal(acc.view(np.int32), ref["pre"][l].view(np.int32)), (l, block)


@pytest.mark.parametrize("family", ["dense", "sparse"])
def test_reference_equals_torch_emulation_bitwise(cases, family):
    """The float64 reference and ``emulate_bf16`` / ``emulate_value_bf16`` (test_gpu_policy.py: fp32 torch on the CPU)
    agree bit for bit on certified cases: pre-activations of both networks, and the policy's tanh."""
    case = cases[family]
    obs = torch.from_numpy(case.obs)
    for net, ref in ((case.policy, case.ref_policy), (case.value, case.ref_value)):
        emu = emulate_value_bf16(obs, net.state_dict()).numpy()
        assert np.array_equal(emu.view(np.int32), ref["out"].view(np.int32))
    mean = emulate_bf16(obs, case.policy.state_dict())
    assert torch.equal(mean, torch.tanh(torch.from_numpy(case.ref_policy["out"])))
    assert PE.ulp_distance(mean.numpy(), PE.mean_of(case.ref_policy["out"])).max() <= 2


def _detected(case, defect):
    """What the GPU tests compare: value and pre-activations bitwise, the mean to 2 ulp of tanh of the pre-activation."""
    hits = 0
    for net, ref in ((case.policy, case.ref_policy), (case.value, case.ref_value)):
        v = PE.forward(case.obs, net, defect=defect)
        hits += int((v["out"].view(np.int32) != ref["out"].view(np.int32)).sum())
    hits += int((PE.ulp_distance(PE.mean_of(case.ref_policy["out"], defect), PE.mean_of(case.ref_policy["out"])) > 2).sum())
    return hits


@pytest.mark.parametrize("defect", PE.DEFECTS)
def test_comparisons_see_each_defect(cases, defect):
    """Each one-line defect changes at least one output bit on the generated cases (the 0.01f branch only exists in the
    sparse family; everything else shows on both or on the dense one)."""
    found = {fam: _detected(case, defect) for fam, case in cases.items()}
    assert sum(found.values()) > 0, found
    if defect == "slope_bf16":
        assert found["sparse"] > 0
    elif defect != "tanh_approx":
        assert found["dense"] > 0, found
    if defect in ("slope_bf16", "bias_bf16", "act_rz"):  # the epilogue defects: visible on the 0.01f branch too
        assert found["sparse"] > 0, found


def test_certificate_rejects_non_lattice_cases(cases, golden_dir):
    import os

    from oracle import policy as OP

    sd = OP.load_golden_weights(np.load(os.path.join(golden_dir, "policy.npz")))
    keys = [k for k in sd if k.endswith(".weight")]
    net = PE.Net([np.asarray(sd[k], np.float64) for k in keys], [np.asarray(sd[k[:-7] + ".bias"], np.float64) for k in keys])
    with pytest.raises(PE.CertificateError, match="layer 0"):
        PE.forward(cases["dense"].obs[:64], net)
    # one lattice case with a single weight moved off the lattice by a low bit
    case = cases["dense"]
    w = [t.copy() for t in case.policy.w]
    w[3][7, 11] += 2.0 ** -30 * np.sign(w[3][7, 11] or 1.0)
    with pytest.raises(PE.CertificateError, match="layer 3"):
        PE.forward(case.obs, PE.Net(w, case.policy.b))
