"""CPU: the width-general reference of policy_width_exact.py equals policy_exact.py's at R = 961 bit for bit and would see
each layer-0 defect a run-time chunk count can make; the new export, its struct and the width checks agree across the
header, the library and ctypes."""
import ctypes
import os
import re
import subprocess
import types

import numpy as np
import pytest

import policy_exact as PE
import policy_width_exact as PW
from isaac_rover_orbit_b200 import _lib, torch_ops

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__

    __graft_entry__.build()


def _bits(x):
    return np.asarray(x, np.float32).view(np.int32)


@pytest.mark.parametrize("family,seed", [("dense", 11), ("sparse", 12)])
def test_general_model_is_policy_exact_at_961(family, seed):
    case = PE.make_case(1500, family, seed)
    general = PW.make_case(1500, 961, family, seed)
    assert np.array_equal(_bits(general.obs), _bits(case.obs))
    for net, gnet, ref in ((case.policy, general.policy, case.ref_policy), (case.value, general.value, case.ref_value)):
        assert all(np.array_equal(a, b) for a, b in zip(net.w + net.b, gnet.w + gnet.b))
        got = PW.forward(case.obs, net, 961)
        want = PE.forward(case.obs, net)
        for a, b, c in zip(got["pre"], want["pre"], ref["pre"]):
            assert np.array_equal(_bits(a), _bits(b)) and np.array_equal(_bits(a), _bits(c))


@pytest.mark.parametrize("r", [1, 62, 256, 3721])
def test_general_cases_certify_in_any_summation_order(r):
    case = PW.make_case(200, r, "dense", seed=r)
    x = PW.encoder_input(case.obs, r)
    w = case.policy.w[0].astype(np.float32)
    g = np.random.default_rng(r)
    for block in (1, 16, 64):
        perm = g.permutation(r)
        acc = np.zeros((case.n, 80), np.float32)
        for k0 in range(0, r, block):
            k = perm[k0:k0 + block]
            acc = acc + x[:, k] @ w[:, k].T
        assert np.array_equal(_bits(acc + case.policy.b[0].astype(np.float32)), _bits(case.ref_policy["pre"][0]))


def _detected(case, defect):
    hits = 0
    for net, ref in ((case.policy, case.ref_policy), (case.value, case.ref_value)):
        v = PW.forward(case.obs, net, case.r, defect=defect)
        hits += int((_bits(v["out"]) != _bits(ref["out"])).sum())
    return hits


@pytest.mark.parametrize("defect,r", [("shift", 81), ("shift", 3721), ("last_col", 81), ("last_col", 1681),
                                      ("tail_k", 61), ("tail_k", 62), ("tail_k", 1021), ("tail_k", 1022),
                                      ("chunk_short", 61), ("chunk_short", 62), ("chunk_short", 1021),
                                      ("chunk_short", 1022), ("chunk_short", 256)])
def test_planted_defects_change_an_output_bit(defect, r):
    # the dense family: every unit reads every column (a sparse unit reads 1..4 of them and may miss the one that moved)
    case = PW.make_case(257, r, "dense", seed=3 * r + 1)
    assert _detected(case, defect) > 0


def test_chunk_counts_step_where_the_tests_look():
    # R = 61 / 62 and 1021 / 1022: ceil((3 + R) / 64) steps (1 -> 2, 16 -> 17); the fp32 32-column count steps there too
    for r0, r1 in ((61, 62), (1021, 1022), (125, 126)):
        assert (3 + r0 + 63) // 64 + 1 == (3 + r1 + 63) // 64
        assert (3 + r0 + 31) // 32 + 1 == (3 + r1 + 31) // 32
    assert PW.tail_start(62) == 61 and PW.tail_start(61) == 0 and PW.tail_start(961) == 15 * 64 - 3


def test_header_lib_and_ctypes_agree_on_the_pass(tmp_path):
    header = open(os.path.join(ROOT, "include", "rover_b200.h")).read()
    assert re.search(r"\bint rover_policy_pass\s*\(const RoverPolicyPass\* pass", header)
    assert "rover_policy_pass" in _lib.SYMBOLS
    lib = _lib.load()
    assert lib.rover_policy_pass.argtypes == [ctypes.POINTER(_lib.PolicyPass), ctypes.c_void_p]
    assert lib.rover_policy_pass.restype == ctypes.c_int
    fields = re.search(r"typedef struct RoverPolicyPass \{(.*?)\} RoverPolicyPass;", header, re.S).group(1)
    names = re.findall(r"\**(\w+);", re.sub(r"/\*.*?\*/", "", fields, flags=re.S))
    assert names == [f[0] for f in _lib.PolicyPass._fields_]
    src = tmp_path / "sz.c"
    offs = "".join(f'printf("%zu ", offsetof(RoverPolicyPass, {n}));' for n in names)
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "rover_b200.h"\nint main(void){'
                   f'printf("%zu ", sizeof(RoverPolicyPass));{offs}'
                   'printf("%d %d", ROVER_OBS_FP32, ROVER_OBS_BF16);return 0;}')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.PolicyPass)
    assert out[1:-2] == [getattr(_lib.PolicyPass, n).offset for n in names]
    assert out[-2:] == [_lib.OBS_FP32, _lib.OBS_BF16]
    assert "policy_pass" in torch_ops.OPS


@pytest.mark.parametrize("bad", [0, -1, 4093, 10 ** 6, 2.5])
def test_out_of_range_width_is_rejected(bad):
    with pytest.raises(ValueError, match="outside"):
        _lib.check_enc_in(bad)
    with pytest.raises(ValueError, match="outside"):
        torch_ops.policy_packed_bytes(bad)
    from isaac_rover_orbit_b200.policy import DeterministicNeuralNetwork, GaussianNeuralNetwork

    for cls in (GaussianNeuralNetwork, DeterministicNeuralNetwork):
        with pytest.raises(ValueError, match="outside"):
            cls(encoder_input_size=bad)


def test_pack_rejects_out_of_range_width_in_c():
    w = _lib.PolicyWeights()
    for bad in (0, 4093):
        w.in_dim[0] = bad
        assert _lib.load().rover_policy_pack(ctypes.byref(w), None, None) == -1
        assert b"outside [1, 4092]" in _lib.load().rover_last_error()


def test_blob_layout_by_width():
    base = torch_ops.policy_packed_bytes()
    assert torch_ops.policy_packed_bytes(961) == base == int(_lib.load().rover_policy_pack(None, None, None))
    for r in (1, 61, 62, 960, 961, 1021, 1022, 4092):
        assert torch_ops.policy_packed_bytes(r) == base + ((3 + r + 63) // 64 - 16) * 10240, r
    assert _lib.check_enc_in(1) == 1 and _lib.check_enc_in(4092) == 4092


def test_rollout_agents_size_states_from_the_policy():
    from isaac_rover_orbit_b200.trainer import PPORolloutAgent, RolloutAgent, RolloutMemory

    for r, cols in ((256, 260), (961, 965), (3721, 3725)):
        mem = RolloutMemory(memory_size=2, num_envs=3, device="cpu")
        RolloutAgent(types.SimpleNamespace(encoder_input_size=r), mem)
        assert mem.get_tensor_by_name("states").shape[-1] == cols
        mem = RolloutMemory(memory_size=2, num_envs=3, device="cpu")
        PPORolloutAgent(types.SimpleNamespace(encoder_input_size=r), object(), mem)
        assert mem.get_tensor_by_name("states").shape[-1] == cols
    mem = RolloutMemory(memory_size=2, num_envs=3, device="cpu")
    PPORolloutAgent(types.SimpleNamespace(encoder_input_size=256), object(), mem, observation_size=12)
    assert mem.get_tensor_by_name("states").shape[-1] == 12
    mem = RolloutMemory(memory_size=2, num_envs=3, device="cpu")
    RolloutAgent(types.SimpleNamespace(), mem)  # a policy without an encoder width: the shipped 965 columns
    assert mem.get_tensor_by_name("states").shape[-1] == 965
