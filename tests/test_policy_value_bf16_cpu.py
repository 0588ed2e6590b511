"""CPU: the C ABI of the two-network pass over the bf16 observation (``rover_policy_value_forward_bf16``,
``rover_policy_value_act_bf16``): declared, exported, typed, an additive change (ABI version 5), and its argument checks
fail before anything touches a device."""
import ctypes
import os
import re

from isaac_rover_orbit_b200 import _lib

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
NEW_SYMBOLS = {"rover_policy_value_forward_bf16", "rover_policy_value_act_bf16"}


def test_new_symbols_are_declared_exported_and_typed():
    header = open(os.path.join(ROOT, "include", "rover_b200.h")).read()
    declared = set(re.findall(r"\b(rover_[a-z_0-9]+)\s*\(", header))
    assert NEW_SYMBOLS <= declared
    assert NEW_SYMBOLS <= set(_lib.SYMBOLS)
    assert int(re.search(r"#define ROVER_B200_ABI_VERSION (\d+)", header).group(1)) == _lib.ABI_VERSION == 5
    lib = _lib.load()
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name)
    # the argument lists of the fp32 entry points, with a bf16 observation
    assert len(lib.rover_policy_value_forward_bf16.argtypes) == len(lib.rover_policy_value_forward.argtypes) == 8
    assert len(lib.rover_policy_value_act_bf16.argtypes) == len(lib.rover_policy_value_act.argtypes) == 13
    for name in NEW_SYMBOLS:
        assert getattr(lib, name).restype is ctypes.c_int


def test_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    vp = lambda v: None if v is None else ctypes.c_void_p(v)  # noqa: E731
    a, a4, a8 = 1 << 20, (1 << 20) + 4, (1 << 20) + 8
    fwd = lib.rover_policy_value_forward_bf16
    act = lib.rover_policy_value_act_bf16
    cases = [
        (fwd, (vp(a), 968, -1, vp(a), vp(a), vp(a), vp(a), None), "negative"),
        (fwd, (vp(a), 968, 4, vp(a), None, vp(a), vp(a), None), "NULL"),
        (fwd, (vp(a), 968, 4, vp(a), vp(a), vp(a), None, None), "NULL"),
        (fwd, (vp(a), 965, 4, vp(a), vp(a), vp(a), vp(a), None), "stride"),    # unpadded rows
        (fwd, (vp(a), 960, 4, vp(a), vp(a), vp(a), vp(a), None), "stride"),    # fewer than 965 columns
        (fwd, (vp(a8), 968, 4, vp(a), vp(a), vp(a), vp(a), None), "16-byte"),  # rows not 16-byte aligned
        (fwd, (vp(a), 968, 4, vp(a4), vp(a), vp(a), vp(a), None), "128B"),
        (fwd, (vp(a), 968, 4, vp(a), vp(a + 64), vp(a), vp(a), None), "128B"),
        (act, (vp(a), 968, -1, vp(a), vp(a), vp(a), vp(a), 0, vp(a), vp(a), vp(a), None, None), "negative"),
        (act, (vp(a), 968, 4, vp(a), None, vp(a), vp(a), 0, vp(a), vp(a), vp(a), None, None), "NULL"),
        (act, (vp(a), 968, 4, vp(a), vp(a), vp(a), vp(a), 0, vp(a), None, vp(a), None, None), "NULL"),
        (act, (vp(a), 968, 4, vp(a), vp(a), vp(a), vp(a), -1, vp(a), vp(a), vp(a), None, None), "env_offset"),
        (act, (vp(a), 968, 4, vp(a), vp(a), vp(a), vp(a4), 0, vp(a), vp(a), vp(a), None, None), "aligned"),
        (act, (vp(a), 968, 4, vp(a), vp(a), vp(a), vp(a), 0, vp(a4), vp(a), vp(a), None, None), "aligned"),
        (act, (vp(a), 966, 4, vp(a), vp(a), vp(a), vp(a), 0, vp(a), vp(a), vp(a), None, None), "stride"),
        (act, (vp(a), 968, 4, vp(a4), vp(a), vp(a), vp(a), 0, vp(a), vp(a), vp(a), None, None), "128B"),
        (act, (vp(a), 968, 4, vp(a), vp(a + 64), vp(a), vp(a), 0, vp(a), vp(a), vp(a), None, None), "128B"),
    ]
    for fn, args, what in cases:
        assert fn(*args) != 0, (fn.__name__, args)
        assert what in lib.rover_last_error().decode(), (fn.__name__, what, lib.rover_last_error())
    # nothing to do: success without a launch
    assert fwd(None, 0, 0, None, None, None, None, None) == 0
    assert act(None, 0, 0, None, None, None, None, 0, None, None, None, None, None) == 0
