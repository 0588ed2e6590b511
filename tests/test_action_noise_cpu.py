"""CPU: the policy's action noise (``normal2`` of ``csrc/rng.cuh``) restated in numpy over ``oracle/philox.py``.

``normal2(seed, step, env)`` = Box-Muller on the first two words of Philox4x32-10 with counter
``(env, step_lo, step_hi, kActionStream)``.  The float64 transcription here is what the GPU tests compare the device's
draw with (within a few ulp: ``logf`` / ``sincospif`` are not correctly rounded); here it is checked to be N(0, 1),
uncorrelated, and keyed apart from the reset path's streams.  The header / export check of ``test_host_cpu`` covers the
new entry points: that is asserted too."""
import os
import re
import sys

import numpy as np
import pytest
from scipy import stats

sys.path.insert(0, os.path.dirname(__file__))

from action_noise_ref import K_ACTION_STREAM, action_counters, normal2_f64  # noqa: E402
from isaac_rover_orbit_b200 import _lib  # noqa: E402
from oracle import philox as PH  # noqa: E402

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
NEW_SYMBOLS = {"rover_policy_act", "rover_policy_act_bf16", "rover_policy_value_act", "rover_action_noise"}


def test_uniforms_avoid_log_of_zero():
    # u1 lies on (0, 1]: the all-zero word maps to 2^-24, the all-one word to exactly 1 (both exact in fp32)
    lo = ((np.uint32(0) >> np.uint32(8)).astype(np.float64) + 1.0) * 2.0 ** -24
    hi = ((np.uint32(0xFFFFFFFF) >> np.uint32(8)).astype(np.float64) + 1.0) * 2.0 ** -24
    assert lo == 2.0 ** -24 and hi == 1.0
    assert np.float32(lo) == lo and np.float32(hi) == hi
    assert np.isfinite(np.sqrt(-2.0 * np.log(lo)))


def test_normal2_is_standard_normal_and_uncorrelated():
    z = normal2_f64(seed=12345, step=7, n=500_000)  # 10^6 draws
    flat = z.reshape(-1)
    assert flat.size == 1_000_000
    ks = stats.kstest(flat, "norm")
    assert ks.pvalue > 1e-3, ks
    for col in (z[:, 0], z[:, 1]):
        assert stats.kstest(col, "norm").pvalue > 1e-3
    assert abs(flat.mean()) < 5e-3 and abs(flat.std() - 1.0) < 5e-3
    r = np.corrcoef(z[:, 0], z[:, 1])[0, 1]
    assert abs(r) < 5e-3, r  # 5 sigma of 1/sqrt(500000)
    # and across neighbouring envs (counter-based: neighbours are independent draws)
    assert abs(np.corrcoef(z[:-1, 0], z[1:, 0])[0, 1]) < 5e-3


def test_draws_do_not_depend_on_batch_size():
    full = normal2_f64(seed=3, step=11, n=4103)
    part = normal2_f64(seed=3, step=11, n=100, env_offset=1000)
    assert np.array_equal(full[1000:1100], part)


@pytest.mark.parametrize("a,b", [((1, 0, 0), (2, 0, 0)),             # seed
                                 ((1, 0, 0), (1, 1, 0)),             # step
                                 ((1, 0, 0), (1, 1 << 32, 0)),       # high word of the step
                                 ((1, 5, 0), (1, 5, 1))])            # env
def test_different_keys_and_counters_differ(a, b):
    (s1, t1, e1), (s2, t2, e2) = a, b
    assert not np.array_equal(normal2_f64(s1, t1, 8, e1), normal2_f64(s2, t2, 8, e2))


def test_action_stream_is_apart_from_the_reset_streams():
    """The reset path uses streams 0 and 1 + q (q < 1024, n_rounds <= 4096) and the spawn key's (0xffffffff, ..,
    0xffffffff) counter; the action stream's counters are none of these, so its words differ from theirs."""
    assert K_ACTION_STREAM not in range(0, 1 + 1024) and K_ACTION_STREAM != 0xFFFFFFFF
    src = open(os.path.join(ROOT, "isaac_rover_orbit_b200", "csrc", "rng.cuh")).read()
    assert int(re.search(r"kActionStream = (0x[0-9a-fA-F]+)u", src).group(1), 16) == K_ACTION_STREAM
    seed, step, n = 99, 4, 64
    key = (seed & 0xFFFFFFFF, seed >> 32)
    act = PH.philox4x32_10(action_counters(step, 0, n), key)
    for stream in (0, 1, 2, 1024):
        assert not np.array_equal(act, PH._env_stream(seed, step, n, stream))
    spawn = PH.philox4x32_10(np.array([[0xFFFFFFFF, step, 0, 0xFFFFFFFF]], dtype=np.uint32), key)
    assert not (act == spawn).all(axis=1).any()


def test_new_symbols_are_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "rover_b200.h")).read()
    declared = set(re.findall(r"\b(rover_[a-z_0-9]+)\s*\(", header))
    assert NEW_SYMBOLS <= declared  # so test_host_cpu's header == exports check covers them
    assert NEW_SYMBOLS <= set(_lib.SYMBOLS)
    assert int(re.search(r"#define ROVER_B200_ABI_VERSION (\d+)", header).group(1)) == _lib.ABI_VERSION == 5
    lib = _lib.load()
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name)
    assert len(lib.rover_policy_act.argtypes) == 11 and len(lib.rover_policy_act_bf16.argtypes) == 11
    assert len(lib.rover_policy_value_act.argtypes) == 13 and len(lib.rover_action_noise.argtypes) == 6


def test_entry_points_reject_bad_arguments_without_a_device():
    """Argument checks run before anything touches a device: NULL, misaligned or out-of-range arguments fail with a
    message in ``rover_last_error``."""
    lib = _lib.load()
    vp = lambda v: None if v is None else __import__("ctypes").c_void_p(v)  # noqa: E731
    a16, a4 = 1 << 20, (1 << 20) + 4
    cases = [
        (lib.rover_policy_act, (vp(a16), 968, 4, None, vp(a16), vp(a16), 0, vp(a16), vp(a16), None, None), "NULL"),
        (lib.rover_policy_act, (vp(a16), 968, 4, vp(a16), vp(a16), vp(a16), -1, vp(a16), vp(a16), None, None), "env_offset"),
        (lib.rover_policy_act, (vp(a16), 968, 4, vp(a16), vp(a16), vp(a4), 0, vp(a16), vp(a16), None, None), "aligned"),
        (lib.rover_policy_act, (vp(a16), 968, 4, vp(a16), vp(a16), vp(a16), 0, vp(a4), vp(a16), None, None), "aligned"),
        (lib.rover_policy_act, (vp(a4), 968, 4, vp(a16), vp(a16), vp(a16), 0, vp(a16), vp(a16), None, None), "16-byte"),
        (lib.rover_policy_act_bf16, (vp(a16), 966, 4, vp(a16), vp(a16), vp(a16), 0, vp(a16), vp(a16), None, None), "stride"),
        (lib.rover_policy_value_act, (vp(a16), 968, 4, vp(a16), None, vp(a16), vp(a16), 0, vp(a16), vp(a16), vp(a16), None,
                                      None), "NULL"),
        (lib.rover_action_noise, (vp(a4), 0, 4, vp(a16), 0, None), "aligned"),
        (lib.rover_action_noise, (vp(a16), -3, 4, vp(a16), 0, None), "env_offset"),
        (lib.rover_action_noise, (vp(a16), 0, -1, vp(a16), 0, None), "negative"),
    ]
    for fn, args, what in cases:
        assert fn(*args) != 0, (fn.__name__, args)
        assert what in lib.rover_last_error().decode(), (fn.__name__, lib.rover_last_error())
    # nothing to do: success without a launch
    assert lib.rover_policy_act(None, 0, 0, None, None, None, 0, None, None, None, None) == 0
