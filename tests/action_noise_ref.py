"""Test support: float64 transcription of ``normal2`` (``isaac_rover_orbit_b200/csrc/rng.cuh``), the policy's action
noise, over ``oracle/philox.py``'s Philox4x32-10."""
import numpy as np

from oracle import philox as PH

K_ACTION_STREAM = 0x80000000


def action_counters(step: int, env_offset: int, n: int) -> np.ndarray:
    ctr = np.zeros((n, 4), dtype=np.uint32)
    ctr[:, 0] = (np.arange(n, dtype=np.uint64) + np.uint64(env_offset)).astype(np.uint32)
    ctr[:, 1] = step & 0xFFFFFFFF
    ctr[:, 2] = (step >> 32) & 0xFFFFFFFF
    ctr[:, 3] = K_ACTION_STREAM
    return ctr


def normal2_f64(seed: int, step: int, n: int, env_offset: int = 0) -> np.ndarray:
    """``[n, 2]`` float64: the device's formula with exact arithmetic after the two fp32-exact uniforms."""
    w = PH.philox4x32_10(action_counters(step, env_offset, n), (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    u1 = ((w[:, 0] >> np.uint32(8)).astype(np.float64) + 1.0) * 2.0 ** -24
    u2 = (w[:, 1] >> np.uint32(8)).astype(np.float64) * 2.0 ** -24
    r = np.sqrt(-2.0 * np.log(u1))
    return np.stack([r * np.cos(2.0 * np.pi * u2), r * np.sin(2.0 * np.pi * u2)], axis=1)
