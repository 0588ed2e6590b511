"""CPU: the pieces of the observation / host-buffer forms of variant 6 that need no GPU.

* ``RayPattern.grid(offset_rot=q)`` rotates the directions with ORBIT's ``quat_apply`` (oracle/orbit_math.py) bit for
  bit and leaves the starts alone; the identity keeps (0, 0, -1) exactly, so the default routing does not change;
* ``RoverEnv``'s ``RayCaster`` passes ``RayCasterCfg.offset_rot``;
* the header, ``_lib.ABI_VERSION`` and the ctypes argument lists of the new entry points agree."""
import math
import os
import re
import types

import numpy as np
import pytest
import torch

from isaac_rover_orbit_b200 import _lib, ops
from isaac_rover_orbit_b200.config import GridPatternCfg, RayCasterCfg
from oracle import orbit_math as OM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bits(t):
    return t.contiguous().view(torch.int32)


def _unit_quats():
    rng = np.random.default_rng(5)
    q = [(1.0, 0.0, 0.0, 0.0), (math.cos(math.radians(5)), 0.0, math.sin(math.radians(5)), 0.0),  # 10 deg pitch
         (math.cos(math.pi / 4), 0.0, 0.0, math.sin(math.pi / 4)), (0.0, 1.0, 0.0, 0.0), (0.5, 0.5, 0.5, 0.5),
         (0.5, -0.5, 0.5, -0.5)]
    for _ in range(6):
        v = rng.standard_normal(4)
        q.append(tuple(float(x) for x in v / np.linalg.norm(v)))
    return q


@pytest.mark.parametrize("direction", [(0.0, 0.0, -1.0), (0.3, 0.1, -1.0), (1.0, 0.0, -1.0)])
@pytest.mark.parametrize("q", _unit_quats())
def test_offset_rot_rotates_directions_with_orbit_quat_apply(q, direction):
    rays = ops.RayPattern.grid("cpu", 0.5, (2.0, 1.0), (0.1, -0.2, 10.0), direction=direction, offset_rot=q)
    n = rays.n_rays
    want = OM.quat_apply(torch.tensor(q, dtype=torch.float32).expand(n, 4),
                         torch.tensor(direction, dtype=torch.float32).expand(n, 3).contiguous())
    assert rays.dirs.dtype == torch.float32 and rays.dirs.shape == (n, 3)
    assert torch.equal(_bits(rays.dirs), _bits(want))
    # the starts are only translated (ORBIT _initialize_rays_impl, SURVEY.md A.3)
    assert torch.equal(_bits(rays.starts), _bits(ops.grid_pattern(0.5, (2.0, 1.0), (0.1, -0.2, 10.0))))
    # and the rotation is the rotation by q (float64 matrix), to fp32 accuracy
    w, x, y, z = q
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                  [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                  [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
    np.testing.assert_allclose(rays.dirs.double().numpy(), np.tile(R @ np.array(direction), (n, 1)), atol=2e-6)


def test_identity_offset_rot_keeps_vertical_down_exactly():
    default = ops.RayPattern.grid("cpu")
    explicit = ops.RayPattern.grid("cpu", offset_rot=(1.0, 0.0, 0.0, 0.0))
    down = torch.tensor([0.0, 0.0, -1.0]).expand(default.n_rays, 3)
    for rays in (default, explicit):
        assert rays.vertical_down
        assert torch.equal(_bits(rays.dirs), _bits(down))  # +0.0, not -0.0, in x and y
    tilted = ops.RayPattern.grid("cpu", offset_rot=(math.cos(math.radians(5)), 0.0, math.sin(math.radians(5)), 0.0))
    assert not tilted.vertical_down


def test_ray_caster_passes_offset_rot():
    from isaac_rover_orbit_b200.env import RayCaster

    env = types.SimpleNamespace(device=torch.device("cpu"))
    assert RayCasterCfg().offset_rot == (1.0, 0.0, 0.0, 0.0)
    assert RayCaster(env, RayCasterCfg()).ray_pattern.vertical_down
    q = (math.cos(math.radians(5)), 0.0, math.sin(math.radians(5)), 0.0)
    sensor = RayCaster(env, RayCasterCfg(offset_rot=q, pattern_cfg=GridPatternCfg(direction=(0.0, 0.1, -1.0))))
    want = ops.RayPattern.grid("cpu", 0.1, (3.0, 3.0), (0.0, 0.0, 10.0), direction=(0.0, 0.1, -1.0), offset_rot=q)
    assert torch.equal(_bits(sensor.ray_pattern.dirs), _bits(want.dirs))
    assert torch.equal(_bits(sensor.ray_pattern.starts), _bits(want.starts))


def _declaration(header, name):
    m = re.search(rf"\bint {name}\s*\((.*?)\);", header, re.S)
    assert m, name
    params = re.sub(r"/\*.*?\*/", "", m.group(1))
    return [p.strip() for p in params.split(",")]


def test_new_entry_points_agree_with_header_and_binding():
    header = open(os.path.join(ROOT, "include", "rover_b200.h")).read()
    assert int(re.search(r"#define ROVER_B200_ABI_VERSION (\d+)", header).group(1)) == _lib.ABI_VERSION == 5
    lib = _lib.load()
    assert lib.rover_abi_version() == 5
    for name in ("rover_ray_cast_obs", "rover_ray_cast_obs_bf16", "rover_ray_cast_host"):
        assert name in _lib.SYMBOLS
        params = _declaration(header, name)
        assert len(getattr(lib, name).argtypes) == len(params), name
        assert params[4].endswith("ray_dirs_local") and params[6].endswith("attach_yaw_only"), name
    # the observation forms take rover_height_scan_obs's arguments without pattern_box, plus directions and frame
    obs = _declaration(header, "rover_height_scan_obs")
    assert [p.split()[-1] for p in _declaration(header, "rover_ray_cast_obs")] == \
        [p.split()[-1] for p in obs[:4] + ["d ray_dirs_local"] + obs[4:5] + ["i attach_yaw_only"] + obs[6:]]
    # the host form: rover_height_scan_host's arguments without pattern_box and variant, plus directions and frame
    host = _declaration(header, "rover_height_scan_host")
    assert [p.split()[-1] for p in _declaration(header, "rover_ray_cast_host")] == \
        [p.split()[-1] for p in host[:4] + ["d ray_dirs_local"] + host[4:5] + ["i attach_yaw_only"] + host[6:15] + host[16:]]
