"""GPU: every ray of every height-scan entry point bit for bit against the numpy model (tests/scan_exact.py).

Ray patterns of 1 to 1025 rays (1 to 4 chunks of 256 per environment, each with more than 8 environments per CTA, partial 128-ray batches, per-ray z, off-centre,
shuffled, wider than a staged window), terrains with exact and rounded arithmetic, holes, general cells, more lines than
the shared tables hold, cells too small for a window and a narrow strip; poses on lattice lines and vertices, on the far
border and one ulp beyond it, with t == max_d and non-finite values; environment counts from 1 to 148 * 33.  The only
tolerance is the bound on the ray start for yaws whose sinf / cosf the host cannot reproduce."""
import numpy as np
import pytest
import torch

from isaac_rover_orbit_b200 import ops, synthetic
from isaac_rover_orbit_b200 import terrain as TR
from isaac_rover_orbit_b200.config import RoverEnvCfg
from isaac_rover_orbit_b200.policy import alloc_obs
import scan_exact as SE

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
F32 = np.float32
U = 2.0 ** -24


def _heightfield(nx, ny, d, seed, holes=False, rocks=False):
    rng = np.random.default_rng(seed)
    xs, ys = np.arange(nx + 1) * d, np.arange(ny + 1) * d
    X, Y = np.meshgrid(xs, ys)
    Z = 0.3 * np.sin(0.7 * X) * np.cos(0.9 * Y) + 0.05 * rng.standard_normal(X.shape)
    v = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32)
    i, j = np.meshgrid(np.arange(nx), np.arange(ny))
    a = (j * (nx + 1) + i).ravel()
    keep = np.ones(len(a), bool)
    if holes:
        keep = rng.random(len(a)) > 0.05
    f = [np.stack([a, a + 1, a + nx + 2], 1)[keep], np.stack([a, a + nx + 2, a + nx + 1], 1)[keep]]
    if rocks:  # pyramids over 2 x 2 cells with the apex on the lattice vertex in their middle: general cells
        extra = []
        for k in range(40):
            ci, cj = rng.integers(2, nx - 2), rng.integers(2, ny - 2)
            c = len(v) + len(extra)
            extra.append([ci * d, cj * d, 0.6])
            ring = [(cj - 1) * (nx + 1) + ci - 1, (cj - 1) * (nx + 1) + ci + 1, (cj + 1) * (nx + 1) + ci + 1, (cj + 1) * (nx + 1) + ci - 1]
            f.append(np.array([[ring[q], ring[(q + 1) % 4], c] for q in range(4)]))
        v = np.concatenate([v, np.array(extra, np.float32)])
    return v, np.concatenate(f).astype(np.int32)


_TERRAINS = {}


def terrain(name, dev):
    if name not in _TERRAINS:
        if name == "dyadic":
            xs, ys, H, diag = SE.dyadic_case("uniform")
            v, f = SE.dyadic_lattice(xs, ys, H, diag)
        elif name == "dyadic_nonuniform":
            xs, ys, H, diag = SE.dyadic_case("nonuniform")
            v, f = SE.dyadic_lattice(xs, ys, H, diag)
        elif name == "random":
            v, f = TR.make_synthetic_terrain(24.0, 0.2, seed=3)
        elif name == "holes":
            v, f = _heightfield(100, 100, 0.2, 1, holes=True)
        elif name == "rocks":
            v, f = _heightfield(100, 100, 0.2, 2, rocks=True)
        elif name == "many_lines":
            v, f = _heightfield(1100, 24, 0.2, 3)
        elif name == "small_cells":
            v, f = _heightfield(300, 300, 0.05, 4)
        elif name == "strip":
            v, f = _heightfield(200, 9, 0.2, 5)
        g = ops.ScanGridHandle.from_mesh(v, f, dev)
        g.ensure_home_grid()
        _TERRAINS[name] = g
    return _TERRAINS[name]


def pattern(r, kind="flat"):
    cols = int(np.ceil(np.sqrt(r)))
    k = np.arange(r)
    spacing = 0.5 if kind == "wide" else 0.1
    p = np.zeros((r, 3), F32)
    p[:, 0] = ((k % cols) - (cols - 1) / 2.0) * spacing
    p[:, 1] = ((k // cols) - (cols - 1) / 2.0) * spacing
    p[:, 2] = 10.0
    p[r // 2, :2] = 0.0  # a ray exactly at the sensor position
    if kind == "zvar":
        p[1::3, 2] = np.nextafter(F32(10.0), F32(11.0))  # one ulp above vz[0]
        p[2::5, 2] = 9.5
    elif kind == "offcentre":
        p[:, 0] += 0.7
        p[:, 1] -= 0.4
    elif kind == "shuffled":
        p = p[np.random.default_rng(r).permutation(r)]
    return p.astype(F32)


def exact_poses(g, n, seed, edges=True):
    """Poses whose frame is exact (identity-like quaternions), some on lattice lines / vertices / borders, t edges."""
    rng = np.random.default_rng(seed)
    xs, ys = g.cells.xs.cpu().numpy(), g.cells.ys.cpu().numpy()
    px = rng.uniform(xs[0] - 1.0, xs[-1] + 1.0, n)
    py = rng.uniform(ys[0] - 1.0, ys[-1] + 1.0, n)
    pz = rng.uniform(0.5, 2.0, n)
    quat = np.zeros((n, 4), F32)
    quat[:, 0] = 1.0
    kinds = rng.integers(0, 5, n)
    quat[kinds == 1] = (-1, 0, 0, 0)
    quat[kinds == 2] = (np.cos(0.2), np.sin(0.2), 0, 0)  # roll
    quat[kinds == 3] = (np.cos(0.5), 0, np.sin(0.5), 0)  # pitch < 90 degrees
    quat[kinds == 4] = 0.0
    pos = np.stack([px, py, pz], 1).astype(F32)
    if edges and n >= 12:
        pos[0, :2] = xs[len(xs) // 2], ys[len(ys) // 3]  # a vertex
        pos[1, 0] = xs[3]                                # an x line
        pos[2, :2] = xs[-1], ys[-1]                      # the far corner
        pos[3, 0] = np.nextafter(xs[-1], F32(np.inf))    # one ulp outside
        pos[4, 1] = np.nextafter(ys[0], F32(-np.inf))
        pos[5, 0] = np.nan
        pos[6, 2] = np.inf
        quat[7] = (np.nan, 0, 0, 0)
        quat[8] = (np.inf, 0, 0, 0)
        pos[9, 0] = -np.inf
    return pos, quat


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)


def assert_exact(where, got, m: SE.ScanResult, want=None):
    got = np.asarray(got, np.float32)
    want = m.h if want is None else want
    bad = np.nonzero(_bits(got) != _bits(want))
    if len(bad[0]):
        e, r = bad[0][0], bad[1][0]
        raise AssertionError(
            f"{where}: {len(bad[0])} rays differ; first env {e} ray {r}: X={m.X[e, r]!r} Y={m.Y[e, r]!r} "
            f"cell={tuple(m.cell[e, r])} tag={m.tag[e, r]} path={SE.PATHS[m.path[e, r]]} "
            f"kernel={got[e, r]!r} ({_bits(got)[e, r]:#010x}) model={want[e, r]!r} ({_bits(want)[e, r]:#010x})")


def _model(g, pos, quat, pat, variant=5, **kw):
    if variant == 0:
        return SE.scan_model(pos, quat, pat, None, g.grid, home_only=True, **kw)
    return SE.scan_model(pos, quat, pat, g.cells, g.grid, **kw)


RAYS = [1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512, 513, 767, 768, 769, 961, 1023, 1024, 1025]


@pytest.mark.parametrize("r", RAYS)
def test_height_scan_variants_every_ray_count(cuda_device, r):
    """Variants 0, 2, 4, 5 on the dyadic and the random terrain, heights and hit positions."""
    pat = pattern(r)
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    for name in ("dyadic", "random"):
        g = terrain(name, cuda_device)
        n = 149 if r <= 256 else 37
        pos, quat = exact_poses(g, n, seed=r)
        P, Q = torch.from_numpy(pos).to(cuda_device), torch.from_numpy(quat).to(cuda_device)
        for variant in (0, 2, 4, 5):
            m = _model(g, pos, quat, pat, variant)
            h = ops.height_scan(P, Q, rays, g, variant=variant).cpu().numpy()
            assert_exact(f"height_scan v{variant} {name} R={r}", h, m)
            if variant in (2, 4, 5):
                h2, hits = ops.height_scan(P, Q, rays, g, variant=variant, return_hits=True)
                assert_exact(f"height_scan v{variant} return_hits {name} R={r}", h2.cpu().numpy(), m)
                assert np.array_equal(_bits(hits.cpu().numpy()), _bits(m.hits)), f"hits v{variant} {name} R={r}"


@pytest.mark.parametrize("kind", ["zvar", "offcentre", "shuffled", "wide"])
@pytest.mark.parametrize("r", [129, 256, 961])
def test_height_scan_pattern_kinds(cuda_device, kind, r):
    pat = pattern(r, kind)
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    for name in ("dyadic_nonuniform", "random"):
        g = terrain(name, cuda_device)
        pos, quat = exact_poses(g, 64, seed=7 + r)
        P, Q = torch.from_numpy(pos).to(cuda_device), torch.from_numpy(quat).to(cuda_device)
        m = _model(g, pos, quat, pat)
        for variant in (2, 4, 5):
            assert_exact(f"v{variant} {kind} {name} R={r}", ops.height_scan(P, Q, rays, g, variant=variant).cpu().numpy(), m)


@pytest.mark.parametrize("name", ["holes", "rocks", "many_lines", "small_cells", "strip"])
@pytest.mark.parametrize("r", [200, 961])
def test_height_scan_terrain_kinds(cuda_device, name, r):
    g = terrain(name, cuda_device)
    if name == "rocks":
        assert g.cells.n_general > 0
    pat = pattern(r)
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    pos, quat = exact_poses(g, 96, seed=11 + r)
    P, Q = torch.from_numpy(pos).to(cuda_device), torch.from_numpy(quat).to(cuda_device)
    for variant in (0, 2, 4, 5):
        m = _model(g, pos, quat, pat, variant)
        assert_exact(f"v{variant} {name} R={r}", ops.height_scan(P, Q, rays, g, variant=variant).cpu().numpy(), m)


def test_height_scan_max_distance_and_base_offset(cuda_device):
    """t == 0, t == max_d (a miss), max_d - ulp, and a base offset other than the default, on exact arithmetic."""
    g = terrain("dyadic", cuda_device)
    pat = pattern(64)
    pos, quat = exact_poses(g, 48, seed=5, edges=False)
    m0 = _model(g, pos, quat, pat)
    t = (m0.Z - m0.hits[..., 2])[np.isfinite(m0.h)]
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    P, Q = torch.from_numpy(pos).to(cuda_device), torch.from_numpy(quat).to(cuda_device)
    for max_d in (float(t.max()), float(np.nextafter(F32(t.max()), F32(0))), float(np.nextafter(F32(t.max()), F32(np.inf))),
                  float(np.median(t))):
        for base in (0.26878, 0.0, -1.5):
            m = _model(g, pos, quat, pat, max_distance=max_d, base_offset=base)
            for variant in (0, 2, 4, 5):
                mm = _model(g, pos, quat, pat, variant, max_distance=max_d, base_offset=base) if variant == 0 else m
                h = ops.height_scan(P, Q, rays, g, max_distance=max_d, base_offset=base, variant=variant).cpu().numpy()
                assert_exact(f"v{variant} max_d={max_d} base={base}", h, mm)
    # t == 0: the sensor exactly on the surface (z of the start = surface height)
    pos0 = pos.copy()
    pos0[:, 2] = np.where(np.isfinite(m0.h[:, 32]), m0.hits[:, 32, 2] - pat[32, 2], pos0[:, 2])
    m = _model(g, pos0, quat, pat)
    assert (m.Z[:, 32] == m.hits[:, 32, 2]).any()
    h = ops.height_scan(torch.from_numpy(pos0).to(cuda_device), Q, rays, g, variant=5).cpu().numpy()
    assert_exact("v5 t == 0", h, m)


@pytest.mark.parametrize("n", [1, 16, 17, 147, 148, 149, 148 * 8 + 3, 148 * 33])
@pytest.mark.parametrize("r", [1, 64, 256])
def test_height_scan_env_counts_small_patterns(cuda_device, n, r):
    """One chunk per environment: the deal moves a consumer warp 15 environments at a time (the ring-barrier phase)."""
    g = terrain("random", cuda_device)
    pat = pattern(r, "offcentre" if r == 64 else "flat")
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    pos, quat = exact_poses(g, n, seed=n + r)
    P, Q = torch.from_numpy(pos).to(cuda_device), torch.from_numpy(quat).to(cuda_device)
    m = _model(g, pos, quat, pat)
    for variant in (4, 5):
        assert_exact(f"v{variant} n={n} R={r}", ops.height_scan(P, Q, rays, g, variant=variant).cpu().numpy(), m)
    head = 4
    obs = torch.full((n, head + r + 3), 7.0, device=cuda_device)
    obs_bf = torch.full((n, head + r + 3), 9.0, dtype=torch.bfloat16, device=cuda_device)
    ops.height_scan_obs(P, Q, rays, g, obs, obs_bf, head_cols=head)
    assert_exact(f"height_scan_obs n={n} R={r}", obs[:, head:head + r].cpu().numpy(), m)


@pytest.mark.parametrize("r,n,kind", [(257, 148 * 9 + 3, "flat"), (513, 148 * 9 + 3, "flat"), (769, 148 * 9 + 3, "zvar"),
                                      (257, 148 * 33, "shuffled")])
def test_height_scan_multi_chunk_many_envs(cuda_device, r, n, kind):
    """2, 3 and 4 chunks of 256 rays per environment with more than 8 environments per CTA: consumer warps advance by
    step_it / step_c with the chunk carry, the 8-stage ring wraps and the producer waits on `empty` barriers that count
    n_chunks arrivals."""
    g = terrain("random", cuda_device)
    pat = pattern(r, kind)
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    pos, quat = exact_poses(g, n, seed=n + r)
    P, Q = torch.from_numpy(pos).to(cuda_device), torch.from_numpy(quat).to(cuda_device)
    m = _model(g, pos, quat, pat)
    for variant in (4, 5):
        assert_exact(f"v{variant} n={n} R={r}", ops.height_scan(P, Q, rays, g, variant=variant).cpu().numpy(), m)
    head = 4
    obs = torch.full((n, head + r + 3), 7.0, device=cuda_device)
    obs_bf = torch.full((n, head + r + 3), 9.0, dtype=torch.bfloat16, device=cuda_device)
    ops.height_scan_obs(P, Q, rays, g, obs, obs_bf, head_cols=head)
    torch.cuda.synchronize()
    assert_exact(f"height_scan_obs n={n} R={r}", obs[:, head:head + r].cpu().numpy(), m)
    assert torch.equal(obs_bf[:, :head + r].cpu(), obs[:, :head + r].cpu().to(torch.bfloat16))


@pytest.mark.parametrize("r", [1, 64, 256, 257, 961, 1024])
@pytest.mark.parametrize("head", [0, 4, 32])
@pytest.mark.parametrize("path", ["fused", "fallback"])
def test_height_scan_obs_exact(cuda_device, r, head, path):
    g = terrain("random", cuda_device)
    pat = pattern(r, "zvar" if r == 257 else "flat")
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    n = 150
    pos, quat = exact_poses(g, n, seed=3 * r + head)
    P, Q = torch.from_numpy(pos).to(cuda_device), torch.from_numpy(quat).to(cuda_device)
    m = _model(g, pos, quat, pat)
    gen = torch.Generator().manual_seed(r)
    width = head + r + 5
    saved = g.cells_struct.entries_planar
    if path == "fallback":
        g.cells_struct.entries_planar = None
    try:
        for bf16_only in (False, True) if path == "fused" else (False,):
            obs = torch.full((n, width), 7.0)
            obs[:, :head] = torch.randn(n, head, generator=gen)
            obs = obs.to(cuda_device)
            before = obs.clone()
            obs_bf = torch.full((n, width), 9.0, dtype=torch.bfloat16, device=cuda_device)
            ops.height_scan_obs(P, Q, rays, g, obs[:, :head + r], obs_bf[:, :head + r], head_cols=head, bf16_only=bf16_only)
            torch.cuda.synchronize()
            o = obs.cpu()
            assert torch.equal(o[:, :head], before[:, :head].cpu()) and bool((o[:, head + r:] == 7.0).all())
            if bf16_only:
                assert torch.equal(o, before.cpu()), "bf16_only wrote fp32 columns"
            else:
                assert_exact(f"height_scan_obs {path} R={r} head={head}", o[:, head:head + r].numpy(), m)
            want_bf = torch.cat([before[:, :head].cpu(), torch.from_numpy(m.h)], 1).to(torch.bfloat16)
            assert torch.equal(obs_bf[:, :head + r].cpu(), want_bf), f"bf16 mirror {path} R={r} head={head} bf16_only={bf16_only}"
            assert bool((obs_bf[:, head + r:] == 9.0).all())
    finally:
        g.cells_struct.entries_planar = saved


@pytest.mark.parametrize("r", [256, 961])
def test_height_scan_out_view_and_host(cuda_device, r):
    g = terrain("random", cuda_device)
    pat = pattern(r)
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    n = 300
    pos, quat = exact_poses(g, n, seed=r)
    P, Q = torch.from_numpy(pos).to(cuda_device), torch.from_numpy(quat).to(cuda_device)
    m = _model(g, pos, quat, pat)
    for variant in (0, 2, 4, 5):
        buf = torch.full((n, 968), 7.0, device=cuda_device)
        ops.height_scan(P, Q, rays, g, out=buf[:, :r], variant=variant)
        mm = _model(g, pos, quat, pat, 0) if variant == 0 else m
        assert_exact(f"out= view v{variant}", buf[:, :r].cpu().numpy(), mm)
        assert bool((buf[:, r:] == 7.0).all())
    work = ops.HostScanWork(n, r, cuda_device)
    for slices in (1, 7):
        out = torch.full((n, r), float("nan")).pin_memory()
        ops.height_scan_host(torch.from_numpy(pos).pin_memory(), torch.from_numpy(quat).pin_memory(), rays, g, out, work,
                             n_slices=slices)
        torch.cuda.synchronize()
        assert_exact(f"height_scan_host slices={slices}", out.numpy(), m)


def _xy_bound(pat, pos):
    """|X - X64| bound for a non-exact yaw (see test_height_scan_general_yaw)."""
    v = np.abs(pat[None, :, :2]).max(-1)
    return 24 * U * v + U * (np.abs(pos[:, None, :2]).max(-1) + 2 * v)


def _rotated_starts(pos, quat, pat):
    """float64 ray starts X, Y with the true yaw of the quaternion."""
    w, x, y, z = np.asarray(quat, np.float64).T
    yaw = np.arctan2(2 * (w * z + x * y), 1 - 2 * (y * y + z * z))
    c, s = np.cos(yaw)[:, None], np.sin(yaw)[:, None]
    p = np.asarray(pos, np.float64)
    return p[:, 0:1] + c * pat[None, :, 0] - s * pat[None, :, 1], p[:, 1:2] + s * pat[None, :, 0] + c * pat[None, :, 1]


def check_misses(where, g, pos, quat, pat, hit):
    """Rays a kernel reports as misses, where the host cannot reproduce the frame: every ray whose float64 start lies
    farther than the ulp bound from the lattice border must hit exactly when the model, evaluated at that start rounded
    to fp32, hits (outside the lattice: a miss; inside: a hit unless t leaves [0, max_d) or the cell is a hole)."""
    X64, Y64 = _rotated_starts(pos, quat, pat)
    b = _xy_bound(pat, pos)
    xs, ys = g.cells.xs.cpu().numpy().astype(np.float64), g.cells.ys.cpu().numpy().astype(np.float64)
    near = ((np.abs(X64 - xs[0]) <= b) | (np.abs(X64 - xs[-1]) <= b) | (np.abs(Y64 - ys[0]) <= b) |
            (np.abs(Y64 - ys[-1]) <= b))
    m = SE.scan_model(pos, quat, pat, g.cells, g.grid, XY=(X64.astype(F32), Y64.astype(F32)))
    want = np.isfinite(m.h)
    bad = np.nonzero(~near & (want != hit))
    if len(bad[0]):
        e, r = bad[0][0], bad[1][0]
        raise AssertionError(f"{where}: {len(bad[0])} rays hit / miss unlike the model at the float64 start; first env {e} "
                             f"ray {r}: X64={X64[e, r]!r} Y64={Y64[e, r]!r} path={SE.PATHS[m.path[e, r]]} kernel hit={hit[e, r]}")


def test_height_scan_general_yaw(cuda_device):
    """Yaws whose sinf / cosf the host cannot reproduce: the model takes X, Y from variant 2's hits and must reproduce
    hz and the height of every hit bit for bit; X, Y themselves lie within the bound of a float64 rotation.
    The bound: cw and sz carry <= 2 ulp each from atan2f / sinf / cosf, the fp32 yaw of the quaternion <= 4 ulp, their
    normalisation <= 2 ulp, so the rotated offset is off by <= ~12 u |v| (u = 2^-24); the four roundings of the
    rotation chain add <= 2 u (|v| + 2|v|) and the final + p <= u |X|.  24 u |v| + u (|p| + 2|v|) covers it."""
    g = terrain("random", cuda_device)
    pat = pattern(961)
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    gen = torch.Generator().manual_seed(4)
    n = 200
    pos = torch.cat([torch.rand(n, 2, generator=gen) * 26 - 1, torch.rand(n, 1, generator=gen) + 0.5], 1)
    quat = synthetic.quat_from_euler(torch.randn(n, generator=gen) * 0.1, torch.randn(n, generator=gen) * 0.1,
                                     (torch.rand(n, generator=gen) * 2 - 1) * np.pi)
    P, Q = pos.to(cuda_device), quat.to(cuda_device)
    h2, hits2 = ops.height_scan(P, Q, rays, g, variant=2, return_hits=True)
    hits2 = hits2.cpu().numpy()
    hit = np.isfinite(hits2[..., 0])
    X, Y = np.where(hit, hits2[..., 0], 0).astype(F32), np.where(hit, hits2[..., 1], 0).astype(F32)
    m = SE.scan_model(pos.numpy(), quat.numpy(), pat, g.cells, g.grid, XY=(X, Y))
    want = np.where(hit, m.h, np.float32(-np.inf)).astype(F32)
    assert_exact("v2 general yaw", h2.cpu().numpy(), m, want)
    assert np.array_equal(_bits(np.where(hit, hits2[..., 2], 0)), _bits(np.where(hit, m.hits[..., 2], 0)))
    for variant in (0, 4, 5):
        h = ops.height_scan(P, Q, rays, g, variant=variant).cpu().numpy()
        if variant == 0:
            mm = SE.scan_model(pos.numpy(), quat.numpy(), pat, None, g.grid, XY=(X, Y), home_only=True)
            assert_exact("v0 general yaw", np.where(hit, h, -np.inf), mm, np.where(hit, mm.h, -np.inf).astype(F32))
        else:
            assert np.array_equal(_bits(h), _bits(h2.cpu().numpy())), f"v{variant} general yaw"
    X64, Y64 = _rotated_starts(pos.numpy(), quat.numpy(), pat)
    bound = _xy_bound(pat, pos.numpy())
    assert (np.abs(X - X64) <= bound)[hit].all() and (np.abs(Y - Y64) <= bound)[hit].all()
    assert hit.any() and (~hit).any()
    check_misses("v2 general yaw", g, pos.numpy(), quat.numpy(), pat, hit)


@pytest.mark.parametrize("r,n", [(1, 148 * 33), (64, 148 * 33), (256, 148 * 33), (257, 148 * 9 + 3), (625, 148 * 9 + 3),
                                 (1024, 148 * 9 + 3), (256, 148 * 4 + 7)])
def test_step_fused_equals_mdp_step_then_scan_any_pattern(cuda_device, r, n):
    """More than 8 environments per CTA (the ring wraps; at <= 256 rays a worker moves up to 15 environments between its
    work units), bit for bit against mdp_step + height_scan and against the model."""
    SIZE, RES = 48.0, 0.2
    v, f = TR.make_synthetic_terrain(SIZE, RES, seed=3)
    g = ops.ScanGridHandle.from_mesh(v, f, cuda_device)
    g.ensure_home_grid()
    pat = pattern(r, "zvar" if r == 257 else "flat")
    rays = ops.RayPattern(torch.from_numpy(pat), cuda_device)
    tables = TR.build_terrain_tables(v, f, n)
    params = ops.mdp_params(RoverEnvCfg(num_envs=n))
    th = ops.TerrainTablesHandle(tables.heightmap, tables.safe_mask, tables.offset_xy, tables.spawn_table, tables.resolution,
                                 cuda_device)
    gen = torch.Generator().manual_seed(60 + r)
    vt = torch.from_numpy(v)
    steps = [synthetic.make_step(n, gen, vt, SIZE, RES, margin=4.0).to(cuda_device) for _ in range(2)]
    pc, hc, ep = synthetic.init_commands(n, gen, steps[0].root_pos_w.cpu())
    bufs, rngs, obss = [], [], []
    for _ in range(2):
        b = ops.MdpBuffers.allocate(n, cuda_device)
        b.pos_cmd_w.copy_(pc)
        b.heading_cmd_w.copy_(hc)
        b.episode_length_buf.copy_(ep)
        b.env_origins.copy_(steps[0].root_pos_w)
        b.time_left.fill_(150.0)
        bufs.append(b)
        rngs.append(ops.ResetRng(77, cuda_device, step=5))
        obss.append(torch.full((n, 4 + r + 3), 7.0, device=cuda_device) if r != 961 else alloc_obs(n, cuda_device))
    for k, s in enumerate(steps):
        roots = [(s.root_pos_w.clone(), s.root_quat_w.clone()) for _ in range(2)]
        ops.mdp_step(bufs[0], params, th, s.actions, s.force_matrix_w, *roots[0], obs=obss[0], rng=rngs[0])
        ops.height_scan(*roots[0], rays, g, out=obss[0][:, 4:4 + r])
        ops.step_fused(bufs[1], params, th, s.actions, s.force_matrix_w, *roots[1], rays, g, obss[1], rngs[1])
        torch.cuda.synchronize()
        assert torch.equal(roots[0][0], roots[1][0]) and torch.equal(roots[0][1], roots[1][1]), (r, k)
        for e in torch.nonzero((obss[0] != obss[1]).any(1) & ~(obss[0].isnan() & obss[1].isnan()).all(1)).squeeze(-1)[:1].tolist():
            raise AssertionError(f"step_fused R={r} step {k}: env {e} differs from mdp_step + height_scan")
        assert torch.equal(obss[0], obss[1]), (r, k)
        # the heights at the returned root poses against the model (X, Y from variant 2's hits)
        P, Q = roots[1]
        _, hits = ops.height_scan(P, Q, rays, g, variant=2, return_hits=True)
        hits = hits.cpu().numpy()
        hit = np.isfinite(hits[..., 0])
        X, Y = np.where(hit, hits[..., 0], 0).astype(F32), np.where(hit, hits[..., 1], 0).astype(F32)
        m = SE.scan_model(P.cpu().numpy(), Q.cpu().numpy(), pat, g.cells, g.grid, XY=(X, Y))
        got = obss[1][:, 4:4 + r].cpu().numpy()
        assert_exact(f"step_fused R={r} step {k} vs model", np.where(hit, got, -np.inf).astype(F32), m,
                     np.where(hit, m.h, -np.inf).astype(F32))
        assert np.array_equal(np.isinf(got), ~hit)
        check_misses(f"step_fused R={r} step {k}", g, P.cpu().numpy(), Q.cpu().numpy(), pat, hit)
