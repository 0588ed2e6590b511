// Height-scan raycaster for rays in any direction (ORBIT RayCasterCfg.attach_yaw_only = False and/or a pattern direction
// other than (0, 0, -1)).  The reference's own configuration (yaw-only, straight down) keeps running the vertical
// kernels of height_scan*.cu; this kernel is the general path (ops.height_scan routes to it, variant 6 forces it).
//
// Replaces ORBIT RayCaster._update_buffers_impl -> raycast_mesh -> warp mesh_query_ray (wired at
// rover_envs/envs/navigation/rover_env_cfg.py:78-86), both branches of the frame, fused with height_scan_rover
// (rover_envs/envs/navigation/mdp/observations.py:35-45).  One thread per ray; a CTA covers 256 consecutive rays of one
// environment and computes the sensor frame once into shared memory:
//   * attach_yaw_only: starts = make_frame + ray_origin (bit-identical to the vertical kernels), directions unrotated;
//     otherwise starts = quat_apply(q, v) + p and directions = quat_apply(q, d), q as given, ORBIT's operation order;
//   * P(t) = S + t * D, 0 <= t < max_distance, t in units of |D| (directions are used as given, not normalised);
//   * vertical rays (D.x == D.y == 0) look up one column of the plane-cell table exactly like variant 2;
//   * other rays are clipped to the lattice box and walk its rectilinear cells in increasing t (2-D DDA).  A closed-form
//     cell is solved on its segment from the entry point relative to the cell corner: g(t) = P_z - z(P_x, P_y) is
//     linear on either side of the crease E = 0, and the first zero / sign change is the hit (double-sided).  A general
//     cell tests the home-grid records that can cover it: plane intersection, then the three edge functions.
// The observation form (rover_ray_cast_obs / _bf16) is the same kernel with the stores of rover_height_scan_obs: heights
// into columns [head_cols, head_cols + n_rays) of the fp32 observation and their bf16 mirror, plus the mirror of the
// head columns [0, head_cols) that the post-step wrote.
#include <cuda_bf16.h>

#include "scan_common.cuh"

namespace rover {
namespace {

constexpr int kRayThreads = 256;

// what the kernel stores: heights (+ hits), fp32 observation + bf16 mirror, or the bf16 mirror only
enum RayStore { kStoreHeights = 0, kStoreObs = 1, kStoreBf16Only = 2 };

struct RayFrame {
    SensorFrame yaw;       // yaw-only frame (attach_yaw_only)
    float qw, qx, qy, qz;  // full quaternion as given (otherwise)
};

// the same column / row search as height_scan.cu's locate (half-open cells, closed far border)
__device__ __forceinline__ int locate_line(const float* __restrict__ lines, int n, float inv_d, float v, bool& inside) {
    const float lo = __ldg(lines), hi = __ldg(lines + n);
    inside = (v >= lo) && (v <= hi);
    int i = (int)fminf(fmaxf(floorf(__fmul_rn(__fsub_rn(v, lo), inv_d)), 0.f), (float)(n - 1));
    while (i > 0 && v < __ldg(lines + i)) --i;
    while (i < n - 1 && v >= __ldg(lines + i + 1)) ++i;
    return i;
}

// ORBIT quat_apply (SURVEY.md A.1): t = 2 * (xyz x v); v + w * t + xyz x t.  Every operation rounded, no contraction.
__device__ __forceinline__ void quat_apply_rn(const RayFrame& f, float vx, float vy, float vz, float& ox, float& oy,
                                              float& oz) {
    const float tx = __fmul_rn(__fsub_rn(__fmul_rn(f.qy, vz), __fmul_rn(f.qz, vy)), 2.f);
    const float ty = __fmul_rn(__fsub_rn(__fmul_rn(f.qz, vx), __fmul_rn(f.qx, vz)), 2.f);
    const float tz = __fmul_rn(__fsub_rn(__fmul_rn(f.qx, vy), __fmul_rn(f.qy, vx)), 2.f);
    const float cx = __fsub_rn(__fmul_rn(f.qy, tz), __fmul_rn(f.qz, ty));
    const float cy = __fsub_rn(__fmul_rn(f.qz, tx), __fmul_rn(f.qx, tz));
    const float cz = __fsub_rn(__fmul_rn(f.qx, ty), __fmul_rn(f.qy, tx));
    ox = __fadd_rn(__fadd_rn(vx, __fmul_rn(f.qw, tx)), cx);
    oy = __fadd_rn(__fadd_rn(vy, __fmul_rn(f.qw, ty)), cy);
    oz = __fadd_rn(__fadd_rn(vz, __fmul_rn(f.qw, tz)), cz);
}

// vertical ray over the home grid: cast_down of height_scan.cu with t = (z - Z) / Dz; the smallest valid t.
// For Dz = -1, t == Z - z exactly and the smallest t is the highest z: cast_down's answer bit for bit.
__device__ __forceinline__ float cast_vertical(const ScanGridDev& g, float X, float Y, float Z, float Dz, float max_d) {
    float best = INFINITY;
    for (int l = 0; l < g.n_levels; ++l) {
        const ScanLevelDev& L = g.level[l];
        const int i = cell_of(X, L.ox, L.inv_cell);
        const int j = cell_of(Y, L.oy, L.inv_cell);
        const int j0 = max(j - g.span, 0), j1 = min(j, L.ncy - 1);
        const int i0 = max(i - g.span, 0), i1 = min(i, L.ncx - 1);
        for (int jj = j0; jj <= j1; ++jj) {
            const float ly = __fsub_rn(Y, __fadd_rn(L.oy, __fmul_rn((float)jj, L.cell)));
            const int* __restrict__ row = g.cell_start + L.start_offset + jj * L.ncx;
            for (int ii = i0; ii <= i1; ++ii) {
                const float lx = __fsub_rn(X, __fadd_rn(L.ox, __fmul_rn((float)ii, L.cell)));
                const int b = __ldg(row + ii), e = __ldg(row + ii + 1);
                for (int r = b; r < e; ++r) {
                    const float4 r0 = __ldg(g.rec + 3 * r), r1 = __ldg(g.rec + 3 * r + 1), r2 = __ldg(g.rec + 3 * r + 2);
                    const float e0 = fmaf(r0.x, lx, fmaf(r0.y, ly, r0.z));
                    const float e1 = fmaf(r0.w, lx, fmaf(r1.x, ly, r1.y));
                    const float e2 = fmaf(r1.z, lx, fmaf(r1.w, ly, r2.x));
                    const float z = fmaf(r2.y, lx, fmaf(r2.z, ly, r2.w));
                    const float t = __fdiv_rn(__fsub_rn(z, Z), Dz);
                    if (fminf(e0, fminf(e1, e2)) >= 0.f && t >= 0.f && t < max_d) best = fminf(best, t);
                }
            }
        }
    }
    return best;
}

// tilted ray segment [t0, t1] through general plane cell (ci, cj): the home-grid records whose homes can cover the
// cell's rectangle; smallest t of a record hit on the segment (a few ulp of slack at its ends: the triangles are real,
// so a hit just outside the segment is still a hit of the mesh), or +inf
__device__ __forceinline__ float cast_general(const ScanGridDev& g, float cx0, float cx1, float cy0, float cy1, float P0x,
                                              float P0y, float P0z, float Dx, float Dy, float Dz, float t0, float t1) {
    float best = INFINITY;
    const float len = __fsub_rn(t1, t0);
    const float slack = __fmul_rn(4.0e-6f, __fadd_rn(1.f, t1));
    for (int l = 0; l < g.n_levels; ++l) {
        const ScanLevelDev& L = g.level[l];
        const int j0 = max(cell_of(cy0, L.oy, L.inv_cell) - g.span, 0), j1 = min(cell_of(cy1, L.oy, L.inv_cell), L.ncy - 1);
        const int i0 = max(cell_of(cx0, L.ox, L.inv_cell) - g.span, 0), i1 = min(cell_of(cx1, L.ox, L.inv_cell), L.ncx - 1);
        for (int jj = j0; jj <= j1; ++jj) {
            const float ly0 = __fsub_rn(P0y, __fadd_rn(L.oy, __fmul_rn((float)jj, L.cell)));
            const int* __restrict__ row = g.cell_start + L.start_offset + jj * L.ncx;
            for (int ii = i0; ii <= i1; ++ii) {
                const float lx0 = __fsub_rn(P0x, __fadd_rn(L.ox, __fmul_rn((float)ii, L.cell)));
                const int b = __ldg(row + ii), e = __ldg(row + ii + 1);
                for (int r = b; r < e; ++r) {
                    const float4 r0 = __ldg(g.rec + 3 * r), r1 = __ldg(g.rec + 3 * r + 1), r2 = __ldg(g.rec + 3 * r + 2);
                    const float g0 = __fsub_rn(P0z, fmaf(r2.y, lx0, fmaf(r2.z, ly0, r2.w)));
                    const float s = __fsub_rn(Dz, fmaf(r2.y, Dx, __fmul_rn(r2.z, Dy)));
                    const float u = g0 == 0.f ? 0.f : __fdiv_rn(-g0, s);
                    if (!(u >= -slack && u <= __fadd_rn(len, slack))) continue;
                    const float lx = fmaf(u, Dx, lx0), ly = fmaf(u, Dy, ly0);
                    const float e0 = fmaf(r0.x, lx, fmaf(r0.y, ly, r0.z));
                    const float e1 = fmaf(r0.w, lx, fmaf(r1.x, ly, r1.y));
                    const float e2 = fmaf(r1.z, lx, fmaf(r1.w, ly, r2.x));
                    if (fminf(e0, fminf(e1, e2)) >= 0.f) best = fminf(best, __fadd_rn(t0, u));
                }
            }
        }
    }
    return best;
}

// g = P_z - z of a closed-form cell at segment parameter u (coordinates relative to the cell corner)
__device__ __forceinline__ float gap(const float4 p, const float4 q, float lx0, float ly0, float pz0, float Dx, float Dy,
                                     float Dz, float u) {
    const float lx = fmaf(u, Dx, lx0), ly = fmaf(u, Dy, ly0);
    const float E = fmaf(q.x, lx, fmaf(q.y, ly, q.z));
    const float z = fmaf(p.w, fminf(E, 0.f), fmaf(p.x, lx, fmaf(p.y, ly, p.z)));
    return __fsub_rn(fmaf(u, Dz, pz0), z);
}

// first u of [ua, ub] where the linear g goes through zero, or -1
__device__ __forceinline__ float root_on(float ua, float ga, float ub, float gb) {
    if (gb == 0.f) return ub;
    if ((ga < 0.f) == (gb < 0.f) || ga != ga || gb != gb) return -1.f;
    const float u = fmaf(__fsub_rn(ub, ua), __fdiv_rn(ga, __fsub_rn(ga, gb)), ua);
    return fminf(fmaxf(u, ua), ub);
}

// the walk of a tilted ray (not D.x == D.y == 0); returns t of the first hit, or +inf
__device__ __forceinline__ float cast_tilted(const ScanGridDev& g, const PlaneCellsDev& pc, float X, float Y, float Z, float Dx, float Dy,
                             float Dz, float max_d) {
    const float x0 = __ldg(pc.xs), x1 = __ldg(pc.xs + pc.nx), y0 = __ldg(pc.ys), y1 = __ldg(pc.ys + pc.ny);
    // 1. clip to the lattice box and to [0, max_d)
    float tin = 0.f, tout = max_d;
    if (Dx != 0.f) {
        const float a = __fdiv_rn(__fsub_rn(x0, X), Dx), b = __fdiv_rn(__fsub_rn(x1, X), Dx);
        tin = fmaxf(tin, fminf(a, b));
        tout = fminf(tout, fmaxf(a, b));
    } else if (!(X >= x0 && X <= x1)) {
        return INFINITY;
    }
    if (Dy != 0.f) {
        const float a = __fdiv_rn(__fsub_rn(y0, Y), Dy), b = __fdiv_rn(__fsub_rn(y1, Y), Dy);
        tin = fmaxf(tin, fminf(a, b));
        tout = fminf(tout, fmaxf(a, b));
    } else if (!(Y >= y0 && Y <= y1)) {
        return INFINITY;
    }
    if (!(tin < max_d) || tin > tout) return INFINITY;
    // 2. first cell: locate's convention at the start (or at the clamped entry point)
    float ex = X, ey = Y;
    if (tin > 0.f) {
        ex = fminf(fmaxf(fmaf(tin, Dx, X), x0), x1);
        ey = fminf(fmaxf(fmaf(tin, Dy, Y), y0), y1);
    }
    bool in_x, in_y;
    int i = locate_line(pc.xs, pc.nx, pc.inv_dx, ex, in_x);
    int j = locate_line(pc.ys, pc.ny, pc.inv_dy, ey, in_y);
    const int sx = Dx > 0.f ? 1 : (Dx < 0.f ? -1 : 0), sy = Dy > 0.f ? 1 : (Dy < 0.f ? -1 : 0);
    float tc = tin;
    float carry = 0.f;  // g at the end of the previous closed-form segment (0: none)
    for (;;) {
        const float tnx = sx > 0 ? __fdiv_rn(__fsub_rn(__ldg(pc.xs + i + 1), X), Dx)
                                 : (sx < 0 ? __fdiv_rn(__fsub_rn(__ldg(pc.xs + i), X), Dx) : INFINITY);
        const float tny = sy > 0 ? __fdiv_rn(__fsub_rn(__ldg(pc.ys + j + 1), Y), Dy)
                                 : (sy < 0 ? __fdiv_rn(__fsub_rn(__ldg(pc.ys + j), Y), Dy) : INFINITY);
        const float tn = fminf(fminf(tnx, tny), tout);
        const float te = fmaxf(tn, tc);
        // 3. the cell on [tc, te], from the segment's entry point
        const float P0x = fmaf(tc, Dx, X), P0y = fmaf(tc, Dy, Y), P0z = fmaf(tc, Dz, Z);
        const float cx0 = __ldg(pc.xs + i), cy0 = __ldg(pc.ys + j);
        const float4* __restrict__ ent = pc.ent + 2 * ((size_t)j * pc.nx + i);
        const float4 p = __ldg(ent), q = __ldg(ent + 1);
        float t_hit = INFINITY;
        if (q.w != 0.f) {
            t_hit = cast_general(g, cx0, __ldg(pc.xs + i + 1), cy0, __ldg(pc.ys + j + 1), P0x, P0y, P0z, Dx, Dy, Dz, tc, te);
            carry = 0.f;
        } else if (p.z == -INFINITY) {
            carry = 0.f;  // empty cell
        } else {
            const float lx0 = __fsub_rn(P0x, cx0), ly0 = __fsub_rn(P0y, cy0);
            const float len = __fsub_rn(te, tc);
            const float ga = gap(p, q, lx0, ly0, P0z, Dx, Dy, Dz, 0.f);
            float u = -1.f;
            if (ga == 0.f || (carry != 0.f && ga == ga && (carry < 0.f) != (ga < 0.f))) {
                u = 0.f;  // on the surface at entry, or crossed it exactly on the border between two cells
            } else {
                // break of g where the ray crosses the crease E = 0 inside the segment
                const float E0 = fmaf(q.x, lx0, fmaf(q.y, ly0, q.z));
                const float eS = fmaf(q.x, Dx, __fmul_rn(q.y, Dy));
                const float ub = eS != 0.f ? __fdiv_rn(-E0, eS) : -1.f;
                float ua = 0.f, gA = ga;
                if (p.w != 0.f && ub > 0.f && ub < len) {
                    const float gb = gap(p, q, lx0, ly0, P0z, Dx, Dy, Dz, ub);
                    u = root_on(0.f, ga, ub, gb);
                    ua = ub;
                    gA = gb;
                }
                if (u < 0.f) {
                    const float ge = gap(p, q, lx0, ly0, P0z, Dx, Dy, Dz, len);
                    u = root_on(ua, gA, len, ge);
                    carry = ge;
                }
            }
            if (u >= 0.f) t_hit = __fadd_rn(tc, u);
        }
        if (t_hit != INFINITY) return t_hit >= 0.f && t_hit < max_d ? t_hit : INFINITY;
        // 4. next cell: the nearer border (both at a lattice vertex)
        if (!(fminf(tnx, tny) < tout)) return INFINITY;
        if (tnx <= tny) i += sx;
        if (tny <= tnx) j += sy;
        if (i < 0 || i >= pc.nx || j < 0 || j >= pc.ny) return INFINITY;
        tc = te;
    }
}

// kStoreHeights: heights to out[env, r] (head_cols == 0), hits optional.  The observation modes: `out` is the fp32
// observation, heights go to out[env, head_cols + r] (kStoreObs only) and their bf16 to obs_bf16[env, head_cols + r];
// the CTAs of chunk 0 mirror out[env, 0:head_cols] into obs_bf16.
template <int kStore>
__global__ void __launch_bounds__(kRayThreads, 2)
ray_cast_kernel(const float* __restrict__ pos_w, const float* __restrict__ quat_w, int n_chunks,
                const float* __restrict__ ray_local, const float* __restrict__ ray_dirs, int n_rays, int yaw_only,
                const __grid_constant__ ScanGridDev g, const __grid_constant__ PlaneCellsDev pc, float max_d,
                float base_offset, float* __restrict__ out, int out_stride, int head_cols, float* __restrict__ hits,
                __nv_bfloat16* __restrict__ obs_bf16, int bf16_stride) {
    const int env = blockIdx.x / n_chunks;
    const int r = (blockIdx.x - env * n_chunks) * kRayThreads + threadIdx.x;
    // the ray pattern is launch-invariant: read it before waiting for the kernel in front of this one
    float vx = 0.f, vy = 0.f, vz = 0.f, dx = 0.f, dy = 0.f, dz = 0.f;
    if (r < n_rays) {
        vx = __ldg(ray_local + 3 * r), vy = __ldg(ray_local + 3 * r + 1), vz = __ldg(ray_local + 3 * r + 2);
        dx = __ldg(ray_dirs + 3 * r), dy = __ldg(ray_dirs + 3 * r + 1), dz = __ldg(ray_dirs + 3 * r + 2);
    }
    grid_dependency_wait();
    __shared__ RayFrame frame_s;
    if (threadIdx.x == 0) {
        const float* q = quat_w + 4 * (size_t)env;
        frame_s.yaw = make_frame(pos_w + 3 * (size_t)env, q);
        frame_s.qw = q[0];
        frame_s.qx = q[1];
        frame_s.qy = q[2];
        frame_s.qz = q[3];
    }
    if (kStore != kStoreHeights && blockIdx.x == env * n_chunks) {
        // the head columns are written by the kernel in front of this one (the post-step): read only after the wait
        const float* head = out + (size_t)env * out_stride;
        __nv_bfloat16* dst = obs_bf16 + (size_t)env * bf16_stride;
        for (int c = threadIdx.x; c < head_cols; c += kRayThreads) dst[c] = __float2bfloat16_rn(head[c]);
    }
    __syncthreads();
    if (r >= n_rays) return;
    const RayFrame f = frame_s;
    float X, Y, Z, Dx = dx, Dy = dy, Dz = dz;
    if (yaw_only) {
        ray_origin(f.yaw, vx, vy, vz, X, Y, Z);
    } else {
        quat_apply_rn(f, vx, vy, vz, X, Y, Z);
        X = __fadd_rn(X, f.yaw.px);
        Y = __fadd_rn(Y, f.yaw.py);
        Z = __fadd_rn(Z, f.yaw.pz);
        quat_apply_rn(f, dx, dy, dz, Dx, Dy, Dz);
    }
    float t = INFINITY;
    const bool vertical = Dx == 0.f && Dy == 0.f;
    if (vertical) {
        if (Dz != 0.f) {
            // variant 2's column lookup with t = (z - Z) / Dz
            bool in_x, in_y;
            const int i = locate_line(pc.xs, pc.nx, pc.inv_dx, X, in_x);
            const int j = locate_line(pc.ys, pc.ny, pc.inv_dy, Y, in_y);
            if (in_x && in_y) {
                const float4* __restrict__ e = pc.ent + 2 * ((size_t)j * pc.nx + i);
                const float4 p = __ldg(e), q = __ldg(e + 1);
                if (q.w == 0.f) {
                    const float lx = __fsub_rn(X, __ldg(pc.xs + i)), ly = __fsub_rn(Y, __ldg(pc.ys + j));
                    const float E = fmaf(q.x, lx, fmaf(q.y, ly, q.z));
                    const float z = fmaf(p.w, fminf(E, 0.f), fmaf(p.x, lx, fmaf(p.y, ly, p.z)));
                    const float tz = __fdiv_rn(__fsub_rn(z, Z), Dz);
                    if (tz >= 0.f && tz < max_d) t = tz;
                } else {
                    t = cast_vertical(g, X, Y, Z, Dz, max_d);
                }
            }
        }
    } else if (isfinite(X) && isfinite(Y) && isfinite(Z) && isfinite(Dx) && isfinite(Dy) && isfinite(Dz)) {
        t = cast_tilted(g, pc, X, Y, Z, Dx, Dy, Dz, max_d);
    }
    float h = -INFINITY, hx = INFINITY, hy = INFINITY, hz = INFINITY;
    if (t != INFINITY) {
        // hit = S + t * D (one rounding per component); for D = (0, 0, -1): (X, Y, Z - t), the vertical kernels' chain
        hx = vertical ? X : fmaf(t, Dx, X);
        hy = vertical ? Y : fmaf(t, Dy, Y);
        hz = fmaf(t, Dz, Z);
        h = __fsub_rn(__fsub_rn(f.yaw.pz, hz), base_offset);
    }
    if (kStore != kStoreBf16Only) out[(size_t)env * out_stride + head_cols + r] = h;
    if (kStore != kStoreHeights) obs_bf16[(size_t)env * bf16_stride + head_cols + r] = __float2bfloat16_rn(h);
    if (kStore == kStoreHeights && hits) {
        float* p3 = hits + ((size_t)env * n_rays + r) * 3;
        p3[0] = hx;
        p3[1] = hy;
        p3[2] = hz;
    }
}

}  // namespace

int make_dev_grid(const RoverScanGrid* grid, ScanGridDev& g);  // height_scan.cu

// the checks and the launch shared by the entry points (`what` names the entry point in messages); n_envs > 0, and
// n_rays > 0 in the heights mode.  In the observation modes n_rays may be 0: one CTA per environment mirrors the head.
template <int kStore>
static int launch_ray_cast(const char* what, const float* pos_w, const float* quat_w, int32_t n_envs,
                           const float* ray_starts_local, const float* ray_dirs_local, int32_t n_rays, int32_t attach_yaw_only,
                           const RoverScanGrid* grid, const RoverPlaneCells* cells, float max_distance, float base_offset,
                           float* out, int32_t out_stride, int32_t head_cols, float* out_hits_w, uint16_t* obs_bf16,
                           int32_t bf16_stride, void* stream) {
    ROVER_CHECK(pos_w && quat_w && (n_rays == 0 || (ray_starts_local && ray_dirs_local)), "%s: NULL tensor", what);
    ROVER_CHECK(cells != nullptr, "%s: the plane-cell table is required", what);
    ROVER_CHECK(cells->xs && cells->ys && cells->entries && cells->nx > 0 && cells->ny > 0, "%s: bad plane-cell table", what);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(cells->entries) & 15) == 0, "%s: plane-cell entries not 16B aligned", what);
    ScanGridDev g;
    if (int rc = make_dev_grid(grid, g)) return rc;
    const int n_chunks = n_rays > 0 ? (n_rays + kRayThreads - 1) / kRayThreads : 1;
    ROVER_CHECK((int64_t)n_envs * n_chunks <= 0x7fffffff, "%s: %d environments x %d chunks is too many", what, n_envs,
                n_chunks);
    const PlaneCellsDev pc{cells->xs, cells->ys, reinterpret_cast<const float4*>(cells->entries), cells->nx, cells->ny,
                           cells->inv_dx, cells->inv_dy};
    ROVER_CUDA(launch_overlapped(ray_cast_kernel<kStore>, dim3(n_envs * n_chunks), dim3(kRayThreads), 0,
                                 static_cast<cudaStream_t>(stream), pos_w, quat_w, n_chunks, ray_starts_local, ray_dirs_local,
                                 n_rays, (int)(attach_yaw_only != 0), g, pc, max_distance, base_offset, out, out_stride,
                                 head_cols, out_hits_w, reinterpret_cast<__nv_bfloat16*>(obs_bf16), bf16_stride));
    return check_launch("ray_cast_kernel");
}

// the observation entry points: fp32 + bf16 (kStoreObs) or bf16 only (kStoreBf16Only)
template <int kStore>
static int ray_cast_obs_impl(const char* what, const float* pos_w, const float* quat_w, int32_t n_envs,
                             const float* ray_starts_local, const float* ray_dirs_local, int32_t n_rays, int32_t attach_yaw_only,
                             const RoverScanGrid* grid, const RoverPlaneCells* cells, float max_distance, float base_offset,
                             float* obs, int32_t obs_stride, int32_t head_cols, uint16_t* obs_bf16, int32_t bf16_stride,
                             void* stream) {
    ROVER_CHECK(n_envs >= 0 && n_rays >= 0 && head_cols >= 0, "%s: negative sizes", what);
    if (n_envs == 0 || n_rays + head_cols == 0) return 0;
    ROVER_CHECK(obs && obs_bf16, "%s: NULL observation buffer", what);
    ROVER_CHECK((int64_t)head_cols + n_rays <= obs_stride && (int64_t)head_cols + n_rays <= bf16_stride,
                "%s: row strides %d / %d < head_cols + n_rays = %lld", what, obs_stride, bf16_stride,
                (long long)head_cols + n_rays);
    return launch_ray_cast<kStore>(what, pos_w, quat_w, n_envs, ray_starts_local, ray_dirs_local, n_rays, attach_yaw_only,
                                   grid, cells, max_distance, base_offset, obs, obs_stride, head_cols, nullptr, obs_bf16,
                                   bf16_stride, stream);
}

}  // namespace rover

extern "C" int rover_ray_cast(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                              const float* ray_dirs_local, int32_t n_rays, int32_t attach_yaw_only,
                              const RoverScanGrid* grid, const RoverPlaneCells* cells, float max_distance,
                              float base_offset, float* out_heights, int32_t out_stride, float* out_hits_w, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0 && n_rays >= 0, "rover_ray_cast: negative sizes");
    if (n_envs == 0 || n_rays == 0) return 0;
    ROVER_CHECK(out_heights, "rover_ray_cast: NULL tensor");
    ROVER_CHECK(out_stride >= n_rays, "rover_ray_cast: out_stride %d < n_rays %d", out_stride, n_rays);
    return launch_ray_cast<kStoreHeights>("rover_ray_cast", pos_w, quat_w, n_envs, ray_starts_local, ray_dirs_local, n_rays,
                                          attach_yaw_only, grid, cells, max_distance, base_offset, out_heights, out_stride,
                                          0, out_hits_w, nullptr, 0, stream);
}

extern "C" int rover_ray_cast_obs(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                                  const float* ray_dirs_local, int32_t n_rays, int32_t attach_yaw_only,
                                  const RoverScanGrid* grid, const RoverPlaneCells* cells, float max_distance,
                                  float base_offset, float* obs, int32_t obs_stride, int32_t head_cols, uint16_t* obs_bf16,
                                  int32_t bf16_stride, void* stream) {
    return rover::ray_cast_obs_impl<rover::kStoreObs>("rover_ray_cast_obs", pos_w, quat_w, n_envs, ray_starts_local,
                                                      ray_dirs_local, n_rays, attach_yaw_only, grid, cells, max_distance,
                                                      base_offset, obs, obs_stride, head_cols, obs_bf16, bf16_stride, stream);
}

extern "C" int rover_ray_cast_obs_bf16(const float* pos_w, const float* quat_w, int32_t n_envs,
                                       const float* ray_starts_local, const float* ray_dirs_local, int32_t n_rays,
                                       int32_t attach_yaw_only, const RoverScanGrid* grid, const RoverPlaneCells* cells,
                                       float max_distance, float base_offset, const float* obs_head, int32_t obs_stride,
                                       int32_t head_cols, uint16_t* obs_bf16, int32_t bf16_stride, void* stream) {
    // the kernel does not store to obs_head in this mode
    return rover::ray_cast_obs_impl<rover::kStoreBf16Only>(
        "rover_ray_cast_obs_bf16", pos_w, quat_w, n_envs, ray_starts_local, ray_dirs_local, n_rays, attach_yaw_only, grid,
        cells, max_distance, base_offset, const_cast<float*>(obs_head), obs_stride, head_cols, obs_bf16, bf16_stride, stream);
}

extern "C" int rover_ray_cast_host(const float* pos_host, const float* quat_host, int32_t n_envs,
                                   const float* ray_starts_local, const float* ray_dirs_local, int32_t n_rays,
                                   int32_t attach_yaw_only, const RoverScanGrid* grid, const RoverPlaneCells* cells,
                                   float max_distance, float base_offset, float* out_host, int32_t out_stride, void* work,
                                   int64_t work_bytes, int32_t n_slices, void* stream) {
    using namespace rover;
    return host_scan_sliced("rover_ray_cast_host", pos_host, quat_host, n_envs, n_rays, out_host, out_stride, work,
                            work_bytes, n_slices, static_cast<cudaStream_t>(stream),
                            [&](const float* pos, const float* quat, int n, float* out, cudaStream_t s) {
                                return rover_ray_cast(pos, quat, n, ray_starts_local, ray_dirs_local, n_rays,
                                                      attach_yaw_only, grid, cells, max_distance, base_offset, out,
                                                      out_stride, nullptr, s);
                            });
}
