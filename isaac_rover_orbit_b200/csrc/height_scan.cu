// Height-scan raycaster for vertical rays over the multi-level home grid (see scan_grid.py).
//
// Replaces ORBIT RayCaster._update_buffers_impl -> raycast_mesh -> warp mesh_query_ray (third-party, wired at
// rover_envs/envs/navigation/rover_env_cfg.py:78-86) fused with height_scan_rover
// (rover_envs/envs/navigation/mdp/observations.py:35-45).  One CTA per environment:
//   * the yaw-only sensor frame is computed once per CTA in the reference's fp32 operation order
//     (ORBIT yaw_quat / quat_apply, SURVEY.md A.1) with contraction disabled, so ray origins match the
//     reference bit for bit up to libm differences in atan2f/sinf/cosf;
//   * every thread walks its rays through the home grid: for each level, the (span+1)^2 home cells whose
//     triangles can cover the ray's cell; a record test is 8 FMAs (3 edge functions + plane);
//   * closest hit along (0,0,-1) == highest z with 0 <= Z - z < max_distance;
//   * heights are written coalesced (consecutive threads = consecutive rays of one env).
#include <cuda_bf16.h>

#include "scan_common.cuh"

namespace rover {

// highest covered z below the ray origin, or -inf
__device__ __forceinline__ float cast_down(const ScanGridDev& g, float X, float Y, float Z, float max_d) {
    float best = -INFINITY;
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
                    const float4 r0 = __ldg(g.rec + 3 * r);
                    const float4 r1 = __ldg(g.rec + 3 * r + 1);
                    const float4 r2 = __ldg(g.rec + 3 * r + 2);
                    test_record(r0, r1, r2, lx, ly, Z, max_d, best);
                }
            }
        }
    }
    return best;
}

constexpr int kScanThreads = 256;

__global__ void __launch_bounds__(kScanThreads)
height_scan_direct_kernel(const float* __restrict__ pos_w, const float* __restrict__ quat_w,
                          const float* __restrict__ ray_local, int n_rays, const __grid_constant__ ScanGridDev g,
                          float max_d, float base_offset, float* __restrict__ out, int out_stride,
                          float* __restrict__ hits) {
    const int env = blockIdx.x;
    __shared__ SensorFrame frame_s;
    if (threadIdx.x == 0) frame_s = make_frame(pos_w + 3 * (size_t)env, quat_w + 4 * (size_t)env);
    __syncthreads();
    const SensorFrame f = frame_s;
    for (int r = threadIdx.x; r < n_rays; r += kScanThreads) {
        const float vx = __ldg(ray_local + 3 * r), vy = __ldg(ray_local + 3 * r + 1), vz = __ldg(ray_local + 3 * r + 2);
        float X, Y, Z;
        ray_origin(f, vx, vy, vz, X, Y, Z);
        const float zhit = cast_down(g, X, Y, Z, max_d);
        float h = -INFINITY, hx = INFINITY, hy = INFINITY, hz = INFINITY;
        if (zhit != -INFINITY) {
            // reference rounding chain: t -> hit.z = Z + t*(-1) -> (pos.z - hit.z) - offset
            const float t = __fsub_rn(Z, zhit);
            hz = __fsub_rn(Z, t);
            hx = X;
            hy = Y;
            h = __fsub_rn(__fsub_rn(f.pz, hz), base_offset);
        }
        out[(size_t)env * out_stride + r] = h;
        if (hits) {
            float* p = hits + ((size_t)env * n_rays + r) * 3;
            p[0] = hx;
            p[1] = hy;
            p[2] = hz;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// variant 2: plane-cell fast path.  One table entry (2 x float4) answers every ray of a closed-form cell:
// 5 FMAs instead of ~8 candidate tests; rays of general cells take the home-grid walk above.
// ---------------------------------------------------------------------------------------------------------
// column (row) of the half-open cell [lines[i], lines[i+1]) containing v; the far border is closed.
__device__ __forceinline__ int locate(const float* __restrict__ lines, int n, float inv_d, float v, bool& inside) {
    const float lo = __ldg(lines), hi = __ldg(lines + n);
    inside = (v >= lo) && (v <= hi);
    int i = (int)fminf(fmaxf(floorf((v - lo) * inv_d), 0.f), (float)(n - 1));
    while (i > 0 && v < __ldg(lines + i)) --i;
    while (i < n - 1 && v >= __ldg(lines + i + 1)) ++i;
    return i;
}

__global__ void __launch_bounds__(kScanThreads)
height_scan_cells_kernel(const float* __restrict__ pos_w, const float* __restrict__ quat_w,
                         const float* __restrict__ ray_local, int n_rays, const __grid_constant__ ScanGridDev g,
                         const __grid_constant__ PlaneCellsDev pc, float max_d, float base_offset,
                         float* __restrict__ out, int out_stride, float* __restrict__ hits) {
    const int env = blockIdx.x;
    __shared__ SensorFrame frame_s;
    if (threadIdx.x == 0) frame_s = make_frame(pos_w + 3 * (size_t)env, quat_w + 4 * (size_t)env);
    __syncthreads();
    const SensorFrame f = frame_s;
    for (int r = threadIdx.x; r < n_rays; r += kScanThreads) {
        const float vx = __ldg(ray_local + 3 * r), vy = __ldg(ray_local + 3 * r + 1), vz = __ldg(ray_local + 3 * r + 2);
        float X, Y, Z;
        ray_origin(f, vx, vy, vz, X, Y, Z);
        bool in_x, in_y;
        const int i = locate(pc.xs, pc.nx, pc.inv_dx, X, in_x);
        const int j = locate(pc.ys, pc.ny, pc.inv_dy, Y, in_y);
        float zhit = -INFINITY;
        if (in_x && in_y) {
            const float4* __restrict__ e = pc.ent + 2 * ((size_t)j * pc.nx + i);
            const float4 p = __ldg(e), q = __ldg(e + 1);
            if (q.w == 0.f) {
                const float lx = __fsub_rn(X, __ldg(pc.xs + i)), ly = __fsub_rn(Y, __ldg(pc.ys + j));
                const float E = fmaf(q.x, lx, fmaf(q.y, ly, q.z));
                const float z = fmaf(p.w, fminf(E, 0.f), fmaf(p.x, lx, fmaf(p.y, ly, p.z)));
                const float t = Z - z;
                if (t >= 0.f && t < max_d) zhit = z;
            } else {
                zhit = cast_down(g, X, Y, Z, max_d);
            }
        }
        float h = -INFINITY, hx = INFINITY, hy = INFINITY, hz = INFINITY;
        if (zhit != -INFINITY) {
            const float t = __fsub_rn(Z, zhit);
            hz = __fsub_rn(Z, t);
            hx = X;
            hy = Y;
            h = __fsub_rn(__fsub_rn(f.pz, hz), base_offset);
        }
        out[(size_t)env * out_stride + r] = h;
        if (hits) {
            float* p3 = hits + ((size_t)env * n_rays + r) * 3;
            p3[0] = hx;
            p3[1] = hy;
            p3[2] = hz;
        }
    }
}

int make_dev_grid(const RoverScanGrid* grid, ScanGridDev& g) {
    ROVER_CHECK(grid != nullptr, "rover_height_scan: grid is NULL");
    ROVER_CHECK(grid->n_levels >= 1 && grid->n_levels <= ROVER_MAX_LEVELS, "rover_height_scan: bad n_levels %d",
                grid->n_levels);
    ROVER_CHECK(grid->span >= 0 && grid->span <= 3, "rover_height_scan: bad span %d", grid->span);
    ROVER_CHECK(grid->cell_start != nullptr, "rover_height_scan: cell_start is NULL");
    ROVER_CHECK(grid->records != nullptr || grid->n_records == 0, "rover_height_scan: records is NULL");
    ROVER_CHECK((reinterpret_cast<uintptr_t>(grid->records) & 15) == 0, "rover_height_scan: records not 16B aligned");
    g.n_levels = grid->n_levels;
    g.span = grid->span;
    for (int l = 0; l < grid->n_levels; ++l) {
        const RoverScanLevel& s = grid->level[l];
        ROVER_CHECK(s.ncx > 0 && s.ncy > 0 && s.cell > 0.f, "rover_height_scan: bad level %d", l);
        g.level[l] = {s.ox, s.oy, s.cell, s.inv_cell, s.ncx, s.ncy, s.start_offset, 0};
    }
    g.cell_start = grid->cell_start;
    g.rec = reinterpret_cast<const float4*>(grid->records);
    return 0;
}

int launch_height_scan_pipelined(const float* pos_w, const float* quat_w, int n_envs, const float* ray_local,
                                 int n_rays, const ScanGridDev& g, const RoverPlaneCells* cells, float4 pattern_box,
                                 float max_d, float base_offset, float* out, int out_stride, float* hits,
                                 cudaStream_t stream);  // height_scan_pipelined.cu

int launch_height_scan_paired(const float* pos_w, const float* quat_w, int n_envs, const float* ray_local, int n_rays,
                              const ScanGridDev& g, const RoverPlaneCells* cells, float4 pattern_box, float max_d,
                              float base_offset, float* out, int out_stride, float* hits, uint16_t* obs_bf16,
                              int bf16_stride, int head_cols, cudaStream_t stream,
                              bool bf16_only = false);  // height_scan_paired.cu

// fallback of rover_height_scan_obs when variant 5 cannot run: mirror obs[:, 0:cols] into bf16
__global__ void obs_to_bf16_kernel(const float* __restrict__ obs, int obs_stride, int n_envs, int cols,
                                   __nv_bfloat16* __restrict__ dst, int dst_stride) {
    const size_t total = (size_t)n_envs * cols;
    for (size_t k = blockIdx.x * (size_t)blockDim.x + threadIdx.x; k < total; k += (size_t)gridDim.x * blockDim.x) {
        const size_t e = k / cols;
        const int c = (int)(k - e * cols);
        dst[e * dst_stride + c] = __float2bfloat16_rn(obs[e * obs_stride + c]);
    }
}

}  // namespace rover

extern "C" int rover_height_scan(const float* pos_w, const float* quat_w, int32_t n_envs,
                                 const float* ray_starts_local, int32_t n_rays, const float* pattern_box,
                                 const RoverScanGrid* grid, const RoverPlaneCells* cells, float max_distance,
                                 float base_offset, float* out_heights, int32_t out_stride, float* out_hits_w,
                                 int32_t variant, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0 && n_rays >= 0, "rover_height_scan: negative sizes");
    if (n_envs == 0 || n_rays == 0) return 0;
    ROVER_CHECK(pos_w && quat_w && ray_starts_local && out_heights, "rover_height_scan: NULL tensor");
    ROVER_CHECK(out_stride >= n_rays, "rover_height_scan: out_stride %d < n_rays %d", out_stride, n_rays);
    ScanGridDev g;
    if (int rc = make_dev_grid(grid, g)) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (variant == 0) {
        height_scan_direct_kernel<<<n_envs, kScanThreads, 0, s>>>(pos_w, quat_w, ray_starts_local, n_rays, g,
                                                                   max_distance, base_offset, out_heights, out_stride,
                                                                   out_hits_w);
        return check_launch("height_scan_direct_kernel");
    }
    // variants 1 (window re-based into shared memory, home grid) and 3 (per-CTA cp.async.bulk window) were measured slower
    // than their neighbours in round 1 and are retired; their numbers stay reserved
    ROVER_CHECK(variant != 1 && variant != 3, "rover_height_scan: variant %d was retired (use 0, 2, 4 or 5)", variant);
    if (variant == 2 || variant == 4 || variant == 5) {
        ROVER_CHECK(cells != nullptr, "rover_height_scan: variants 2, 4, 5 need the plane-cell table");
        ROVER_CHECK(cells->xs && cells->ys && cells->entries && cells->nx > 0 && cells->ny > 0,
                    "rover_height_scan: bad plane-cell table");
        ROVER_CHECK((reinterpret_cast<uintptr_t>(cells->entries) & 15) == 0,
                    "rover_height_scan: plane-cell entries not 16B aligned");
        if (variant == 5 && n_rays <= 1024) {
            ROVER_CHECK(pattern_box != nullptr, "rover_height_scan: variant 5 needs pattern_box (host, 4 floats)");
            const float4 box = make_float4(pattern_box[0], pattern_box[1], pattern_box[2], pattern_box[3]);
            return launch_height_scan_paired(pos_w, quat_w, n_envs, ray_starts_local, n_rays, g, cells, box,
                                             max_distance, base_offset, out_heights, out_stride, out_hits_w, nullptr, 0, 0, s);
        }
        if (variant >= 4 && n_rays <= 1024) {
            ROVER_CHECK(pattern_box != nullptr, "rover_height_scan: variant 4 needs pattern_box (host, 4 floats)");
            const float4 box = make_float4(pattern_box[0], pattern_box[1], pattern_box[2], pattern_box[3]);
            return launch_height_scan_pipelined(pos_w, quat_w, n_envs, ray_starts_local, n_rays, g, cells, box,
                                                max_distance, base_offset, out_heights, out_stride, out_hits_w, s);
        }
        // variant 2, and variants 4 / 5 with a pattern too large for their shared-memory tables
        PlaneCellsDev pc{cells->xs, cells->ys, reinterpret_cast<const float4*>(cells->entries), cells->nx, cells->ny,
                         cells->inv_dx, cells->inv_dy};
        height_scan_cells_kernel<<<n_envs, kScanThreads, 0, s>>>(pos_w, quat_w, ray_starts_local, n_rays, g, pc,
                                                                  max_distance, base_offset, out_heights, out_stride,
                                                                  out_hits_w);
        return check_launch("height_scan_cells_kernel");
    }
    return fail("rover_height_scan: unknown variant %d", variant);
}

// ---- host-buffer entry point: the call a caller with poses / heights in HOST memory makes
namespace rover {
struct HostScanStreams {
    cudaStream_t copy = nullptr;
    cudaEvent_t scanned[64] = {};
    cudaEvent_t done = nullptr;
    int device = -1;
};
// the poses' share of the work area, rounded up so that the heights start on a 64 KB boundary (the device-to-host DMA of
// 15.7 MB per step is what the end-to-end step costs; keep it on large-page-aligned source addresses)
static inline int64_t host_scan_pose_bytes(int64_t n_envs) { return ((7 * n_envs * 4 + 65535) / 65536) * 65536; }

static int host_scan_streams(HostScanStreams*& out) {
    static HostScanStreams per_device[64];
    int dev = 0;
    ROVER_CUDA(cudaGetDevice(&dev));
    ROVER_CHECK(dev >= 0 && dev < 64, "rover_height_scan_host: device ordinal %d out of range", dev);
    HostScanStreams& h = per_device[dev];
    if (h.device != dev) {
        ROVER_CUDA(cudaStreamCreateWithFlags(&h.copy, cudaStreamNonBlocking));
        for (auto& e : h.scanned) ROVER_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ROVER_CUDA(cudaEventCreateWithFlags(&h.done, cudaEventDisableTiming));
        h.device = dev;
    }
    out = &h;
    return 0;
}
}  // namespace rover

int rover::host_scan_sliced(const char* what, const float* pos_host, const float* quat_host, int n_envs, int n_rays,
                            float* out_host, int out_stride, void* work, int64_t work_bytes, int n_slices, cudaStream_t s,
                            const HostSliceScan& scan) {
    ROVER_CHECK(n_envs >= 0 && n_rays >= 0, "%s: negative sizes", what);
    const int64_t need = rover_height_scan_host_work_bytes(n_envs, out_stride);
    if (n_envs == 0 || n_rays == 0) return 0;
    ROVER_CHECK(pos_host && quat_host && out_host && work, "%s: NULL buffer", what);
    ROVER_CHECK(out_stride >= n_rays, "%s: out_stride %d < n_rays %d", what, out_stride, n_rays);
    ROVER_CHECK(work_bytes >= need && (reinterpret_cast<uintptr_t>(work) & 255) == 0,
                "%s: work area of %lld bytes (256-byte aligned) needed, got %lld", what, (long long)need,
                (long long)work_bytes);
    ROVER_CHECK(n_slices >= 1 && n_slices <= 64, "%s: n_slices %d not in [1, 64]", what, n_slices);
    HostScanStreams* hs = nullptr;
    if (int rc = host_scan_streams(hs)) return rc;
    float* d_pos = static_cast<float*>(work);
    float* d_quat = d_pos + 3 * (size_t)n_envs;
    float* d_out = reinterpret_cast<float*>(static_cast<unsigned char*>(work) + host_scan_pose_bytes(n_envs));
    ROVER_CUDA(cudaMemcpyAsync(d_pos, pos_host, 12 * (size_t)n_envs, cudaMemcpyHostToDevice, s));
    ROVER_CUDA(cudaMemcpyAsync(d_quat, quat_host, 16 * (size_t)n_envs, cudaMemcpyHostToDevice, s));
    const int slices = n_slices < n_envs ? n_slices : n_envs;
    if (slices == 1) {  // one launch, everything in order on the caller's stream (no second stream to join)
        if (int rc = scan(d_pos, d_quat, n_envs, d_out, s)) return rc;
        ROVER_CUDA(cudaMemcpyAsync(out_host, d_out, (size_t)n_envs * out_stride * 4, cudaMemcpyDeviceToHost, s));
        return 0;
    }
    for (int k = 0; k < slices; ++k) {
        // slice k's heights travel to the host on the copy stream while slice k + 1 is scanned on the caller's stream
        const int e0 = (int)((int64_t)n_envs * k / slices), e1 = (int)((int64_t)n_envs * (k + 1) / slices);
        if (int rc = scan(d_pos + 3 * (size_t)e0, d_quat + 4 * (size_t)e0, e1 - e0, d_out + (size_t)e0 * out_stride, s))
            return rc;
        ROVER_CUDA(cudaEventRecord(hs->scanned[k], s));
        ROVER_CUDA(cudaStreamWaitEvent(hs->copy, hs->scanned[k], 0));
        ROVER_CUDA(cudaMemcpyAsync(out_host + (size_t)e0 * out_stride, d_out + (size_t)e0 * out_stride,
                                   (size_t)(e1 - e0) * out_stride * 4, cudaMemcpyDeviceToHost, hs->copy));
    }
    // join: the caller's stream is complete when the heights are in host memory (and the work area may be reused)
    ROVER_CUDA(cudaEventRecord(hs->done, hs->copy));
    ROVER_CUDA(cudaStreamWaitEvent(s, hs->done, 0));
    return 0;
}

extern "C" int rover_height_scan_host(const float* pos_host, const float* quat_host, int32_t n_envs,
                                      const float* ray_starts_local, int32_t n_rays, const float* pattern_box,
                                      const RoverScanGrid* grid, const RoverPlaneCells* cells, float max_distance,
                                      float base_offset, float* out_host, int32_t out_stride, void* work, int64_t work_bytes,
                                      int32_t n_slices, int32_t variant, void* stream) {
    using namespace rover;
    return host_scan_sliced("rover_height_scan_host", pos_host, quat_host, n_envs, n_rays, out_host, out_stride, work,
                            work_bytes, n_slices, static_cast<cudaStream_t>(stream),
                            [&](const float* pos, const float* quat, int n, float* out, cudaStream_t s) {
                                return rover_height_scan(pos, quat, n, ray_starts_local, n_rays, pattern_box, grid, cells,
                                                         max_distance, base_offset, out, out_stride, nullptr, variant, s);
                            });
}

extern "C" int64_t rover_height_scan_host_work_bytes(int32_t n_envs, int32_t out_stride) {
    if (n_envs < 0 || out_stride < 0) return -1;
    return rover::host_scan_pose_bytes(n_envs) + (int64_t)n_envs * out_stride * 4;
}

static int height_scan_obs_impl(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                                int32_t n_rays, const float* pattern_box, const RoverScanGrid* grid,
                                const RoverPlaneCells* cells, float max_distance, float base_offset, float* obs,
                                int32_t obs_stride, int32_t head_cols, uint16_t* obs_bf16, int32_t bf16_stride, void* stream,
                                bool bf16_only) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0 && n_rays >= 0 && head_cols >= 0, "rover_height_scan_obs: negative sizes");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs && obs_bf16, "rover_height_scan_obs: NULL observation buffer");
    ROVER_CHECK(obs_stride >= head_cols + n_rays && bf16_stride >= head_cols + n_rays,
                "rover_height_scan_obs: row strides %d / %d < head_cols + n_rays = %d", obs_stride, bf16_stride,
                head_cols + n_rays);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool fused = cells != nullptr && cells->entries_planar != nullptr && n_rays >= 1 && n_rays <= 1024 &&
                       head_cols <= 32 && pattern_box != nullptr;
    if (fused) {
        ROVER_CHECK(pos_w && quat_w && ray_starts_local, "rover_height_scan_obs: NULL tensor");
        ROVER_CHECK(cells->xs && cells->ys && cells->entries && cells->nx > 0 && cells->ny > 0,
                    "rover_height_scan_obs: bad plane-cell table");
        ScanGridDev g;
        if (int rc = make_dev_grid(grid, g)) return rc;
        const float4 box = make_float4(pattern_box[0], pattern_box[1], pattern_box[2], pattern_box[3]);
        return launch_height_scan_paired(pos_w, quat_w, n_envs, ray_starts_local, n_rays, g, cells, box, max_distance,
                                         base_offset, obs + head_cols, obs_stride, nullptr, obs_bf16, bf16_stride, head_cols,
                                         s, bf16_only);
    }
    // any other table / pattern: the best variant that applies, then one conversion pass (the fp32 heights are written
    // on this path also in the bf16-only mode: it is the staging buffer of the conversion)
    const int variant = cells != nullptr ? 2 : 0;
    if (int rc = rover_height_scan(pos_w, quat_w, n_envs, ray_starts_local, n_rays, pattern_box, grid, cells, max_distance,
                                   base_offset, obs + head_cols, obs_stride, nullptr, variant, stream))
        return rc;
    obs_to_bf16_kernel<<<1184, 256, 0, s>>>(obs, obs_stride, n_envs, head_cols + n_rays,
                                            reinterpret_cast<__nv_bfloat16*>(obs_bf16), bf16_stride);
    return check_launch("obs_to_bf16_kernel");
}

extern "C" int rover_height_scan_obs(const float* pos_w, const float* quat_w, int32_t n_envs,
                                     const float* ray_starts_local, int32_t n_rays, const float* pattern_box,
                                     const RoverScanGrid* grid, const RoverPlaneCells* cells, float max_distance,
                                     float base_offset, float* obs, int32_t obs_stride, int32_t head_cols,
                                     uint16_t* obs_bf16, int32_t bf16_stride, void* stream) {
    return height_scan_obs_impl(pos_w, quat_w, n_envs, ray_starts_local, n_rays, pattern_box, grid, cells, max_distance,
                                base_offset, obs, obs_stride, head_cols, obs_bf16, bf16_stride, stream, false);
}

extern "C" int rover_height_scan_obs_bf16(const float* pos_w, const float* quat_w, int32_t n_envs,
                                          const float* ray_starts_local, int32_t n_rays, const float* pattern_box,
                                          const RoverScanGrid* grid, const RoverPlaneCells* cells, float max_distance,
                                          float base_offset, const float* obs_head, int32_t obs_stride, int32_t head_cols,
                                          uint16_t* obs_bf16, int32_t bf16_stride, void* stream) {
    return height_scan_obs_impl(pos_w, quat_w, n_envs, ray_starts_local, n_rays, pattern_box, grid, cells, max_distance,
                                base_offset, const_cast<float*>(obs_head), obs_stride, head_cols, obs_bf16, bf16_stride,
                                stream, true);
}
