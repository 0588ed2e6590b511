// Device structs and helpers shared by the height-scan kernels.
#pragma once
#include <functional>

#include "common.cuh"

namespace rover {

struct ScanLevelDev {
    float ox, oy, cell, inv_cell;
    int ncx, ncy, start_offset, pad;
};

struct ScanGridDev {
    int n_levels;
    int span;
    ScanLevelDev level[ROVER_MAX_LEVELS];
    const int* __restrict__ cell_start;
    const float4* __restrict__ rec;
};

struct PlaneCellsDev {
    const float* __restrict__ xs;
    const float* __restrict__ ys;
    const float4* __restrict__ ent;
    int nx, ny;
    float inv_dx, inv_dy;
};

struct SensorFrame {
    float cw, sz;      // yaw-only unit quaternion (cw, 0, 0, sz)
    float px, py, pz;  // sensor position
};

// ORBIT yaw_quat (A.1): yaw = atan2(2(wz+xy), 1-2(yy+zz)); (cos(yaw/2),0,0,sin(yaw/2)) / max(norm, 1e-9)
__device__ __forceinline__ SensorFrame make_frame(const float* __restrict__ pos, const float* __restrict__ q) {
    const float w = q[0], x = q[1], y = q[2], z = q[3];
    const float siny = __fmul_rn(2.f, __fadd_rn(__fmul_rn(w, z), __fmul_rn(x, y)));
    const float cosy = __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(__fmul_rn(y, y), __fmul_rn(z, z))));
    const float half = __fdiv_rn(atan2f(siny, cosy), 2.f);
    const float s = sinf(half), c = cosf(half);
    const float n = fmaxf(sqrtf(__fadd_rn(__fmul_rn(c, c), __fmul_rn(s, s))), 1e-9f);
    SensorFrame f;
    f.cw = __fdiv_rn(c, n);
    f.sz = __fdiv_rn(s, n);
    f.px = pos[0];
    f.py = pos[1];
    f.pz = pos[2];
    return f;
}

// ORBIT quat_apply (A.1) specialised to (cw,0,0,sz):  v + w*t + xyz x t,  t = 2 * (xyz x v); then + pos.
__device__ __forceinline__ void ray_origin(const SensorFrame& f, float vx, float vy, float vz, float& X, float& Y,
                                           float& Z) {
    const float tx = __fmul_rn(-__fmul_rn(f.sz, vy), 2.f);
    const float ty = __fmul_rn(__fmul_rn(f.sz, vx), 2.f);
    const float rx = __fadd_rn(__fadd_rn(vx, __fmul_rn(f.cw, tx)), -__fmul_rn(f.sz, ty));
    const float ry = __fadd_rn(__fadd_rn(vy, __fmul_rn(f.cw, ty)), __fmul_rn(f.sz, tx));
    X = __fadd_rn(rx, f.px);
    Y = __fadd_rn(ry, f.py);
    Z = __fadd_rn(vz, f.pz);
}

__device__ __forceinline__ int cell_of(float x, float o, float inv) {
    // identical to scan_grid.cell_index_f32: floor((x - o) * inv) in fp32, no contraction
    const float f = floorf(__fmul_rn(__fsub_rn(x, o), inv));
    return (int)fminf(fmaxf(f, -1.0e9f), 1.0e9f);
}

__device__ __forceinline__ void test_record(const float4 r0, const float4 r1, const float4 r2, float lx, float ly,
                                            float Z, float max_d, float& best) {
    const float e0 = fmaf(r0.x, lx, fmaf(r0.y, ly, r0.z));
    const float e1 = fmaf(r0.w, lx, fmaf(r1.x, ly, r1.y));
    const float e2 = fmaf(r1.z, lx, fmaf(r1.w, ly, r2.x));
    const float z = fmaf(r2.y, lx, fmaf(r2.z, ly, r2.w));
    const float t = Z - z;
    if (fminf(e0, fminf(e1, e2)) >= 0.f && t >= 0.f && t < max_d) best = fmaxf(best, z);
}

// The body of the host-buffer entry points (height_scan.cu): copy the poses into the work area, run `scan` on each of
// `n_slices` slices of environments and copy each slice's heights to out_host, slice k's copy overlapping the scan of
// slice k + 1.  `what` names the entry point in error messages.
using HostSliceScan = std::function<int(const float* pos, const float* quat, int n_envs, float* out, cudaStream_t s)>;
int host_scan_sliced(const char* what, const float* pos_host, const float* quat_host, int n_envs, int n_rays,
                     float* out_host, int out_stride, void* work, int64_t work_bytes, int n_slices, cudaStream_t s,
                     const HostSliceScan& scan);

}  // namespace rover
