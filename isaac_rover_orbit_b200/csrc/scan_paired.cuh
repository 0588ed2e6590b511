// Building blocks of the paired (packed-fp32) plane-cell height scan, shared by height_scan_paired.cu (variant 5) and
// fused_scan_policy.cu (the scan whose heights feed the tcgen05 policy without leaving the SM): lane <-> ray mapping,
// stage layout, packed-fp32 helpers, the per-pair resolver, the rare out-of-line paths and the lane-parallel producer.
// Functions that touch the shared tables are templated on the shared-memory struct (members vx, vy, xpair, ypair and
// sm_vz()) so that both kernels lay out their own shared memory.
#pragma once
#include <cuda_bf16.h>

#include "scan_pipe.cuh"

#ifndef ROVER_SCAN_DBG
#define ROVER_SCAN_DBG 0  // bring-up experiments only: 1 = consumers skip the ray work, 2 = TMA loads only for the first ring pass
#endif

namespace rover {

#if ROVER_SCAN_DBG == 3  // timeline of CTA 0 and CTA 100 in SM cycles since the CTA started (bring-up builds only)
__device__ unsigned long long g_scan_dbg[2][512];
__device__ unsigned long long g_scan_cta[2][256];  // [0][b] = globaltimer at CTA start, [1][b] = at its last warp's end
__device__ __forceinline__ unsigned long long dbg_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define DBG_STAMP(slot)                                                                             \
    do {                                                                                            \
        if (lane == 0 && (blockIdx.x == 0 || blockIdx.x == 100) && (slot) < 512)                    \
            g_scan_dbg[blockIdx.x != 0][slot] = (unsigned long long)(clock64() - dbg_t0);           \
    } while (0)
#define DBG_STAMP_ANY(slot)                                                                         \
    do {                                                                                            \
        if ((blockIdx.x == 0 || blockIdx.x == 100) && (slot) < 512)                                 \
            g_scan_dbg[blockIdx.x != 0][slot] = (unsigned long long)(clock64() - dbg_t0);           \
    } while (0)
#else
#define DBG_STAMP(slot) \
    do {                \
    } while (0)
#define DBG_STAMP_ANY(slot) \
    do {                    \
    } while (0)
#endif

#ifndef ROVER_PAIR_WARPS
#define ROVER_PAIR_WARPS 15
#endif
// 1 producer + 15 consumer warps = 512 threads x 128 registers = the whole register file.  (Round 1 ran 14 consumers;
// round 2, same box, profiles/time_scan_sizes.py: 15 consumers 21.5 / 56.3 / 184.3 us at 4096 / 16384 / 65536 envs against
// 22.5 / 56.4 / 189.4 us for 14; 17 consumers at 96 registers spill and take 25.6 / 62.5 / 207.9 us.)
constexpr int kPairConsumerWarps = ROVER_PAIR_WARPS;
constexpr int kPairThreads = 32 * (1 + kPairConsumerWarps);
constexpr int kPairStages = 8;          // ring depth (data)
#ifndef ROVER_PAIR_EARLY
#define ROVER_PAIR_EARLY 8
#endif
constexpr int kPairEarly = ROVER_PAIR_EARLY;  // windows whose TMA load is issued in the prologue (<= kPairStages)
constexpr int kPairFullBars = 32;       // `full` barriers: four per stage, see the note on phase aliasing below
constexpr int kPairWin = 26;            // window cells per axis
constexpr int kPairPitch = 27;          // cells per staged row: odd, so that consecutive rows shift by one 16-byte bank
                                        // group and a quarter-warp's LDS.128 of 8 neighbouring cells is conflict free
constexpr int kPairPlane = kPairWin * kPairPitch;             // float4 per plane
constexpr uint32_t kPairStageBytes = 2u * kPairPlane * 16u;   // bytes one TMA load delivers
#ifndef ROVER_PAIR_CHUNK
#define ROVER_PAIR_CHUNK 256
#endif
constexpr int kPairBatch = 128;         // rays per pass of a warp: 2 pair slots x 32 lanes x 2 rays
constexpr int kPairChunk = ROVER_PAIR_CHUNK;  // rays per work unit (a whole number of batches)
static_assert(kPairChunk % kPairBatch == 0, "a chunk is a whole number of batches");
constexpr int kPairMaxRays = 1024;      // pattern held in shared memory (3 float arrays)
constexpr int kPairMaxLines = 1024;     // grid-line pairs per axis held in shared memory
constexpr float kFloorMagic = 12582912.0f;  // 1.5 * 2^23: fl_rm(v + magic) has floor(v) in its mantissa for |v| < 2^22
constexpr int kFloorMagicBits = 0x4B400000;

// Lane <-> ray mapping inside a batch of 128 rays [b0, b0 + 128): lane l, slot u (0/1) resolves the pair
//   A = b0 + 32u + l,  B = A + 64.
// One instruction therefore serves 32 CONSECUTIVE rays (0.1 m apart: a quarter-warp touches ~4 cells, not 8, and
// its stores fill whole sectors), while the two rays of a pair still come out of one LDS.64: the pattern arrays are
// held in slot order, slot(A) = b0 + 64u + 2l, slot(B) = slot(A) + 1.
__host__ __device__ __forceinline__ int ray_of_slot(int s) {
    const int j = s & 127;
    return (s & ~127) + 64 * (j & 1) + 32 * (j >> 6) + ((j & 63) >> 1);
}
__host__ __device__ __forceinline__ int slot_of_ray(int r) {
    const int j = r & 127;
    return (r & ~127) + 64 * ((j >> 5) & 1) + 2 * (j & 31) + (j >> 6);
}

struct PairHeader {
    float cw, sz, px, py;
    float pz;
    int ic0, jr0, ncols;
    int nrows, mode, pad0, pad1;  // mode 1: window staged in shared memory, 0: read the table from global memory
};

// ---- packed fp32 pairs (one 64-bit register pair; lo = ray 2k, hi = ray 2k+1)
typedef unsigned long long f32x2;

// The constants of the consumer loop for one environment: (v, v) register pairs for the packed-fp32 chain and the
// shared-memory offsets of the window.  A consumer warp builds them from the header for every 256-ray chunk (4 x ~70 of
// the ~2070 warp-instructions an environment costs).  Having the PRODUCER publish them ready to load
// (ROVER_PAIR_CTX_FROM_PRODUCER) was built and measured in round 2: slower (see height_scan_paired.cu).
struct __align__(16) PairCtx {
    f32x2 CW, SZ, NSZ, S2, NS2, PX, PY, PZ, NWX0, NWY0, IDX, IDY, MAGIC, BASE, NEG0, ZFLAT;
    float pz, max_d;
    uint32_t xoff, yoff, eoff;  // byte offsets into shared memory of the window's line pairs / p plane
    uint32_t cmax, rmax;        // last column / row of the window
    uint32_t pad;
};
static_assert(sizeof(PairCtx) == 160, "PairCtx is loaded as ten 16-byte words");

// Planes of the window: p[row][col] = (a, b, c, k), q[row][col] = (A, B, C, tag) of cell (jr0 + row, ic0 + col).
// (With the interleaved 32-byte entries of the other variants every LDS.128 of a quarter-warp could reach only the
// even 16-byte bank groups: 2.5x the minimum number of shared-memory wavefronts, measured with ncu.)
struct __align__(128) PairStage {
    float4 p[kPairPlane];
    float4 q[kPairPlane];
    PairHeader hdr;
    PairCtx ctx;  // only with ROVER_PAIR_CTX_FROM_PRODUCER (valid when hdr.mode == 1)
};
static_assert(offsetof(PairStage, q) == kPairPlane * 16, "planes must be contiguous: one 3-D TMA box fills both");

struct PairSmem {
    PairStage stage[kPairStages];
    float vx[kPairMaxRays], vy[kPairMaxRays], vz[kPairMaxRays];
    LinePair2 xpair[kPairMaxLines], ypair[kPairMaxLines];
    unsigned long long full_bar[kPairFullBars];
    unsigned long long empty_bar[kPairStages];
    int next_chunk;  // dynamic hand-out of (environment, chunk) work units, in order
};
// Phase aliasing: a consumer warp does not visit every environment, so it may reach environment E while the TMA load
// of an earlier environment on the same barrier is still in flight (loads complete out of order, and an environment
// whose window is not staged completes its barrier as soon as the header is published); a parity wait on a barrier
// two phases behind would pass on a stale phase.  Environment E therefore signals on barrier E % F with parity
// (E / F) & 1, F = kPairFullBars, and the wait is sound when E - F has completed.  With W = 15 consumer warps and
// S = 8 stages: the warp's previous work unit is at most W units back, so its environment is >= E - W (one chunk per
// environment, <= 256 rays, is the worst case); that environment was issued, the producer issues strictly in order
// and issues environment X only after X - S was consumed, so every environment <= E - W - S was consumed.  F >= W + S
// makes E - F one of them.  (F = 16 held only at >= 2 chunks per environment.)  The same bound holds for a dynamic
// hand-out: of the W units handed out just before E's, at most W - 1 can still be held by the other warps.  Environments
// E < F wait on a barrier's first phase, which only their own arrivals complete.
static_assert(kPairFullBars >= kPairConsumerWarps + kPairStages, "full barriers: see the phase-aliasing note");

static_assert(sizeof(PairSmem) <= 227 * 1024, "PairSmem exceeds the shared memory of one SM");
__device__ __forceinline__ float sm_vz(const PairSmem& sm, int slot) { return sm.vz[slot]; }

// Where a resolved height goes.  kSinkGlobal: the fp32 output row (+ the bf16 mirror row with kBf) -- variant 5.
// kSinkOperand / kSinkOperandAndGlobal (fused_scan_policy.cu): bf16 into the K-major SWIZZLE_NONE shared-memory operand of
// the layer-0 MMA (row = env slot of the batch, k = observation column), optionally also the fp32 output row.
constexpr int kSinkGlobal = 0, kSinkOperand = 1, kSinkOperandAndGlobal = 2;
constexpr int kOperandLbo = 272;   // bytes between K-adjacent core matrices of the observation operand: 16 env rows x 16 B
                                   // + 16 B skew, so that the 2-byte stores of a warp (32 consecutive k) spread over the banks
constexpr int kOperandHead = 4;    // observation columns in front of the scan (actions(2), distance, angle)
constexpr int kOperandDropK = 964; // obs[:, 964] is not an input of the policy (models.py:95 slices [3:-1]); its weight is
                                   // zero, but a missed ray there is -inf and -inf * 0 = NaN: store 0 instead
__device__ __forceinline__ void operand_store(unsigned char* __restrict__ row, int ray, float h) {
    const int k = kOperandHead + ray;
    const __nv_bfloat16 v = __float2bfloat16_rn(k == kOperandDropK ? 0.f : h);
    *reinterpret_cast<__nv_bfloat16*>(row + (k >> 3) * kOperandLbo + (k & 7) * 2) = v;
}

// one 3-D TMA tile load (UTMALDG): box (set in the tensor map) = kPairPitch cells x kPairWin rows x 2 planes of the
// planar table, starting at cell (col, row); lands as PairStage::p followed by PairStage::q
__device__ __forceinline__ void tma_load_window_planar(void* dst, const CUtensorMap* tmap, int col, int row,
                                                       unsigned long long* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::
            "r"(s_addr(dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(col * 4), "r"(row), "r"(0), "r"(s_addr(bar))
        : "memory");
}

__device__ __forceinline__ f32x2 pk(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ f32x2 dup(float v) { return pk(v, v); }
__device__ __forceinline__ float lo_of(f32x2 v) {
    return __uint_as_float((unsigned)(v & 0xffffffffull));
}
__device__ __forceinline__ float hi_of(f32x2 v) {
    return __uint_as_float((unsigned)(v >> 32));
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// a * b rounded once, as a product that ptxas cannot contract with a following add: ptxas (12.9) fuses
// mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even with -fmad=false, which would drop the reference's intermediate
// rounding.  fma(a, b, -0.0) == fl(a * b) for every input (sign of zero included); `nz` holds -0.0 behind a value the
// compiler cannot fold, so the instruction stays an FFMA2 and the following FADD2 stays an add.
__device__ __forceinline__ f32x2 mul2_unfused(f32x2 a, f32x2 b, f32x2 nz) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(nz));
    return r;
}
__device__ __forceinline__ f32x2 add2_rm(f32x2 a, f32x2 b) {  // round toward -inf
    f32x2 r;
    asm("add.rm.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// The context of one environment, built from its header (producer side of variant 5; per chunk in the fused kernel).
// smem_base: address of the dynamic shared memory the offsets are relative to.
template <class SM>
__device__ __forceinline__ PairCtx make_pair_ctx(const PairHeader& h, const SM& sm, const PairStage& st,
                                                 const unsigned char* smem_base, float inv_dx, float inv_dy, float base_offset,
                                                 float max_d, float vz0, int opaque_zero) {
    PairCtx cx;
    const float sz2 = __fmul_rn(h.sz, 2.f);  // fl(fl(sz*v)*2) == fl(fl(2*sz)*v): scaling by 2 is exact
    const float wx0 = sm.xpair[h.ic0].lo, wy0 = sm.ypair[h.jr0].lo;
    cx.CW = dup(h.cw), cx.SZ = dup(h.sz), cx.NSZ = dup(-h.sz), cx.S2 = dup(sz2), cx.NS2 = dup(-sz2);
    cx.PX = dup(h.px), cx.PY = dup(h.py), cx.PZ = dup(h.pz);
    cx.NWX0 = dup(-wx0), cx.NWY0 = dup(-wy0), cx.IDX = dup(inv_dx), cx.IDY = dup(inv_dy);
    cx.MAGIC = dup(kFloorMagic), cx.BASE = dup(base_offset);
    cx.NEG0 = dup(__uint_as_float(0x80000000u | (unsigned)opaque_zero));  // -0.0, opaque to the compiler
    cx.pz = h.pz, cx.max_d = max_d;
    cx.ZFLAT = dup(__fadd_rn(vz0, h.pz));
    cx.cmax = (uint32_t)(h.ncols - 1), cx.rmax = (uint32_t)(h.nrows - 1);
    cx.xoff = (uint32_t)(reinterpret_cast<const unsigned char*>(sm.xpair + h.ic0) - smem_base);
    cx.yoff = (uint32_t)(reinterpret_cast<const unsigned char*>(sm.ypair + h.jr0) - smem_base);
    cx.eoff = (uint32_t)(reinterpret_cast<const unsigned char*>(st.p) - smem_base);
    cx.pad = 0u;
    return cx;
}

// Rare path (a): a ray whose cell guess missed, that lies on the closed far border / outside the grid, or sits in a
// general cell.  Out of line so that it does not raise the register pressure of the consumer loop.
template <class SM>
static __device__ __noinline__ void pair_resolve_deferred_ray(const SM* sm, const PairStage* st, const ScanGridDev& g,
                                                              float inv_dx, float inv_dy, float X, float Y, float Z, float pz,
                                                              float max_d, float base_offset, float* __restrict__ out,
                                                              __nv_bfloat16* __restrict__ out_bf) {
    const PairHeader& h = st->hdr;
    const int cmax = h.ncols - 1, rmax = h.nrows - 1;
    const LinePair2* xp = sm->xpair + h.ic0;
    const LinePair2* yp = sm->ypair + h.jr0;
    const float wx0 = xp[0].lo, wy0 = yp[0].lo, wx1 = xp[cmax].hi, wy1 = yp[rmax].hi;
    float zhit = -INFINITY;
    if (X >= wx0 && X <= wx1 && Y >= wy0 && Y <= wy1) {
        int ci = min(max(__float2int_rd((X - wx0) * inv_dx), 0), cmax);
        int cj = min(max(__float2int_rd((Y - wy0) * inv_dy), 0), rmax);
        while (ci > 0 && X < xp[ci].lo) --ci;
        while (ci < cmax && X >= xp[ci].hi) ++ci;
        while (cj > 0 && Y < yp[cj].lo) --cj;
        while (cj < rmax && Y >= yp[cj].hi) ++cj;
        const int e = cj * kPairPitch + ci;
        const float4 q = st->q[e];
        zhit = (q.w == 0.f) ? eval_cell(st->p[e], q, __fsub_rn(X, xp[ci].lo), __fsub_rn(Y, yp[cj].lo), Z, max_d)
                            : walk_home_grid(g, X, Y, Z, max_d);
    }
    float height;
    store_result(pz, X, Y, Z, zhit, base_offset, &height, nullptr);
    if (out != nullptr) *out = height;  // (out == nullptr: the bf16-only observation mode)
    if (out_bf != nullptr) *out_bf = __float2bfloat16_rn(height);
}

// Rare path (b): a chunk of an environment whose window is not staged (too large, not covered on a non-uniform
// lattice, or more grid lines than the shared table holds).
template <class SM>
static __device__ __noinline__ void pair_resolve_chunk_from_global(const SM* sm, int lane, int r_begin, int r_end,
                                                                   const PairHeader h, const ScanGridDev& g,
                                                                   const PlaneCellsDev& pc, float max_d, float base_offset,
                                                                   float* __restrict__ out_row,
                                                                   __nv_bfloat16* __restrict__ bf_row) {
    const float sz2 = __fmul_rn(h.sz, 2.f);
    for (int r = r_begin + lane; r < r_end; r += 32) {
        const int sl = slot_of_ray(r);
        const float vx = sm->vx[sl], vy = sm->vy[sl];
        const float tx = -__fmul_rn(sz2, vy), ty = __fmul_rn(sz2, vx);
        const float X = __fadd_rn(__fadd_rn(__fadd_rn(vx, __fmul_rn(h.cw, tx)), -__fmul_rn(h.sz, ty)), h.px);
        const float Y = __fadd_rn(__fadd_rn(__fadd_rn(vy, __fmul_rn(h.cw, ty)), __fmul_rn(h.sz, tx)), h.py);
        const float Z = __fadd_rn(sm_vz(*sm, sl), h.pz);
        float height;
        store_result(h.pz, X, Y, Z, resolve_from_global(g, pc, X, Y, Z, max_d), base_offset, &height, nullptr);
        if (out_row != nullptr) out_row[r] = height;
        if (bf_row != nullptr) bf_row[r] = __float2bfloat16_rn(height);
    }
}

// One pair slot: rays (r, r+1).  Everything that can go wrong is deferred, so the body is branch-free up to the stores.
// Returns a 2-bit mask of the rays that need the rare path.
// kFull: the whole batch lies inside the pattern (no per-ray validity predicates); kFlatZ: every ray starts at the
// same local z (grid patterns), so Z is a per-environment constant.
// kBf = 1: the heights are also stored as bf16 (round to nearest even) at ob[0] / ob[64] -- the observation mirror that
// feeds rover_policy_forward_bf16; kBf = 2: ONLY the bf16 mirror is stored (the fp32 row is not written).
template <bool kFull, bool kFlatZ, int kBf, int kSink = kSinkGlobal, class SM = PairSmem>
__device__ __forceinline__ unsigned resolve_pair(const unsigned char* __restrict__ smem, const SM& sm,
                                                 const PairCtx& c, int slot, int ray_a, int n_rays,
                                                 float* __restrict__ o, __nv_bfloat16* __restrict__ ob,
                                                 unsigned char* __restrict__ operand_row = nullptr) {
    const bool valid0 = kFull || ray_a < n_rays, valid1 = kFull || ray_a + 64 < n_rays;
    const int idx = slot;  // slots beyond the pattern hold zeros
    const f32x2 VX = *reinterpret_cast<const f32x2*>(sm.vx + idx);
    const f32x2 VY = *reinterpret_cast<const f32x2*>(sm.vy + idx);
    // ORBIT quat_apply_yaw + pos, same roundings as ray_origin(): tx = -(2sz * vy), ty = 2sz * vx,
    // X = ((vx + cw*tx) + (-(sz*ty))) + px, Y = ((vy + cw*ty) + sz*tx) + py, Z = vz + pz.  Negations are exact.
    const f32x2 TX = mul2(c.NS2, VY), TY = mul2(c.S2, VX);
    const f32x2 X = add2(add2(add2(VX, mul2_unfused(c.CW, TX, c.NEG0)), mul2_unfused(c.NSZ, TY, c.NEG0)), c.PX);
    const f32x2 Y = add2(add2(add2(VY, mul2_unfused(c.CW, TY, c.NEG0)), mul2_unfused(c.SZ, TX, c.NEG0)), c.PY);
    f32x2 Z = c.ZFLAT;
    if constexpr (!kFlatZ) Z = add2(*reinterpret_cast<const f32x2*>(sm.vz + idx), c.PZ);
    // window-relative cell guess: floor((X - wx0) * inv_dx) left in the mantissa, clamped on the raw bits
    const f32x2 BX = add2_rm(mul2(add2(X, c.NWX0), c.IDX), c.MAGIC);
    const f32x2 BY = add2_rm(mul2(add2(Y, c.NWY0), c.IDY), c.MAGIC);
    float nz[2];
    unsigned defer = 0;
    bool keep[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const float x = k ? hi_of(X) : lo_of(X), y = k ? hi_of(Y) : lo_of(Y);
        // one unsigned min clamps both ends: bits below the bias (negative index, NaN ...) wrap to a huge value
        const uint32_t bi = min(__float_as_uint(k ? hi_of(BX) : lo_of(BX)) - (uint32_t)kFloorMagicBits, c.cmax);
        const uint32_t bj = min(__float_as_uint(k ? hi_of(BY) : lo_of(BY)) - (uint32_t)kFloorMagicBits, c.rmax);
        const float2 xp = *reinterpret_cast<const float2*>(smem + (c.xoff + bi * 8u));
        const float2 yp = *reinterpret_cast<const float2*>(smem + (c.yoff + bj * 8u));
#if ROVER_SCAN_DBG == 5  // timing experiment: conflict-free entry loads (results are wrong)
        const uint32_t e = c.eoff + ((threadIdx.x & 31) * 16u) + ((bj + bi) & 1u) * 1024u;
        const float4 q = *reinterpret_cast<const float4*>(smem + e + 512);
        const float4 p = *reinterpret_cast<const float4*>(smem + e);
        const bool fast = (x >= xp.x) & (x < xp.y) & (y >= yp.x) & (y < yp.y);
#else
        const uint32_t e = c.eoff + bj * (uint32_t)(kPairPitch * 16) + bi * 16u;
        const float4 q = *reinterpret_cast<const float4*>(smem + e + kPairPlane * 16);
        const float4 p = *reinterpret_cast<const float4*>(smem + e);
        const bool fast = (x >= xp.x) & (x < xp.y) & (y >= yp.x) & (y < yp.y) & (q.w == 0.f);
#endif
        const float lx = __fsub_rn(x, xp.x), ly = __fsub_rn(y, yp.x);
        const float E = fmaf(q.x, lx, fmaf(q.y, ly, q.z));
        // -z, with z = fma(k, min(E, 0), fma(a, lx, fma(b, ly, c))) exactly as eval_cell (negation commutes with rn)
        nz[k] = fmaf(-p.w, fminf(E, 0.f), -fmaf(p.x, lx, fmaf(p.y, ly, p.z)));
        const bool valid = k ? valid1 : valid0;
        keep[k] = valid && fast;
        defer |= (valid && !fast) ? (1u << k) : 0u;
    }
    // reference rounding chain: t = Z - z, hit.z = Z - t, height = (pos.z - hit.z) - offset; miss -> -inf
    const f32x2 T = add2(Z, pk(nz[0], nz[1]));
    const f32x2 H = sub2(sub2(c.PZ, sub2(Z, T)), c.BASE);
    const float t0 = lo_of(T), t1 = hi_of(T);
    const float h0 = (t0 >= 0.f && t0 < c.max_d) ? lo_of(H) : -INFINITY;
    const float h1 = (t1 >= 0.f && t1 < c.max_d) ? hi_of(H) : -INFINITY;
    if (kSink != kSinkOperand && kBf != 2) {
        if (keep[0]) o[0] = h0;
        if (keep[1]) o[64] = h1;
    }
    if (kBf) {
        if (keep[0]) ob[0] = __float2bfloat16_rn(h0);
        if (keep[1]) ob[64] = __float2bfloat16_rn(h1);
    }
    if (kSink != kSinkGlobal) {
        if (keep[0]) operand_store(operand_row, ray_a, h0);
        if (keep[1]) operand_store(operand_row, ray_a + 64, h1);
    }
    return defer;
}

// ---- producer side: one environment per lane
struct ProducerEnv {
    float pv[3], qv[4];  // raw pose
    float cw, sz, px, py, pz;
    int ic0, jr0, ncols, nrows;
    bool have, ok;
};

__device__ __forceinline__ void producer_load(ProducerEnv& e, int it, int n_iter, const float* __restrict__ pos_w,
                                              const float* __restrict__ quat_w) {
    e.have = it < n_iter;
    const size_t env = (size_t)blockIdx.x + (size_t)(e.have ? it : 0) * gridDim.x;
#pragma unroll
    for (int k = 0; k < 3; ++k) e.pv[k] = __ldg(pos_w + 3 * env + k);
#pragma unroll
    for (int k = 0; k < 4; ++k) e.qv[k] = __ldg(quat_w + 4 * env + k);
    e.px = e.pv[0], e.py = e.pv[1], e.pz = e.pv[2];
}

// window from the position alone: every ray origin lies within pattern_radius of (px, py)
__device__ __forceinline__ void producer_window(ProducerEnv& e, const PlaneCellsDev& pc, float radius) {
    const float gx_lo = __ldg(pc.xs), gy_lo = __ldg(pc.ys);
    const int ic1 = min(max(guess_col(e.px + radius, gx_lo, pc.inv_dx) + 1, 0), pc.nx - 1);
    const int jr1 = min(max(guess_col(e.py + radius, gy_lo, pc.inv_dy) + 1, 0), pc.ny - 1);
    e.ic0 = min(max(guess_col(e.px - radius, gx_lo, pc.inv_dx) - 1, 0), pc.nx - 1);
    e.jr0 = min(max(guess_col(e.py - radius, gy_lo, pc.inv_dy) - 1, 0), pc.ny - 1);
    e.ncols = ic1 - e.ic0 + 1;
    e.nrows = jr1 - e.jr0 + 1;
}

__device__ __forceinline__ void producer_frame(ProducerEnv& e) {
    const SensorFrame f = make_frame(e.pv, e.qv);
    e.cw = f.cw, e.sz = f.sz;
}

// does the window fit the stage and (for lattices where the arithmetic guess is not exact +-1) cover the pattern?
template <class SM>
__device__ __forceinline__ void producer_verdict(ProducerEnv& e, const SM& sm, const PlaneCellsDev& pc,
                                                 float radius, bool lines_in_smem) {
    bool ok = lines_in_smem && (e.ncols <= kPairWin) && (e.nrows <= kPairWin);
    if (ok) {
        const float gx_lo = sm.xpair[0].lo, gx_hi = sm.xpair[pc.nx - 1].hi;
        const float gy_lo = sm.ypair[0].lo, gy_hi = sm.ypair[pc.ny - 1].hi;
        ok = (sm.xpair[e.ic0].lo <= fmaxf(e.px - radius, gx_lo)) &&
             (sm.xpair[e.ic0 + e.ncols - 1].hi >= fminf(e.px + radius, gx_hi)) &&
             (sm.ypair[e.jr0].lo <= fmaxf(e.py - radius, gy_lo)) &&
             (sm.ypair[e.jr0 + e.nrows - 1].hi >= fminf(e.py + radius, gy_hi));
    }
    e.ok = ok;
}

}  // namespace rover
