// Shapes, packed-weight layout and PTX wrappers shared by the policy kernels (policy.cu: tile-serial v1;
// policy_ws.cu: warp-specialised v2).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>

#include <cstdlib>

#include "common.cuh"
#include "rng.cuh"

namespace rover {

constexpr int kPolThreads = 256;
constexpr int kTileM = 128;
constexpr int kObsCols = 965;
constexpr int kEncIn = 961;       // obs[:, 3:964]
constexpr int kEncInOffset = 3;
constexpr int kChunkK = 64;
constexpr int kNumChunks = 16;    // observation columns [0, 1024) in chunks of 64; columns outside [3, 964) are zeroed
constexpr int kAPlane = kTileM * 16 + 16;  // A plane stride (bytes), +16 B skew: conflict-free 16 B stores per plane
constexpr int kNumLayers = 6;
constexpr int kStagesF = 4;  // fp32 observation stages (prefetch distance 3 chunks)
constexpr int kStagesW = 3;  // layer-0 weight-chunk stages (prefetch distance 2 chunks)

// padded layer shapes: K (multiple of 16), N (multiple of 16)
__host__ __device__ constexpr int layer_k(int l) { return l == 0 ? 1024 : l == 1 ? 80 : l == 2 ? 64 : l == 3 ? 256 : l == 4 ? 160 : 128; }
__host__ __device__ constexpr int layer_n(int l) { return l == 0 ? 80 : l == 1 ? 64 : l == 2 ? 256 : l == 3 ? 160 : l == 4 ? 128 : 16; }
__host__ __device__ constexpr int layer_k_real(int l) { return l == 0 ? 961 : l == 1 ? 80 : l == 2 ? 64 : l == 3 ? 256 : l == 4 ? 160 : 128; }
__host__ __device__ constexpr int layer_n_real(int l) { return l == 0 ? 80 : l == 1 ? 60 : l == 2 ? 256 : l == 3 ? 160 : l == 4 ? 128 : 2; }

// packed blob: [W0: 16 chunks x (8 planes x 80 rows x 16 B)] [W1..W5: (K/8 planes x N rows x 16 B)] [biases fp32]
constexpr int kW0ChunkBytes = 8 * 80 * 16;  // 10,240
__host__ __device__ constexpr int weight_bytes(int l) { return l == 0 ? kNumChunks * kW0ChunkBytes : (layer_k(l) / 8) * layer_n(l) * 16; }
__host__ __device__ constexpr int weight_offset(int l) {
    int off = 0;
    for (int i = 0; i < l; ++i) off += weight_bytes(i);
    return off;
}
constexpr int kBiasOffset = weight_offset(kNumLayers);
__host__ __device__ constexpr int bias_offset(int l) {
    int off = kBiasOffset;
    for (int i = 0; i < l; ++i) off += layer_n(i) * 4;
    return off;
}
constexpr int kPackedBytes = bias_offset(kNumLayers);

// ---------------------------------------------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t sptr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(unsigned long long* b, uint32_t n) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sptr(b)), "r"(n) : "memory");
}
__device__ __forceinline__ void mb_expect_tx(unsigned long long* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sptr(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_wait(unsigned long long* b, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(sptr(b)), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, unsigned long long* b) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(sptr(dst)),
                 "l"(src), "r"(bytes), "r"(sptr(b))
                 : "memory");
}
__device__ __forceinline__ void tma_2d(void* dst, const CUtensorMap* map, int x, int y, unsigned long long* b) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
            "r"(sptr(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(sptr(b))
        : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor, K-major, SWIZZLE_NONE: LBO = byte stride between the two 8-element K chunks of one
// MMA (= plane stride), SBO = byte stride between 8-row groups (= 128 B), version 1 (Blackwell)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((128u >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
// instruction descriptor, kind::f16: D = F32, A = B = BF16, both K-major, M = 128
__device__ __forceinline__ uint32_t make_idesc(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
}
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(unsigned long long* b) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(sptr(b)) : "memory");
}
__device__ __forceinline__ void tmem_ld8_nowait(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float leaky(float x) { return x > 0.f ? x : 0.01f * x; }

// clamp(x, lo, hi) that keeps a NaN NaN, as torch.clamp does: PTX max.NaN / min.NaN (one FMNMX each, like fmaxf /
// fminf, which return the other operand and would turn a NaN into a bound)
__device__ __forceinline__ float clamp_keep_nan(float x, float lo, float hi) {
    float y;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(y) : "f"(x), "f"(lo));
    asm("min.NaN.f32 %0, %0, %1;" : "+f"(y) : "f"(hi));
    return y;
}

// skrl 1.1.0 GaussianMixin.act for one environment (models.py:65-67: clip_log_std, min -20, max 2): log_std clamped to
// [-20, 2], the reparameterised sample mean + std * eps clipped to the action box [-1, 1], log-prob of the clipped action
// under Normal(mean, std) summed over the two action dimensions.  Both clamps keep NaN (torch.clamp): a NaN mean -- a
// missed ray's -inf height through the network -- gives a NaN action and log-prob, not the action -1.  Shared by
// gaussian_act_kernel and the sampling epilogue of the forward pass, so both give the same bits.
__device__ __forceinline__ float gaussian_sample(const float (&mean)[2], const float (&log_std)[2], const float (&eps)[2],
                                                 float (&actions)[2]) {
    float lp = 0.f;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float ls = clamp_keep_nan(log_std[j], -20.f, 2.f);
        const float sd = expf(ls);
        const float m = mean[j];
        const float a = clamp_keep_nan(fmaf(sd, eps[j], m), -1.f, 1.f);
        actions[j] = a;
        const float d = a - m;
        lp += -(d * d) / (2.f * sd * sd) - ls - 0.91893853320467274178f;
    }
    return lp;
}

// What the forward pass needs to sample in its last epilogue (rover_policy_act): eps = normal2({seed, step}, env_offset + env)
struct SampleArgs {
    const float* log_std;      // [2]
    unsigned long long* rng;   // {seed, step}, advanced once per launch
    uint32_t env_offset;
    float* actions;            // [N, 2]
    float* log_prob;           // [N] or nullptr
};

constexpr int kWsPlane = kTileM * 16;  // bytes between K-adjacent core matrices of a 128-row A operand (SWIZZLE_NONE)

// shared-memory matrix descriptor, K-major SWIZZLE_128B (the layout a 128-byte-wide SWIZZLE_128B TMA box lands in):
// 8-row groups are 1024 B apart (SBO), LBO is not used by swizzled K-major layouts, layout type 2, version 1
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((1024u >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

__device__ __forceinline__ void mb_arrive(unsigned long long* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(sptr(b)) : "memory");
}
__device__ __forceinline__ void layer_group_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
        "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]),
          "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]),
          "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

// 16 accumulator columns nq .. nq + 15 of one tile row: +bias -> LeakyReLU -> bf16 -> two A planes of the next layer
__device__ __forceinline__ void epilogue_16(const uint32_t* raw, int nq, const float* __restrict__ bias,
                                            unsigned char* __restrict__ act, int row, const float* inject) {
    float v[16];
#pragma unroll
    for (int j4 = 0; j4 < 4; ++j4) {
        const float4 b = *reinterpret_cast<const float4*>(bias + nq + 4 * j4);  // broadcast LDS.128
        const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 4; j += 2) {
            // two columns per FADD2 / FMUL2 (per-lane IEEE fp32: same values as the scalar ops, half the issue slots)
            unsigned long long acc2, b2, x2, t2;
            const unsigned long long slope2 = 0x3c23d70a3c23d70aull;  // (0.01f, 0.01f)
            asm("mov.b64 %0, {%1, %2};" : "=l"(acc2) : "r"(raw[4 * j4 + j]), "r"(raw[4 * j4 + j + 1]));
            asm("mov.b64 %0, {%1, %2};" : "=l"(b2) : "f"(bb[j]), "f"(bb[j + 1]));
            asm("add.rn.f32x2 %0, %1, %2;" : "=l"(x2) : "l"(acc2), "l"(b2));
            asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(t2) : "l"(x2), "l"(slope2));
            const float x0 = __uint_as_float((unsigned)(x2 & 0xffffffffull)), x1 = __uint_as_float((unsigned)(x2 >> 32));
            const float t0 = __uint_as_float((unsigned)(t2 & 0xffffffffull)), t1 = __uint_as_float((unsigned)(t2 >> 32));
            v[4 * j4 + j] = fmaxf(x0, t0);  // == x > 0 ? x : 0.01 x (LeakyReLU, slope 0.01)
            v[4 * j4 + j + 1] = fmaxf(x1, t1);
        }
    }
    if (inject != nullptr && nq == 48) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[12 + j] = inject[j];
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        uint4 o;
        o.x = pack_bf16(v[8 * h + 0], v[8 * h + 1]);
        o.y = pack_bf16(v[8 * h + 2], v[8 * h + 3]);
        o.z = pack_bf16(v[8 * h + 4], v[8 * h + 5]);
        o.w = pack_bf16(v[8 * h + 6], v[8 * h + 7]);
        *reinterpret_cast<uint4*>(act + ((nq >> 3) + h) * kWsPlane + row * 16) = o;
    }
}

// Epilogue of one layer for one tile row: D[row, 0:n_cols] -> +bias -> LeakyReLU -> bf16 -> A planes of the next layer.
// inject != nullptr: columns 60..63 are replaced by inject[0..3] (layer 2 consumes [e(60), obs[:, 0:4]]).
// Batches of 32 columns per tcgen05.ld (then a 16-column tail): the load's latency (~50 cycles before the first value can
// be used; ptxas schedules every load directly in front of its first use, so a source-level double buffer does not overlap
// it with the previous batch's arithmetic) is paid once per 32 columns.  profiles/microbench/tmem_read.cu: TMEM delivers
// 160-250 B/cycle/SM, the conversion arithmetic is what an epilogue costs.
__device__ __forceinline__ void epilogue_to_act(uint32_t taddr, int n_cols, const float* __restrict__ bias,
                                                unsigned char* __restrict__ act, int row, const float* inject) {
    int nq = 0;
    for (; nq + 32 <= n_cols; nq += 32) {
        uint32_t raw[32];
        tmem_ld32_nowait(taddr + nq, raw);
        tmem_wait_ld();
        epilogue_16(raw, nq, bias, act, row, inject);
        epilogue_16(raw + 16, nq + 16, bias, act, row, inject);
    }
    if (nq < n_cols) {
        uint32_t raw[16];
        tmem_ld16_nowait(taddr + nq, raw);
        tmem_wait_ld();
        epilogue_16(raw, nq, bias, act, row, inject);
    }
}

}  // namespace rover
