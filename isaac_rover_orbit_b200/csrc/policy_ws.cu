// Gaussian policy forward, warp-specialised (v2): the observation stream of tile i+1 overlaps layers 1-5 of tile i.
//
// Why (ncu on v1, profiles/r01_policy_v1_tcgen05.md): v1 runs one 128-env tile at a time per SM with every phase
// behind a CTA-wide barrier -- issue slots 15 % busy, tensor pipe 8 %, HBM idle during layers 1-5; 130 us at cfg-4
// where the 254 MB of fp32 observations alone take 39 us at the measured HBM rate.
//
// Roles (one persistent CTA per SM, 11 warps -- 15 with fp32 observations --, all 512 TMEM columns):
//   warp 8      TMA producer: obs chunks (128 envs x 32 columns fp32, SWIZZLE_128B) into a 5-stage ring, running ahead
//               across tiles (up to 80 KB of HBM reads in flight per SM).
//   warp 10     W0 producer: the matching 5 KB slice of the packed W0 image into a 3-stage ring.  (A single producer
//               thread serving both rings stalled the observation stream on the shallower W0 ring: 84 us.)
//   warps 4-7   converters: fp32 stage -> bf16 A operand (K-major core-matrix layout), 2-stage ring; warps 11-14: the
//               second converter warpgroup (each thread converts half of its row's chunk).
//   warp 9      layer-0 MMA issuer: 2 tcgen05.mma per chunk into D0[tile parity] (two 80-column accumulators);
//               tcgen05.commit frees the A / W0 stages and, after the last chunk, publishes D0.
//   warps 0-3   layer group: epilogue of layer l (tcgen05.ld -> +bias -> LeakyReLU -> bf16) writes the A operand of
//               layer l+1; its thread 0 streams W1..W5 (bulk copies into one 40 KB buffer; W3 in two K halves) and
//               issues the MMAs of layers 1-5 into one 256-column accumulator.
// Same arithmetic as v1 (bf16 operands, fp32 accumulation, same K order inside a layer), so the means are identical.
//
// kDual (fp32 observations): policy AND value network in one pass over the observation (models.py:89-102 + :151-162; the
// rollout needs both every step).  The tile's A operand meets both W0 images (two 80-column accumulators per D0 buffer),
// the layer group then runs layers 1-5 once per network.  TMEM: 2 x 160 D0 columns + a 192-column accumulator, so layer 2
// (N = 256) runs as two N halves and its input operand sits in planes 24-31, which the first half's output (planes
// 0-15) does not touch.  Same arithmetic per network, so both outputs equal the two single passes bit for bit.
//
// kDual && kBf16In: the same two-network pass over the bf16 observation.  Each 64-column TMA stage meets both W0 images
// (the policy's four K = 16 MMAs into D0[buf] columns 0-79, then the value network's four into columns 80-159); 352
// threads, no converter warps; the TMEM plan is the fp32 dual plan.  Shared memory: the 4-stage observation ring of the
// dual layout, and a W0 ring of TWO 20 KB stages (both networks' 10 KB chunks) overlaid on a_bf16[] + w0[] (46 KB).
//
// Encoder width: `enc_in` = R (1 <= R <= kEncInMax) is a launch argument.  Layer 0 streams ceil((3 + R) / 32) fp32 or
// ceil((3 + R) / 64) bf16 chunks of observation columns and as many W0 ring stages; the tensor map ends the observation
// at column 4 + R (fp32; the converters zero columns outside [3, 3 + R)) or 3 + R (bf16) and zero-fills the tail chunk.
// Layers 1-5 and the biases sit w0_shift(R) bytes further along the blob than at R = 961.  Nothing else depends on R:
// W0 is streamed, so no stage, TMEM column or epilogue grows with it.
#include "policy_common.cuh"

#ifndef ROVER_POLICY_DBG
#define ROVER_POLICY_DBG 0  // 1: timeline of CTA 0 in SM cycles (bring-up builds only, profiles/policy_timeline.py)
#endif

namespace rover {

#if ROVER_POLICY_DBG
__device__ long long g_pol_dbg[2048];
__device__ unsigned long long g_pol_cta[2][256];  // globaltimer (ns) at CTA start / end
#define PDBG(slot)                                                                     \
    do {                                                                               \
        if (blockIdx.x == 0 && (slot) < 2048) g_pol_dbg[slot] = clock64() - dbg_t0;    \
    } while (0)
#else
#define PDBG(slot) \
    do {           \
    } while (0)
#endif

constexpr int kWsThreads = 352;        // bf16 observations: warps 0-10
constexpr int kWsThreadsF32 = 480;     // fp32 observations: + warps 11-14, a second converter warpgroup
constexpr int kWsChunkK = 32;
constexpr int kWsStagesF = 5;
constexpr int kWsStagesFDual = 4;  // the second W0 image takes the shared memory of one observation stage
constexpr int kWsStagesA = 2;
constexpr int kWsStagesW = 3;
constexpr int kWsW0Chunk = (kWsChunkK / 8) * 80 * 16;  // 5,120 B of the packed W0 image per chunk
constexpr int kWsWBuf = 40 * 1024;                 // largest single weight load: W4, or one K half of W3
constexpr uint32_t kWsColD0 = 0, kWsColD0Stride = 128, kWsColAcc = 256;
constexpr uint32_t kWsColD0StrideDual = 160, kWsColAccDual = 320;  // D0[buf] = [policy 80 | value 80]; accumulator: 192 columns
constexpr int kWsBiasFloats = 80 + 64 + 256 + 160 + 128 + 16;

static_assert(weight_bytes(1) <= kWsWBuf && weight_bytes(2) <= kWsWBuf && weight_bytes(3) == 2 * kWsWBuf &&
                  weight_bytes(4) <= kWsWBuf && weight_bytes(5) <= kWsWBuf,
              "weight buffer plan");
static_assert(kW0ChunkBytes == 2 * kWsW0Chunk, "a 32-column chunk is half of a packed 64-column chunk");
// bf16-observation mode (kBf16In): the observation arrives as bf16 [N, stride] (written by the height scan, see
// rover_height_scan_obs), so a TMA tile of 64 columns x tile rows (128 B per row, SWIZZLE_128B) IS the A operand of
// the MMA (canonical K-major SWIZZLE_128B layout) -- no conversion stage, half the HBM bytes.
constexpr int kBfChunkK = 64;
constexpr int kBfStagesW = 3;                 // 10 KB W0 chunks in the space of a_bf16[] + w0[]
constexpr int kBfStagesWDual = 2;             // 2 x 10 KB (policy + value) W0 chunks in the same space of the dual layout

template <bool kDual>
struct WsSmemT {
    static constexpr int kNets = kDual ? 2 : 1;
    static constexpr int kStagesFT = kDual ? kWsStagesFDual : kWsStagesF;
    float stage_f[kStagesFT][kTileM * kWsChunkK];         // 5 (4) x 16 KB, TMA destinations (1024-byte aligned)
    unsigned char a_bf16[kWsStagesA][4 * kWsPlane];       // 2 x 8 KB   } bf16-observation mode: three 10 KB W0
    unsigned char w0[kWsStagesW][kNets * kWsW0Chunk];     // 3 x 5 KB   } chunks live in these two arrays
    unsigned char act[32 * kWsPlane];                     // A operand of layers 1..5 (K <= 256): 64 KB
    unsigned char w[kWsWBuf];                             // weights of the current layer
    float bias[kNets][kWsBiasFloats];
    unsigned long long f_full[kWsStagesF], f_empty[kWsStagesF];
    unsigned long long a_full[kWsStagesA], a_empty[kWsStagesA];
    unsigned long long w0_full[kWsStagesW], w0_empty[kWsStagesW];
    unsigned long long d0_full[2], d0_empty[2];
    unsigned long long w_full, acc_done;
    uint32_t tmem_base;
};
using WsSmem = WsSmemT<false>;
static_assert(sizeof(WsSmem) + 1024 <= 227 * 1024 && sizeof(WsSmemT<true>) + 1024 <= 227 * 1024,
              "WsSmem exceeds the shared memory of one SM");
static_assert(kWsBiasFloats * 4 == kPackedBytes - kBiasOffset, "bias block of the packed blob");
static_assert(offsetof(WsSmem, w0) == offsetof(WsSmem, a_bf16) + kWsStagesA * 4 * kWsPlane &&
                  kBfStagesW * kW0ChunkBytes <= kWsStagesA * 4 * kWsPlane + kWsStagesW * kWsW0Chunk,
              "bf16-observation mode: W0 ring overlays a_bf16[] + w0[]");
static_assert(kTileM * kBfChunkK * 2 == kTileM * kWsChunkK * 4, "both modes use the same 16 KB stages");
static_assert(offsetof(WsSmemT<true>, w0) == offsetof(WsSmemT<true>, a_bf16) + kWsStagesA * 4 * kWsPlane &&
                  kBfStagesWDual * 2 * kW0ChunkBytes <= kWsStagesA * 4 * kWsPlane + kWsStagesW * 2 * kWsW0Chunk &&
                  (kBfStagesWDual + 1) * 2 * kW0ChunkBytes > kWsStagesA * 4 * kWsPlane + kWsStagesW * 2 * kWsW0Chunk,
              "bf16 two-network mode: two (not three) W0 stages of both networks overlay a_bf16[] + w0[]");
static_assert(kBfStagesWDual <= kWsStagesW, "w0_full[] / w0_empty[] cover the ring");

// kDual: `packed` = policy, `packed2` = value network, outputs `mean` [N, 2] and `value2` [N]; else one network
// (value_head: linear [N] output instead of tanh [N, 2]).
// kSample (policy head): the last epilogue also samples skrl's GaussianMixin.act -- eps = normal2({seed, step},
// env_offset + env) in registers, then gaussian_sample(), the function gaussian_act_kernel runs -- and stores `actions`
// and `log_prob` beside `mean`.  {seed, step} is taken once per CTA after griddepcontrol.wait; the launch advances the
// step once (rng.cuh, take_step).
template <bool kBf16In, bool kDual = false, bool kSample = false>
__global__ void __launch_bounds__(kBf16In ? kWsThreads : kWsThreadsF32, 1)
policy_forward_ws_kernel(const __grid_constant__ CUtensorMap obs_map, const float* __restrict__ obs, int obs_stride,
                         int n_envs, int tile_rows, const unsigned char* __restrict__ packed, float* __restrict__ mean,
                         int value_head, const unsigned char* __restrict__ packed2, float* __restrict__ value2,
                         const __grid_constant__ SampleArgs sample, int enc_in) {
    using Smem = WsSmemT<kDual>;
    constexpr int kNets = Smem::kNets, kStagesFK = Smem::kStagesFT;
    constexpr uint32_t kColD0Stride = kDual ? kWsColD0StrideDual : kWsColD0Stride, kColAcc = kDual ? kWsColAccDual : kWsColAcc;
    extern __shared__ unsigned char smem_dyn[];
    // 1024-byte alignment (SWIZZLE_128B atoms) by pointer arithmetic on the __shared__ array, so that the compiler keeps
    // the address space (an integer round-trip turns every access into a generic LD/ST)
    Smem& sm = *reinterpret_cast<Smem*>(smem_dyn + ((1024u - (sptr(smem_dyn) & 1023u)) & 1023u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // A tile holds tile_rows <= 128 environments (multiple of 8, chosen by the launcher so that the tiles fill whole
    // rounds of the grid: 65536 envs on 148 SMs -> 586 tiles of 112 instead of 512 of 128 = 3.96 instead of 3.46 -> 4
    // rounds).  The MMAs stay M = 128; accumulator rows >= tile_rows hold garbage and are never stored.
    const int n_tiles = (n_envs + tile_rows - 1) / tile_rows;
    constexpr int kChunkK = kBf16In ? kBfChunkK : kWsChunkK;        // observation columns per chunk
    const int n_chunks = (kEncInOffset + enc_in + kChunkK - 1) / kChunkK;  // layer-0 K chunks: columns [0, 3 + R)
    const int w_shift = w0_shift(enc_in);                           // layers 1-5 and biases behind the W0 chunks
    const int blob_bytes = kPackedBytes + w_shift;
    constexpr int kStagesW = kBf16In ? (kDual ? kBfStagesWDual : kBfStagesW) : kWsStagesW;
    constexpr int kW0Chunk = kBf16In ? kW0ChunkBytes : kWsW0Chunk;  // bytes of ONE packed W0 image per chunk
    constexpr int kW0Stage = kNets * kW0Chunk;                      // bytes of a W0 ring stage
    const uint32_t chunk_bytes = (uint32_t)tile_rows * 128u;        // 32 fp32 or 64 bf16 columns per row
    unsigned char* const w0_ring = kBf16In ? &sm.a_bf16[0][0] : &sm.w0[0][0];
#if ROVER_POLICY_DBG
    const long long dbg_t0 = clock64();
    if (threadIdx.x == 0 && blockIdx.x < 256) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        g_pol_cta[0][blockIdx.x] = t;
    }
#endif

    if (tid == 8 * 32) {
        // the producer sets up its own ring and starts the first loads before the CTA-wide barrier below
        asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&obs_map)) : "memory");
        for (int i = 0; i < kStagesFK; ++i) {
            mb_init(&sm.f_full[i], 1);
            mb_init(&sm.f_empty[i], kBf16In ? 1 : 8);  // converter warps, or the commit of the MMAs that read the stage
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        // the observation is what the kernel in front of this one writes: under a programmatic dependent launch
        // (common.cuh) everything above -- and the weight loads, the TMEM allocation of the other warps -- overlaps its tail
        grid_dependency_wait();
        if ((int)blockIdx.x < n_tiles)
            for (int c = 0; c < kStagesFK && c < n_chunks; ++c) {
                mb_expect_tx(&sm.f_full[c], chunk_bytes);
                tma_2d(sm.stage_f[c], &obs_map, c * kChunkK, blockIdx.x * tile_rows, &sm.f_full[c]);
            }
    }
    if (tid == 0) {
        for (int i = 0; i < kWsStagesA; ++i) {
            mb_init(&sm.a_full[i], 8);  // the eight converter warps
            mb_init(&sm.a_empty[i], 1);  // tcgen05.commit
        }
        for (int i = 0; i < kWsStagesW; ++i) {
            mb_init(&sm.w0_full[i], 1);
            mb_init(&sm.w0_empty[i], 1);  // tcgen05.commit
        }
        for (int i = 0; i < 2; ++i) {
            mb_init(&sm.d0_full[i], 1);   // tcgen05.commit
            mb_init(&sm.d0_empty[i], 1);  // thread 0 of the layer group
        }
        mb_init(&sm.w_full, 1);
        mb_init(&sm.acc_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {  // one warp allocates all 512 TMEM columns (one CTA per SM)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sptr(&sm.tmem_base)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    __shared__ RngKey s_key;    // kSample: {seed, step} of this launch (unused otherwise)
    grid_dependency_wait();     // every thread, before anything of the predecessor's is read or `mean` is written
    grid_dependency_trigger();  // (the sampling kernel behind this one only saves its launch latency)

    if (warp == 8) {
        // =============================================================== TMA producer
        if (lane == 0) {
            int sf = 0;
            uint32_t pf = 0;  // completed passes over the ring (parity)
            int dbg_g = 0;
            bool first = true;  // chunks 0 .. kStagesFK-1 of the first tile were issued in the prologue
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int row0 = tile * tile_rows;
                for (int c = 0; c < n_chunks; ++c) {
                    if (!(first && c < kStagesFK)) {
                        mb_wait(&sm.f_empty[sf], (pf & 1u) ^ 1u);
                        mb_expect_tx(&sm.f_full[sf], chunk_bytes);
                        tma_2d(sm.stage_f[sf], &obs_map, c * kChunkK, row0, &sm.f_full[sf]);
                    }
                    if (dbg_g < 128) PDBG(dbg_g);
                    ++dbg_g;
                    if (++sf == kStagesFK) sf = 0, ++pf;
                }
                first = false;
            }
        }
    } else if (warp == 10) {
        // =============================================================== W0 producer
        if (lane == 0) {
            int sw = 0;
            uint32_t pw = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                for (int c = 0; c < n_chunks; ++c) {
                    mb_wait(&sm.w0_empty[sw], (pw & 1u) ^ 1u);
                    mb_expect_tx(&sm.w0_full[sw], kW0Stage);
                    bulk_g2s(w0_ring + sw * kW0Stage, packed + (size_t)c * kW0Chunk, kW0Chunk, &sm.w0_full[sw]);
                    if (kDual)
                        bulk_g2s(w0_ring + sw * kW0Stage + kW0Chunk, packed2 + (size_t)c * kW0Chunk, kW0Chunk, &sm.w0_full[sw]);
                    if (++sw == kStagesW) sw = 0, ++pw;
                }
            }
        }
    } else if (warp == 9) {
        // =============================================================== layer-0 MMA issuer
        if (lane == 0) {
            const uint32_t idesc0 = make_idesc(layer_n(0));
            int sa = 0, sw = 0, i = 0;
            uint32_t pa = 0, pw = 0;
            int dbg_g = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++i) {
                const int buf = i & 1;
                mb_wait(&sm.d0_empty[buf], (((uint32_t)i >> 1) & 1u) ^ 1u);  // the layer group has drained D0[buf]
                tc_fence_after();
                const uint32_t d0 = tmem + kWsColD0 + buf * kColD0Stride;
                for (int c = 0; c < n_chunks; ++c) {
                    if (kBf16In) mb_wait(&sm.f_full[sa], pa & 1u);  // sa / pa walk the 5-stage TMA ring in this mode
                    else mb_wait(&sm.a_full[sa], pa & 1u);
                    mb_wait(&sm.w0_full[sw], pw & 1u);
                    tc_fence_after();
                    const uint32_t b0 = sptr(w0_ring + sw * kW0Stage);
                    if (kBf16In && kDual) {
                        const uint32_t a0 = sptr(sm.stage_f[sa]);
#pragma unroll
                        for (int net = 0; net < 2; ++net)
#pragma unroll
                            for (int j = 0; j < kBfChunkK / 16; ++j)
                                umma(d0 + net * 80, make_desc_sw128(a0 + j * 32),
                                     make_desc(b0 + net * kW0Chunk + j * 2 * 80 * 16, 80 * 16), idesc0, (c | j) != 0);
                        umma_commit(&sm.f_empty[sa]);
                    } else if (kBf16In) {
                        const uint32_t a0 = sptr(sm.stage_f[sa]);
#pragma unroll
                        for (int j = 0; j < kBfChunkK / 16; ++j)  // 16 bf16 = 32 B further along K inside the 128 B rows
                            umma(d0, make_desc_sw128(a0 + j * 32), make_desc(b0 + j * 2 * 80 * 16, 80 * 16), idesc0, (c | j) != 0);
                        umma_commit(&sm.f_empty[sa]);  // the TMA stage is free once these MMAs retire
                    } else {
                        const uint32_t a0 = sptr(sm.a_bf16[sa]);
#pragma unroll
                        for (int net = 0; net < kNets; ++net)
#pragma unroll
                            for (int j = 0; j < kWsChunkK / 16; ++j)
                                umma(d0 + net * 80, make_desc(a0 + j * 2 * kWsPlane, kWsPlane),
                                     make_desc(b0 + net * kW0Chunk + j * 2 * 80 * 16, 80 * 16), idesc0, (c | j) != 0);
                        umma_commit(&sm.a_empty[sa]);  // A stage and W0 stage are free once these MMAs retire
                    }
                    if (dbg_g < 128) PDBG(512 + dbg_g);
                    ++dbg_g;
                    umma_commit(&sm.w0_empty[sw]);
                    if (++sa == (kBf16In ? kStagesFK : kWsStagesA)) sa = 0, ++pa;
                    if (++sw == kStagesW) sw = 0, ++pw;
                }
                umma_commit(&sm.d0_full[buf]);
            }
        }
    } else if (warp >= 4 && kBf16In) {
        // bf16-observation mode: no conversion stage; these warps only pull the packed weights into L2
        for (int off = (tid - 128) * 128; off < blob_bytes; off += 128 * 128) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(packed + off));
            if (kDual) asm volatile("prefetch.global.L2 [%0];" ::"l"(packed2 + off));
        }
    } else if (warp >= 4) {
        // =============================================================== converters: fp32 stage -> bf16 A operand
        // first the packed weights into L2 (326 KB; after an L2 flush every layer's first load was a cold miss that the
        // layer group waited for: 21 k instead of 13 k cycles for the first tile)
        // Two warpgroups (warps 4-7 and 11-14): a thread converts HALF of its row's chunk (planes 2 * half, 2 * half + 1).
        // With one warpgroup a chunk took 506 cycles -- the wait -> LDS -> pack -> STS -> fence -> arrive chain of one warp
        // per scheduler -- which bounds the stream whenever the observation comes from L2 (the closed loop: 8.2 us per tile).
        const int half = warp >= 11 ? 1 : 0;
        const int row = half ? tid - kWsThreads : tid - 128;  // tile row
        for (int off = (half * 128 + row) * 128; off < blob_bytes; off += 256 * 128) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(packed + off));
            if (kDual) asm volatile("prefetch.global.L2 [%0];" ::"l"(packed2 + off));
        }
        const int sx = row & 7;     // SWIZZLE_128B: 16-byte unit u of row r sits at unit u ^ (r & 7)
        int sf = 0, sa = 0;
        uint32_t pf = 0, pa = 0;
        int dbg_g = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            for (int c = 0; c < n_chunks; ++c) {
                mb_wait(&sm.f_full[sf], pf & 1u);
                if (tid == 128 && dbg_g < 128) PDBG(128 + dbg_g);
                mb_wait(&sm.a_empty[sa], (pa & 1u) ^ 1u);
                if (tid == 128 && dbg_g < 128) PDBG(256 + dbg_g);
                const unsigned char* src = reinterpret_cast<const unsigned char*>(sm.stage_f[sf]) + row * (kWsChunkK * 4);
                unsigned char* dst = sm.a_bf16[sa] + row * 16;
#pragma unroll
                for (int pl = 0; pl < kWsChunkK / 16; ++pl) {
                    const int plane = 2 * half + pl;
                    if (row >= tile_rows) break;  // rows beyond the tile: never loaded, never stored
                    const float4 lo = *reinterpret_cast<const float4*>(src + (((2 * plane) ^ sx) << 4));
                    const float4 hi = *reinterpret_cast<const float4*>(src + (((2 * plane + 1) ^ sx) << 4));
                    float v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
                    if (c == 0 || c == n_chunks - 1) {  // encoder input = observation columns [3, 3 + R) (models.py:95)
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const int col = c * kWsChunkK + plane * 8 + j;
                            if (col < kEncInOffset || col >= kEncInOffset + enc_in) v[j] = 0.f;
                        }
                    }
                    uint4 o;
                    o.x = pack_bf16(v[0], v[1]);
                    o.y = pack_bf16(v[2], v[3]);
                    o.z = pack_bf16(v[4], v[5]);
                    o.w = pack_bf16(v[6], v[7]);
                    *reinterpret_cast<uint4*>(dst + plane * kWsPlane) = o;
                }
                fence_async_smem();  // the bf16 stage is read by the tensor core (async proxy)
                __syncwarp();
                if (lane == 0) {
                    mb_arrive(&sm.a_full[sa]);
                    mb_arrive(&sm.f_empty[sf]);
                }
                if (tid == 128 && dbg_g < 128) PDBG(384 + dbg_g);
                ++dbg_g;
                if (++sf == kStagesFK) sf = 0, ++pf;
                if (++sa == kWsStagesA) sa = 0, ++pa;
            }
        }
    } else {
        // =============================================================== layer group (warps 0-3): layers 1..5
        const int row = tid;  // TMEM lane == tile row; warp w may touch lanes 32w .. 32w+31
        const uint32_t t_lane = (uint32_t)(warp * 32) << 16;
        const uint32_t acc = tmem + kColAcc;
        const uint32_t a0 = sptr(sm.act), b0 = sptr(sm.w);
        uint32_t ph_w = 0, ph_acc = 0;
        // weights of layer l (or one K half of layer 3) of network `net` into the single weight buffer; only thread 0
        // calls these
        auto load_w = [&](int net, int byte_offset, int bytes) {
            mb_expect_tx(&sm.w_full, (uint32_t)bytes);
            bulk_g2s(sm.w, (kDual && net ? packed2 : packed) + w_shift + byte_offset, (uint32_t)bytes, &sm.w_full);
        };
        // D[128 x nn] (+)= A[planes plane0 ..] x W^T, k_steps MMAs of K = 16; then commit to acc_done.  The weight image in
        // the buffer has n_image rows per plane; the MMA uses rows n_row0 .. n_row0 + nn - 1 of it.
        auto issue_mma = [&](int plane0, int k_steps, int nn, bool accumulate, int n_image, int n_row0) {
            tc_fence_after();
            mb_wait(&sm.w_full, ph_w);
            const uint32_t idesc = make_idesc(nn);
            for (int j = 0; j < k_steps; ++j)
                umma(acc, make_desc(a0 + (plane0 + 2 * j) * kWsPlane, kWsPlane),
                     make_desc(b0 + j * 2 * n_image * 16 + n_row0 * 16, n_image * 16), idesc, accumulate || j != 0);
            umma_commit(&sm.acc_done);
        };
        auto wait_acc = [&]() {
            mb_wait(&sm.acc_done, ph_acc);
            ph_acc ^= 1u;
            tc_fence_after();
        };
        auto publish_act = [&]() {  // this thread's A-operand stores are visible to the tensor core; TMEM reads done
            tc_fence_before();
            fence_async_smem();
            layer_group_sync();
        };
        if (tid == 0) load_w(0, weight_offset(1), weight_bytes(1));
        {   // biases: cold global loads that only this group needs (and only ~one tile-time from now), so they stay out
            // of the CTA-wide prologue that the observation stream waits for
            constexpr int kPer = (kWsBiasFloats + 127) / 128;
            float b[kNets][kPer];
#pragma unroll
            for (int net = 0; net < kNets; ++net)
#pragma unroll
                for (int k = 0; k < kPer; ++k)
                    b[net][k] = tid + 128 * k < kWsBiasFloats
                                    ? __ldg(reinterpret_cast<const float*>((kDual && net ? packed2 : packed) + w_shift + kBiasOffset) + tid + 128 * k)
                                    : 0.f;
#pragma unroll
            for (int net = 0; net < kNets; ++net)
#pragma unroll
                for (int k = 0; k < kPer; ++k)
                    if (tid + 128 * k < kWsBiasFloats) sm.bias[net][tid + 128 * k] = b[net][k];
            if (kSample && tid == 0) s_key = take_step(sample.rng, gridDim.x, true);  // (after griddepcontrol.wait above)
            layer_group_sync();
        }
        // layer 2's input operand: planes 0.. (one network), planes 24..31 in the two-network pass, where layer 2 runs
        // as two N halves and the first half's output (planes 0..15) must not overwrite it
        constexpr int kA2Plane = kDual ? 24 : 0;
        int i = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++i) {
            const int buf = i & 1;
            const int grow = tile * tile_rows + row;
            const bool live = row < tile_rows && grow < n_envs;
            float inject[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (kBf16In)  // obs points at bf16 rows; the values are re-rounded to bf16 below either way
                    inject[j] = live ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(obs)[(size_t)grow * obs_stride + j])
                                     : 0.f;
                else
                    inject[j] = live ? __ldg(obs + (size_t)grow * obs_stride + j) : 0.f;
            }
#define LDBG(k)                                                       \
    do {                                                              \
        if (tid == 0 && i < 8 && net == 0) PDBG(1024 + 16 * i + (k)); \
    } while (0)
#pragma unroll
            for (int net = 0; net < kNets; ++net) {
                const float* bias = sm.bias[net];
                const bool last_net = net == kNets - 1;
                // ---- layer 0 epilogue: D0[buf][net] -> A1 (80 columns)
                LDBG(0);
                if (net == 0) {
                    mb_wait(&sm.d0_full[buf], ((uint32_t)i >> 1) & 1u);
                    tc_fence_after();
                }
                LDBG(1);
                epilogue_to_act(tmem + t_lane + kWsColD0 + buf * kColD0Stride + net * 80, layer_n(0), bias, sm.act, row, nullptr);
                publish_act();
                if (tid == 0) {
                    if (last_net) mb_arrive(&sm.d0_empty[buf]);  // the layer-0 issuer may start tile i+2 into D0[buf]
                    issue_mma(0, layer_k(1) / 16, layer_n(1), false, layer_n(1), 0);
                }
                ph_w ^= 1u;
                LDBG(2);
                wait_acc();
                LDBG(3);
                if (tid == 0) load_w(net, weight_offset(2), weight_bytes(2));
                // ---- layer 1 epilogue -> A2 = [e(60), obs[:, 0:4]]
                epilogue_to_act(acc + t_lane, layer_n(1), bias + (bias_offset(1) - kBiasOffset) / 4, sm.act + kA2Plane * kWsPlane, row,
                                inject);
                publish_act();
                if (!kDual) {
                    if (tid == 0) issue_mma(0, layer_k(2) / 16, layer_n(2), false, layer_n(2), 0);
                    ph_w ^= 1u;
                    LDBG(4);
                    wait_acc();
                    LDBG(5);
                    if (tid == 0) load_w(net, weight_offset(3), kWsWBuf);  // W3, K planes 0..15
                    // ---- layer 2 epilogue -> A3 (256 columns); layer 3 in two K halves through the 40 KB weight buffer
                    epilogue_to_act(acc + t_lane, layer_n(2), bias + (bias_offset(2) - kBiasOffset) / 4, sm.act, row, nullptr);
                    publish_act();
                } else {
                    // ---- layer 2 as two N halves through the 192-column accumulator (W2 stays in the weight buffer)
                    constexpr int kHalf = layer_n(2) / 2;
                    if (tid == 0) issue_mma(kA2Plane, layer_k(2) / 16, kHalf, false, layer_n(2), 0);
                    ph_w ^= 1u;
                    wait_acc();
                    epilogue_to_act(acc + t_lane, kHalf, bias + (bias_offset(2) - kBiasOffset) / 4, sm.act, row, nullptr);
                    publish_act();
                    if (tid == 0) {  // (w_full completed its phase above: the second half must not wait on it again)
                        tc_fence_after();
                        const uint32_t idesc = make_idesc(kHalf);
                        for (int j = 0; j < layer_k(2) / 16; ++j)
                            umma(acc, make_desc(a0 + (kA2Plane + 2 * j) * kWsPlane, kWsPlane),
                                 make_desc(b0 + j * 2 * layer_n(2) * 16 + kHalf * 16, layer_n(2) * 16), idesc, j != 0);
                        umma_commit(&sm.acc_done);
                    }
                    wait_acc();
                    if (tid == 0) load_w(net, weight_offset(3), kWsWBuf);  // W3, K planes 0..15
                    epilogue_to_act(acc + t_lane, kHalf, bias + (bias_offset(2) - kBiasOffset) / 4 + kHalf,
                                    sm.act + (kHalf / 8) * kWsPlane, row, nullptr);
                    publish_act();
                }
                if (tid == 0) issue_mma(0, 8, layer_n(3), false, layer_n(3), 0);
                ph_w ^= 1u;
                LDBG(6);
                wait_acc();
                LDBG(7);
                if (tid == 0) {
                    load_w(net, weight_offset(3) + kWsWBuf, kWsWBuf);  // W3, K planes 16..31
                    issue_mma(16, 8, layer_n(3), true, layer_n(3), 0);
                }
                ph_w ^= 1u;
                wait_acc();
                LDBG(8);
                if (tid == 0) load_w(net, weight_offset(4), weight_bytes(4));
                // ---- layer 3 epilogue -> A4
                epilogue_to_act(acc + t_lane, layer_n(3), bias + (bias_offset(3) - kBiasOffset) / 4, sm.act, row, nullptr);
                publish_act();
                if (tid == 0) issue_mma(0, layer_k(4) / 16, layer_n(4), false, layer_n(4), 0);
                ph_w ^= 1u;
                LDBG(9);
                wait_acc();
                LDBG(10);
                if (tid == 0) load_w(net, weight_offset(5), weight_bytes(5));
                // ---- layer 4 epilogue -> A5
                epilogue_to_act(acc + t_lane, layer_n(4), bias + (bias_offset(4) - kBiasOffset) / 4, sm.act, row, nullptr);
                publish_act();
                if (tid == 0) issue_mma(0, layer_k(5) / 16, layer_n(5), false, layer_n(5), 0);
                ph_w ^= 1u;
                LDBG(11);
                wait_acc();
                LDBG(12);
                // the next W1: the other network's for this tile, or the first network's for the next tile
                if (tid == 0 && (!last_net || tile + (int)gridDim.x < n_tiles)) load_w(last_net ? 0 : net + 1, weight_offset(1), weight_bytes(1));
                // ---- last layer: mean = tanh(D5 + b5), two real columns; value = D5 + b5, one real column
                {
                    float v[8];
                    tmem_ld8(acc + t_lane, v);
                    const float* b5 = bias + (bias_offset(5) - kBiasOffset) / 4;
                    const bool linear = kDual ? net == 1 : value_head != 0;
                    float* dst = kDual && net == 1 ? value2 : mean;
                    if (live && linear) {
                        dst[grow] = v[0] + b5[0];  // DeterministicNeuralNetwork (models.py:151-162): linear output, no tanh
                    } else if (live) {
                        float2 m;
                        m.x = tanhf(v[0] + b5[0]);
                        m.y = tanhf(v[1] + b5[1]);
                        *reinterpret_cast<float2*>(dst + 2 * (size_t)grow) = m;
                        if (kSample) {  // GaussianMixin.act on the mean just computed (the policy is network 0)
                            const float2 e2 = normal2(s_key, sample.env_offset + (uint32_t)grow);
                            const float mm[2] = {m.x, m.y}, e[2] = {e2.x, e2.y};
                            const float ls[2] = {__ldg(sample.log_std), __ldg(sample.log_std + 1)};
                            float a[2];
                            const float lp = gaussian_sample(mm, ls, e, a);
                            *reinterpret_cast<float2*>(sample.actions + 2 * (size_t)grow) = make_float2(a[0], a[1]);
                            if (sample.log_prob != nullptr) sample.log_prob[grow] = lp;
                        }
                    }
                }
                LDBG(13);
                tc_fence_before();
                layer_group_sync();  // every TMEM read of this pass is done before the next layer-1 MMA overwrites acc
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
#if ROVER_POLICY_DBG
    if (threadIdx.x == 0 && blockIdx.x < 256) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        g_pol_cta[1][blockIdx.x] = t;
    }
#endif
}

typedef CUresult (*WsEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// obs: fp32 [N, obs_stride] (bf16_in == false) or bf16 [N, obs_stride] (bf16_in == true; strides in elements).
// packed2 != nullptr: policy (`packed` -> mean [N, 2]) and value network (`packed2` -> value2 [N]) in one pass over the
// observation (either dtype).
// sample != nullptr (policy head): the pass also samples the actions (kSample).
// enc_in: encoder width R (the callers check 1 <= R <= kEncInMax and obs_stride against it; blobs packed for R).
int launch_policy_forward_ws(const void* obs, int obs_stride, int n_envs, const void* packed, float* mean,
                             bool value_head, bool bf16_in, cudaStream_t stream, const void* packed2, float* value2,
                             const SampleArgs* sample, int enc_in) {
    static WsEncodeTiledFn encode = nullptr;
    static int n_sms = 0;
    constexpr int kSmemBytes = (int)sizeof(WsSmem) + 1024, kSmemBytesDual = (int)sizeof(WsSmemT<true>) + 1024;
    const bool dual = packed2 != nullptr;
    ROVER_CHECK(!(dual && (value2 == nullptr || value_head)), "policy + value pass: two outputs");
    ROVER_CHECK(!(sample && value_head), "sampling needs the policy head");
    if (!encode) {
        int dev = 0;
        ROVER_CUDA(cudaGetDevice(&dev));
        ROVER_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_ws_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_ws_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_ws_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kSmemBytesDual));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_ws_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kSmemBytes));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_ws_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kSmemBytes));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_ws_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kSmemBytesDual));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_ws_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kSmemBytesDual));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_ws_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        kSmemBytesDual));
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        ROVER_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
        ROVER_CHECK(fn && q == cudaDriverEntryPointSuccess, "rover_policy_forward: cuTensorMapEncodeTiled unavailable");
        encode = reinterpret_cast<WsEncodeTiledFn>(fn);
    }
    // rows per tile: fill whole rounds of the grid (see the kernel); multiple of 8 (core-matrix rows), at most 128
    const int rounds = (n_envs + kTileM * n_sms - 1) / (kTileM * n_sms);
    int tile_rows = (n_envs + rounds * n_sms - 1) / (rounds * n_sms);
    tile_rows = ((tile_rows + 7) / 8) * 8;
    if (tile_rows > kTileM) tile_rows = kTileM;
    alignas(64) CUtensorMap map;
    // fp32: columns [0, 4 + R), the converter zeroes what lies outside [3, 3 + R).  bf16: the tile is the MMA operand as
    // it lands, so the map ends at column 3 + R (the ray the reference's slicing drops is zero-filled; columns 0..2 are
    // finite and meet zero weights).  Beyond the map's end the tail chunk is zero-filled.
    const cuuint64_t gdim[2] = {(cuuint64_t)(kEncInOffset + enc_in + (bf16_in ? 0 : 1)), (cuuint64_t)n_envs};
    const cuuint64_t gstride[1] = {(cuuint64_t)obs_stride * (bf16_in ? 2ull : 4ull)};
    const cuuint32_t box[2] = {(cuuint32_t)(bf16_in ? kBfChunkK : kWsChunkK), (cuuint32_t)tile_rows};
    const cuuint32_t estr[2] = {1u, 1u};
    const CUresult rc = encode(&map, bf16_in ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                               const_cast<void*>(obs), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    ROVER_CHECK(rc == CUDA_SUCCESS, "rover_policy_forward: cuTensorMapEncodeTiled failed (%d)", (int)rc);
    const int n_tiles = (n_envs + tile_rows - 1) / tile_rows;
    const int grid = n_tiles < n_sms ? n_tiles : n_sms;
    const unsigned char* no_net = nullptr;
    float* no_out = nullptr;
    const SampleArgs sa = sample ? *sample : SampleArgs{nullptr, nullptr, 0u, nullptr, nullptr};
    // kernel<kBf16In, kDual, kSample>: one launch of the instantiation the arguments select
    auto launch = [&](auto kernel, int threads, int smem) {
        return launch_overlapped(kernel, dim3(grid), dim3(threads), (size_t)smem, stream, map, static_cast<const float*>(obs),
                                 obs_stride, n_envs, tile_rows, static_cast<const unsigned char*>(packed), mean,
                                 value_head ? 1 : 0, dual ? static_cast<const unsigned char*>(packed2) : no_net,
                                 dual ? value2 : no_out, sa, enc_in);
    };
    if (dual && bf16_in && sample) ROVER_CUDA(launch(policy_forward_ws_kernel<true, true, true>, kWsThreads, kSmemBytesDual));
    else if (dual && bf16_in) ROVER_CUDA(launch(policy_forward_ws_kernel<true, true>, kWsThreads, kSmemBytesDual));
    else if (dual && sample) ROVER_CUDA(launch(policy_forward_ws_kernel<false, true, true>, kWsThreadsF32, kSmemBytesDual));
    else if (dual) ROVER_CUDA(launch(policy_forward_ws_kernel<false, true>, kWsThreadsF32, kSmemBytesDual));
    else if (bf16_in && sample) ROVER_CUDA(launch(policy_forward_ws_kernel<true, false, true>, kWsThreads, kSmemBytes));
    else if (bf16_in) ROVER_CUDA(launch(policy_forward_ws_kernel<true>, kWsThreads, kSmemBytes));
    else if (sample) ROVER_CUDA(launch(policy_forward_ws_kernel<false, false, true>, kWsThreadsF32, kSmemBytes));
    else ROVER_CUDA(launch(policy_forward_ws_kernel<false>, kWsThreadsF32, kSmemBytes));
    return check_launch(sample ? "policy_forward_ws_kernel (sampling)" : "policy_forward_ws_kernel");
}

}  // namespace rover

#if ROVER_POLICY_DBG
extern "C" int rover_debug_policy_timeline(long long* host_dst) {
    return (int)cudaMemcpyFromSymbol(host_dst, rover::g_pol_dbg, sizeof(rover::g_pol_dbg));
}
extern "C" int rover_debug_policy_ctas(unsigned long long* host_dst) {
    return (int)cudaMemcpyFromSymbol(host_dst, rover::g_pol_cta, sizeof(rover::g_pol_cta));
}
#endif
