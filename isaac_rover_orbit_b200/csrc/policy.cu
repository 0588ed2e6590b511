// Gaussian policy forward on the 5th-generation tensor cores (tcgen05 + TMEM), bf16 operands, fp32 accumulation.
//
// Replaces GaussianNeuralNetwork.compute + HeightmapEncoder of the reference
// (rover_envs/envs/navigation/learning/skrl/models.py:24-36, 89-102; built by gaussian_model_skrl,
// configure_models.py:37-53):
//     x = s[:, 0:4];  e = LReLU(W1 LReLU(W0 s[:, 3:964] + b0) + b1)        (961 -> 80 -> 60; heading column included,
//     y = tanh(W5 LReLU(W4 LReLU(W3 LReLU(W2 [x, e] + b2) + b3) + b4) + b5)  last ray dropped -- reference quirk kept)
// and skrl's GaussianMixin.act sampling (rover_gaussian_act).  319,520 FLOP per environment.
//
// One persistent CTA per SM, 256 threads, tile = 128 environments (UMMA M = 128, cta_group::1):
//   layer 0  K = observation column (16-byte aligned TMA box origins; columns outside [3, 964) are zeroed and carry
//            zero weights), streamed in 16 chunks of 64 columns: a 2-D TMA tensor-map load (fp32, 128 x 64)
//            + a bulk copy of the matching 80 x 64 bf16 weight chunk land on one mbarrier; all threads convert the
//            chunk to bf16 in the UMMA K-major no-swizzle ("interleaved") layout; one thread issues the
//            tcgen05.mma's (D0[128 x 80] in TMEM) and commits to the stage's mbarrier; two stages overlap
//            TMA / convert / MMA.
//   layers 1-5  the epilogue of layer l (tcgen05.ld -> +bias -> LeakyReLU -> bf16) writes the A operand of layer
//            l+1 straight into shared memory; weights arrive by bulk copy from the pre-packed blob; accumulators
//            alternate between two TMEM regions.  The last epilogue applies tanh and stores mean[128, 2].
// Operand layout (SWIZZLE_NONE, K-major): 8 x 8 bf16 core matrices; element (row r, k) lives at
//     (k / 8) * plane_stride + r * 16 + (k % 8) * 2,   descriptor LBO = plane_stride, SBO = 128 B.
#include "policy_common.cuh"

namespace rover {

// ---------------------------------------------------------------------------------------------------- shared memory
struct __align__(128) PolSmem {
    union {
        struct {  // layer 0 streaming
            float stage_f32[kStagesF][kTileM * kChunkK];       // 4 x 32 KB, TMA destinations (3 chunks in flight)
            unsigned char a_bf16[2][8 * kAPlane];              // 2 x 16.1 KB
            unsigned char w0[kStagesW][kW0ChunkBytes];         // 3 x 10 KB
        } l0;
        struct {  // layers 1..5
            unsigned char act[2][32 * kAPlane];                // up to K = 256 -> 32 planes, 2 x 64.5 KB
            unsigned char w[(256 / 8) * 160 * 16];             // largest weight image (layer 3): 80 KB
        } ln;
    };
    unsigned long long full[kStagesF];   // observation chunk landed in stage_f32[s]
    unsigned long long w0_full[kStagesW];  // weight chunk landed in w0[s]
    unsigned long long mma_done;     // the MMAs of the previous layer-0 chunk retired
    float bias[80 + 64 + 256 + 160 + 128 + 16];  // all layer biases (padded), loaded once per CTA
    unsigned long long w_full;       // weights of the current layer (l >= 1) landed
    unsigned long long acc_done;     // accumulator of the current layer complete
    uint32_t tmem_base;
};

// ---------------------------------------------------------------------------------------------------- kernel
__global__ void __launch_bounds__(kPolThreads, 1)
policy_forward_kernel(const __grid_constant__ CUtensorMap obs_map, const float* __restrict__ obs, int obs_stride,
                      int n_envs, const unsigned char* __restrict__ packed, float* __restrict__ mean, int debug_stop,
                      int value_head) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PolSmem& sm = *reinterpret_cast<PolSmem*>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n_tiles = (n_envs + kTileM - 1) / kTileM;

    if (tid == 0) {
        for (int i = 0; i < kStagesF; ++i) mb_init(&sm.full[i], 1);
        for (int i = 0; i < kStagesW; ++i) mb_init(&sm.w0_full[i], 1);
        mb_init(&sm.mma_done, 1);
        mb_init(&sm.w_full, 1);
        mb_init(&sm.acc_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < (kPackedBytes - kBiasOffset) / 4; i += kPolThreads)
        sm.bias[i] = __ldg(reinterpret_cast<const float*>(packed + kBiasOffset) + i);
    if (warp == 0) {  // one warp allocates all 512 TMEM columns (one CTA per SM)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sptr(&sm.tmem_base)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = sm.tmem_base;
    if (debug_stop == 1) {  // bring-up aid (ROVER_POLICY_DEBUG_STOP): TMEM alloc / dealloc only
        __syncthreads();
        if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
        return;
    }

    if (debug_stop >= 4 && debug_stop <= 6) {  // bring-up aid: isolate the async copies
        if (tid == 0) {
            const uint32_t bytes = (debug_stop == 4 ? kTileM * kChunkK * 4 : 0) + (debug_stop == 5 ? kW0ChunkBytes : 0) +
                                   (debug_stop == 6 ? kTileM * kChunkK * 4 + kW0ChunkBytes : 0);
            mb_expect_tx(&sm.full[0], bytes);
            if (debug_stop != 5) tma_2d(sm.l0.stage_f32[0], &obs_map, 0, 0, &sm.full[0]);
            if (debug_stop != 4) bulk_g2s(sm.l0.w0[0], packed, kW0ChunkBytes, &sm.full[0]);
        }
        mb_wait(&sm.full[0], 0);
        if (tid < 2 && blockIdx.x == 0) mean[tid] = debug_stop == 5 ? (float)sm.l0.w0[0][tid] : sm.l0.stage_f32[0][tid];
        __syncthreads();
        if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
        return;
    }

    // barrier phase bookkeeping (each barrier completes once per use; parity flips per completion)
    uint32_t ph_full = 0, ph_w0 = 0, ph_mma = 0, ph_w = 0, ph_acc = 0;  // bit s = parity of stage s

    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int row0 = tile * kTileM;
        // =========================================================== layer 0: stream K in 16 chunks of 64 columns
        const uint32_t idesc0 = make_idesc(layer_n(0));
        if (tid == 0) {  // prologue: observation chunks 0..2 and weight chunks 0..1 in flight
            for (int c = 0; c < kStagesF - 1; ++c) {
                mb_expect_tx(&sm.full[c], kTileM * kChunkK * 4);
                tma_2d(sm.l0.stage_f32[c], &obs_map, c * kChunkK, row0, &sm.full[c]);
            }
            for (int c = 0; c < kStagesW - 1; ++c) {
                mb_expect_tx(&sm.w0_full[c], kW0ChunkBytes);
                bulk_g2s(sm.l0.w0[c], packed + (size_t)c * kW0ChunkBytes, kW0ChunkBytes, &sm.w0_full[c]);
            }
        }
        for (int c = 0; c < kNumChunks; ++c) {
            const int sf = c % kStagesF, sw = c % kStagesW, sa = c & 1;
            if (tid == 0) {
                if (c >= 1) {  // MMAs of chunk c-1 (and all earlier ones) retired: a_bf16[sa^1] and w0[(c-1)%3] are free
                    mb_wait(&sm.mma_done, ph_mma & 1u);
                    ph_mma ^= 1u;
                }
                if (c + kStagesF - 1 < kNumChunks) {  // stage of chunk c-1: its conversion ended before the last sync
                    const int cn = c + kStagesF - 1, sn = cn % kStagesF;
                    mb_expect_tx(&sm.full[sn], kTileM * kChunkK * 4);
                    tma_2d(sm.l0.stage_f32[sn], &obs_map, cn * kChunkK, row0, &sm.full[sn]);
                }
                if (c + kStagesW - 1 < kNumChunks) {
                    const int cn = c + kStagesW - 1, sn = cn % kStagesW;
                    mb_expect_tx(&sm.w0_full[sn], kW0ChunkBytes);
                    bulk_g2s(sm.l0.w0[sn], packed + (size_t)cn * kW0ChunkBytes, kW0ChunkBytes, &sm.w0_full[sn]);
                }
            }
            mb_wait(&sm.full[sf], (ph_full >> sf) & 1u);
            ph_full ^= 1u << sf;
            // a_bf16[sa] was last read by the MMAs of chunk c-2: thread 0 waited for them one iteration ago, before
            // that iteration's __syncthreads, which orders every thread's stores below after that wait.
            // ---- convert fp32 [128][64] -> bf16 planes [8][128 rows][8]
            const float* __restrict__ src = sm.l0.stage_f32[sf];
            unsigned char* dst = sm.l0.a_bf16[sa];
#pragma unroll
            for (int i = 0; i < (kTileM * 8) / kPolThreads; ++i) {
                const int p = tid + i * kPolThreads;
                const int plane = p & 7, row = p >> 3;
                const float4 lo = *reinterpret_cast<const float4*>(src + row * kChunkK + plane * 8);
                const float4 hi = *reinterpret_cast<const float4*>(src + row * kChunkK + plane * 8 + 4);
                float v[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
                if (c == 0 || c == kNumChunks - 1) {  // encoder input = observation columns [3, 964) (models.py:95)
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int col = c * kChunkK + plane * 8 + j;
                        if (col < kEncInOffset || col >= kEncInOffset + kEncIn) v[j] = 0.f;
                    }
                }
                uint4 o;
                o.x = pack_bf16(v[0], v[1]);
                o.y = pack_bf16(v[2], v[3]);
                o.z = pack_bf16(v[4], v[5]);
                o.w = pack_bf16(v[6], v[7]);
                *reinterpret_cast<uint4*>(dst + plane * kAPlane + row * 16) = o;
            }
            fence_async_smem();
            __syncthreads();
            if (tid == 0 && debug_stop != 2) {
                tc_fence_after();
                mb_wait(&sm.w0_full[sw], (ph_w0 >> sw) & 1u);
                ph_w0 ^= 1u << sw;
                const uint32_t a0 = sptr(sm.l0.a_bf16[sa]), b0 = sptr(sm.l0.w0[sw]);
#pragma unroll
                for (int j = 0; j < kChunkK / 16; ++j)
                    umma(tmem + 0, make_desc(a0 + j * 2 * kAPlane, kAPlane), make_desc(b0 + j * 2 * 80 * 16, 80 * 16),
                         idesc0, (c | j) != 0);
                umma_commit(&sm.mma_done);
            } else if (tid == 0) {  // bring-up stop 2: no MMAs; keep the barrier protocol balanced
                mb_wait(&sm.w0_full[sw], (ph_w0 >> sw) & 1u);
                ph_w0 ^= 1u << sw;
                asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(sptr(&sm.mma_done)) : "memory");
            }
        }
        if (tid == 0) {  // drain the last chunk's MMAs, then start the bulk copy of W1 into the layer region
            mb_wait(&sm.mma_done, ph_mma & 1u);
            ph_mma ^= 1u;
            mb_expect_tx(&sm.w_full, weight_bytes(1));
            bulk_g2s(sm.ln.w, packed + weight_offset(1), weight_bytes(1), &sm.w_full);
        }
        __syncthreads();  // everyone may now read D0 from TMEM and overwrite the layer-0 shared buffers
        tc_fence_after();
        if (debug_stop == 2 || debug_stop == 3) {  // bring-up aid: stop after the layer-0 stream
            if (tid == 0) mb_wait(&sm.w_full, ph_w);
            __syncthreads();
            break;
        }

        // =========================================================== layers: epilogue of l feeds layer l+1
#pragma unroll 1
        for (int l = 0; l < kNumLayers; ++l) {
            const int n_pad = layer_n(l);
            const uint32_t d_col = (l & 1) ? 256u : 0u;  // accumulator region of layer l
            const float* bias = sm.bias + (bias_offset(l) - kBiasOffset) / 4;
            const int row = (warp & 3) * 32 + lane;       // TMEM lane == tile row
            const int half = warp >> 2;                   // column half handled by this warp
            const int cols_per_half = n_pad / 2;
            const uint32_t t_lane = (uint32_t)((warp & 3) * 32) << 16;
            unsigned char* act_out = sm.ln.act[l & 1];    // A operand of layer l+1
            if (l < kNumLayers - 1) {
                // all TMEM loads of this thread's columns are issued back to back (one wait per 40 columns at most)
                for (int nb = half * cols_per_half; nb < (half + 1) * cols_per_half; nb += 40) {
                    const int ngroups = min(5, ((half + 1) * cols_per_half - nb) / 8);
                    uint32_t raw[5][8];
#pragma unroll
                    for (int q = 0; q < 5; ++q)
                        if (q < ngroups) tmem_ld8_nowait(tmem + t_lane + d_col + nb + q * 8, raw[q]);
                    tmem_wait_ld();
#pragma unroll
                    for (int q = 0; q < 5; ++q) {
                        if (q >= ngroups) continue;
                        const int n0 = nb + q * 8;
                        float v[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) v[j] = leaky(__uint_as_float(raw[q][j]) + bias[n0 + j]);
                        if (l == 1 && n0 == 56) {
                            // layer 2 consumes [e(60), obs[:,0:4]] (W2's columns are permuted accordingly at pack time)
                            const int grow = row0 + row;
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                v[4 + j] = grow < n_envs ? __ldg(obs + (size_t)grow * obs_stride + j) : 0.f;
                        }
                        uint4 o;
                        o.x = pack_bf16(v[0], v[1]);
                        o.y = pack_bf16(v[2], v[3]);
                        o.z = pack_bf16(v[4], v[5]);
                        o.w = pack_bf16(v[6], v[7]);
                        *reinterpret_cast<uint4*>(act_out + (n0 >> 3) * kAPlane + row * 16) = o;
                    }
                }
                tc_fence_before();
                fence_async_smem();
                __syncthreads();
                // ---- layer l+1: D = act_out x W^T
                if (tid == 0) {
                    tc_fence_after();
                    mb_wait(&sm.w_full, ph_w);
                    const int ln = l + 1, k_pad = layer_k(ln), nn = layer_n(ln);
                    const uint32_t idesc = make_idesc(nn), a0 = sptr(act_out), b0 = sptr(sm.ln.w);
                    const uint32_t dn = (ln & 1) ? 256u : 0u;
                    for (int j = 0; j < k_pad / 16; ++j)
                        umma(tmem + dn, make_desc(a0 + j * 2 * kAPlane, kAPlane), make_desc(b0 + j * 2 * nn * 16, nn * 16),
                             idesc, j != 0);
                    umma_commit(&sm.acc_done);
                    mb_wait(&sm.acc_done, ph_acc);  // accumulator complete, weight buffer free
                    if (ln + 1 < kNumLayers) {      // prefetch the next layer's weights during this layer's epilogue
                        mb_expect_tx(&sm.w_full, weight_bytes(ln + 1));
                        bulk_g2s(sm.ln.w, packed + weight_offset(ln + 1), weight_bytes(ln + 1), &sm.w_full);
                    }
                }
                ph_w ^= 1;
                ph_acc ^= 1;
                __syncthreads();
                tc_fence_after();
            } else {
                // ---- last layer: mean = tanh(D5 + b5), two real columns
                if (half == 0) {
                    float v[8];
                    tmem_ld8(tmem + t_lane + d_col, v);
                    const int grow = row0 + row;
                    if (grow < n_envs && value_head) {
                        mean[grow] = v[0] + bias[0];  // DeterministicNeuralNetwork: one linear output, no tanh
                    } else if (grow < n_envs) {
                        float2 m;
                        m.x = tanhf(v[0] + bias[0]);
                        m.y = tanhf(v[1] + bias[1]);
                        *reinterpret_cast<float2*>(mean + 2 * (size_t)grow) = m;
                    }
                }
                tc_fence_before();
                __syncthreads();  // TMEM reads finished before the next tile's MMAs overwrite the accumulators
                tc_fence_after();
            }
        }
    }

    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------- packing
struct PackArgs {
    const float* w[6];
    const float* b[6];
    int in_dim[6], out_dim[6];
};

__global__ void policy_pack_kernel(const __grid_constant__ PackArgs a, unsigned char* __restrict__ packed) {
    const int l = blockIdx.y;
    const int k_pad = layer_k(l), n_pad = layer_n(l), k_real = layer_k_real(l), n_real = a.out_dim[l];
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(packed + weight_offset(l));
    const int total = (l == 0 ? kNumChunks * kChunkK : k_pad) * n_pad;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        // idx enumerates (plane-major) the packed image: [chunk][plane][n][8] for layer 0, [plane][n][8] otherwise
        const int j = idx & 7;
        const int n = (idx >> 3) % n_pad;
        const int plane_g = (idx >> 3) / n_pad;  // global plane index = k / 8 (layer 0: chunk * 8 + plane)
        const int k = plane_g * 8 + j;
        float v = 0.f;
        int src_k = k;
        if (l == 0) src_k = k - kEncInOffset;               // layer-0 K index = observation column
        if (l == 2) src_k = (k < 60) ? k + 4 : k - 60;      // operand order [e(60), obs[:,0:4]] -> reference [x(4), e(60)]
        if (n < n_real && src_k >= 0 && src_k < k_real) v = a.w[l][(size_t)n * a.in_dim[l] + src_k];
        dst[idx] = __float2bfloat16_rn(v);
    }
    float* bdst = reinterpret_cast<float*>(packed + bias_offset(l));
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < n_pad; n += gridDim.x * blockDim.x)
        bdst[n] = n < n_real ? a.b[l][n] : 0.f;
}

__global__ void gaussian_act_kernel(const float* __restrict__ mean, const float* __restrict__ log_std,
                                    const float* __restrict__ eps, int n, float* __restrict__ actions,
                                    float* __restrict__ log_prob) {
    grid_dependency_wait();  // launched as a programmatic dependent of the forward pass (common.cuh)
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float m[2] = {mean[2 * i], mean[2 * i + 1]};
    const float ls[2] = {__ldg(log_std), __ldg(log_std + 1)};
    const float e[2] = {eps[2 * i], eps[2 * i + 1]};
    float a[2];
    const float lp = gaussian_sample(m, ls, e, a);
    actions[2 * i] = a[0];
    actions[2 * i + 1] = a[1];
    if (log_prob) log_prob[i] = lp;
}

// eps [N, 2] that the next sampling launch with this {seed, step} draws (rover_action_noise); advance: take the step
__global__ void action_noise_kernel(unsigned long long* __restrict__ rng, uint32_t env_offset, int n, float* __restrict__ eps,
                                    int advance) {
    __shared__ RngKey key;
    grid_dependency_wait();
    if (threadIdx.x == 0) key = take_step(rng, gridDim.x, advance != 0);
    __syncthreads();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        *reinterpret_cast<float2*>(eps + 2 * (size_t)i) = normal2(key, env_offset + (uint32_t)i);
}

// The sampling's functions that are not correctly rounded (logf, expf, sincospif), evaluated elementwise by the device
// code the policy kernels run (this library's flags and libdevice): an fp32 model of the sampling takes them from here.
__global__ void policy_math_kernel(int op, const float* __restrict__ a, float* __restrict__ out0, float* __restrict__ out1,
                                   int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = a[i];
    if (op == ROVER_POLICY_MATH_LOG) {
        out0[i] = logf(x);
    } else if (op == ROVER_POLICY_MATH_EXP) {
        out0[i] = expf(x);
    } else {
        float s, c;
        sincospif(x, &s, &c);
        out0[i] = s;
        out1[i] = c;
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int launch_policy_forward_ws(const void* obs, int obs_stride, int n_envs, const void* packed, float* out,
                             bool value_head, bool bf16_in, cudaStream_t stream, const void* packed2 = nullptr,
                             float* value2 = nullptr, const SampleArgs* sample = nullptr);  // policy_ws.cu

}  // namespace rover

extern "C" int64_t rover_policy_pack(const RoverPolicyWeights* weights, void* packed, void* stream) {
    using namespace rover;
    if (packed == nullptr) return kPackedBytes;
    if (weights == nullptr) {
        fail("rover_policy_pack: weights is NULL");
        return -1;
    }
    PackArgs a;
    for (int l = 0; l < 6; ++l) {
        const bool out_ok = weights->out_dim[l] == layer_n_real(l) || (l == 5 && weights->out_dim[l] == 1);  // value head
        if (!weights->w[l] || !weights->b[l] || weights->in_dim[l] < layer_k_real(l) || !out_ok) {
            fail("rover_policy_pack: layer %d has shape [%d,%d], expected [%d,%d]", l, weights->out_dim[l],
                 weights->in_dim[l], layer_n_real(l), layer_k_real(l));
            return -1;
        }
        a.w[l] = weights->w[l];
        a.b[l] = weights->b[l];
        a.in_dim[l] = weights->in_dim[l];
        a.out_dim[l] = weights->out_dim[l];
    }
    policy_pack_kernel<<<dim3(64, 6), 256, 0, static_cast<cudaStream_t>(stream)>>>(a, static_cast<unsigned char*>(packed));
    return check_launch("policy_pack_kernel") ? -1 : kPackedBytes;
}

static int policy_or_value_forward(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed, float* mean,
                                   void* stream, bool value_head) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_policy_forward: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs && packed && mean, "rover_policy_forward: NULL argument");
    ROVER_CHECK(obs_stride >= kObsCols && obs_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(obs) & 15) == 0,
                "rover_policy_forward: obs rows must be 16-byte aligned (obs_stride %% 4 == 0, got %d); allocate the "
                "observation buffer with ops.alloc_obs()", obs_stride);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(packed) & 127) == 0, "rover_policy_forward: packed blob not 128B aligned");
    {   // default: the warp-specialised kernel (policy_ws.cu); ROVER_POLICY_KERNEL=v1 selects the tile-serial one
        const char* which = getenv("ROVER_POLICY_KERNEL");
        if (which == nullptr || which[0] != 'v' || which[1] != '1')
            return launch_policy_forward_ws(obs, obs_stride, n_envs, packed, mean, value_head, false,
                                            static_cast<cudaStream_t>(stream));
    }
    static EncodeTiledFn encode = nullptr;
    static int n_sms = 0;
    if (!encode) {
        int dev = 0;
        ROVER_CUDA(cudaGetDevice(&dev));
        ROVER_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
        ROVER_CUDA(cudaFuncSetAttribute(policy_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)sizeof(PolSmem)));
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        ROVER_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
        ROVER_CHECK(fn && q == cudaDriverEntryPointSuccess, "rover_policy_forward: cuTensorMapEncodeTiled unavailable");
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    alignas(64) CUtensorMap map;
    const cuuint64_t gdim[2] = {(cuuint64_t)kObsCols, (cuuint64_t)n_envs};
    const cuuint64_t gstride[1] = {(cuuint64_t)obs_stride * 4ull};
    const cuuint32_t box[2] = {(cuuint32_t)kChunkK, (cuuint32_t)kTileM};
    const cuuint32_t estr[2] = {1u, 1u};
    const CUresult rc = encode(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(obs), gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    ROVER_CHECK(rc == CUDA_SUCCESS, "rover_policy_forward: cuTensorMapEncodeTiled failed (%d)", (int)rc);
    const int n_tiles = (n_envs + kTileM - 1) / kTileM;
    const int grid = n_tiles < n_sms ? n_tiles : n_sms;
    const char* dbg = getenv("ROVER_POLICY_DEBUG_STOP");
    policy_forward_kernel<<<grid, kPolThreads, sizeof(PolSmem), static_cast<cudaStream_t>(stream)>>>(
        map, obs, obs_stride, n_envs, static_cast<const unsigned char*>(packed), mean, dbg ? atoi(dbg) : 0,
        value_head ? 1 : 0);
    return check_launch("policy_forward_kernel");
}

extern "C" int rover_policy_forward(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed,
                                    float* mean, void* stream) {
    return policy_or_value_forward(obs, obs_stride, n_envs, packed, mean, stream, false);
}

extern "C" int rover_policy_value_forward(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed_policy,
                                          const void* packed_value, float* mean, float* value, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_policy_value_forward: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs && packed_policy && packed_value && mean && value, "rover_policy_value_forward: NULL argument");
    ROVER_CHECK(obs_stride >= kObsCols && obs_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(obs) & 15) == 0,
                "rover_policy_value_forward: obs rows must be 16-byte aligned (obs_stride %% 4 == 0, got %d); allocate the "
                "observation buffer with ops.alloc_obs()", obs_stride);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(packed_policy) & 127) == 0 && (reinterpret_cast<uintptr_t>(packed_value) & 127) == 0,
                "rover_policy_value_forward: packed blob not 128B aligned");
    return launch_policy_forward_ws(obs, obs_stride, n_envs, packed_policy, mean, false, false, static_cast<cudaStream_t>(stream),
                                    packed_value, value);
}

static int forward_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed, float* out,
                        void* stream, bool value_head) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_*_forward_bf16: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs_bf16 && packed && out, "rover_*_forward_bf16: NULL argument");
    ROVER_CHECK(stride >= kObsCols && stride % 8 == 0 && (reinterpret_cast<uintptr_t>(obs_bf16) & 15) == 0,
                "rover_*_forward_bf16: bf16 observation rows must be 16-byte aligned (stride %% 8 == 0, got %d)", stride);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(packed) & 127) == 0, "rover_*_forward_bf16: packed blob not 128B aligned");
    return launch_policy_forward_ws(obs_bf16, stride, n_envs, packed, out, value_head, true, static_cast<cudaStream_t>(stream));
}

extern "C" int rover_policy_forward_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed,
                                         float* mean, void* stream) {
    return forward_bf16(obs_bf16, stride, n_envs, packed, mean, stream, false);
}

extern "C" int rover_value_forward_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed,
                                        float* value, void* stream) {
    return forward_bf16(obs_bf16, stride, n_envs, packed, value, stream, true);
}

extern "C" int rover_policy_value_forward_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs,
                                               const void* packed_policy, const void* packed_value, float* mean, float* value,
                                               void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_policy_value_forward_bf16: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs_bf16 && packed_policy && packed_value && mean && value, "rover_policy_value_forward_bf16: NULL argument");
    ROVER_CHECK(stride >= kObsCols && stride % 8 == 0 && (reinterpret_cast<uintptr_t>(obs_bf16) & 15) == 0,
                "rover_policy_value_forward_bf16: bf16 observation rows must be 16-byte aligned (stride %% 8 == 0, got %d)",
                stride);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(packed_policy) & 127) == 0 && (reinterpret_cast<uintptr_t>(packed_value) & 127) == 0,
                "rover_policy_value_forward_bf16: packed blob not 128B aligned");
    return launch_policy_forward_ws(obs_bf16, stride, n_envs, packed_policy, mean, false, true, static_cast<cudaStream_t>(stream),
                                    packed_value, value);
}

extern "C" int rover_value_forward(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed,
                                   float* value, void* stream) {
    return policy_or_value_forward(obs, obs_stride, n_envs, packed, value, stream, true);
}

extern "C" int rover_gaussian_act(const float* mean, const float* log_std, const float* eps, int32_t n_envs,
                                  float* actions, float* log_prob, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_gaussian_act: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(mean && log_std && eps && actions, "rover_gaussian_act: NULL argument");
    ROVER_CUDA(launch_overlapped(gaussian_act_kernel, dim3((n_envs + 255) / 256), dim3(256), 0, static_cast<cudaStream_t>(stream),
                                 mean, log_std, eps, (int)n_envs, actions, log_prob));
    return check_launch("gaussian_act_kernel");
}

// ---------------------------------------------------------------------------------------------------- sampling in the pass
static int check_act_args(const char* who, int32_t n_envs, const void* packed, const float* log_std, const int64_t* rng_state,
                          int32_t env_offset, const float* mean, const float* actions) {
    using namespace rover;
    ROVER_CHECK(packed && log_std && rng_state && mean && actions, "%s: NULL argument", who);
    ROVER_CHECK(env_offset >= 0, "%s: env_offset must be >= 0 (got %d)", who, env_offset);
    ROVER_CHECK((uint64_t)env_offset + (uint64_t)n_envs <= (1ull << 32), "%s: env_offset + n_envs exceeds 2^32", who);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(packed) & 127) == 0, "%s: packed blob not 128B aligned", who);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(rng_state) & 7) == 0 && (reinterpret_cast<uintptr_t>(log_std) & 3) == 0,
                "%s: rng_state must be 8-byte and log_std 4-byte aligned", who);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(mean) & 7) == 0 && (reinterpret_cast<uintptr_t>(actions) & 7) == 0,
                "%s: mean and actions must be 8-byte aligned [N, 2] arrays", who);
    return 0;
}

extern "C" int rover_policy_act(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed, const float* log_std,
                                int64_t* rng_state, int32_t env_offset, float* mean, float* actions, float* log_prob,
                                void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_policy_act: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs != nullptr, "rover_policy_act: NULL argument");
    if (int rc = check_act_args("rover_policy_act", n_envs, packed, log_std, rng_state, env_offset, mean, actions)) return rc;
    ROVER_CHECK(obs_stride >= kObsCols && obs_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(obs) & 15) == 0,
                "rover_policy_act: obs rows must be 16-byte aligned (obs_stride %% 4 == 0, got %d); allocate the "
                "observation buffer with ops.alloc_obs()", obs_stride);
    const SampleArgs s{log_std, reinterpret_cast<unsigned long long*>(rng_state), (uint32_t)env_offset, actions, log_prob};
    return launch_policy_forward_ws(obs, obs_stride, n_envs, packed, mean, false, false, static_cast<cudaStream_t>(stream),
                                    nullptr, nullptr, &s);
}

extern "C" int rover_policy_act_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed,
                                     const float* log_std, int64_t* rng_state, int32_t env_offset, float* mean, float* actions,
                                     float* log_prob, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_policy_act_bf16: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs_bf16 != nullptr, "rover_policy_act_bf16: NULL argument");
    if (int rc = check_act_args("rover_policy_act_bf16", n_envs, packed, log_std, rng_state, env_offset, mean, actions)) return rc;
    ROVER_CHECK(stride >= kObsCols && stride % 8 == 0 && (reinterpret_cast<uintptr_t>(obs_bf16) & 15) == 0,
                "rover_policy_act_bf16: bf16 observation rows must be 16-byte aligned (stride %% 8 == 0, got %d)", stride);
    const SampleArgs s{log_std, reinterpret_cast<unsigned long long*>(rng_state), (uint32_t)env_offset, actions, log_prob};
    return launch_policy_forward_ws(obs_bf16, stride, n_envs, packed, mean, false, true, static_cast<cudaStream_t>(stream),
                                    nullptr, nullptr, &s);
}

extern "C" int rover_policy_value_act(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed_policy,
                                      const void* packed_value, const float* log_std, int64_t* rng_state, int32_t env_offset,
                                      float* mean, float* value, float* actions, float* log_prob, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_policy_value_act: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs && packed_value && value, "rover_policy_value_act: NULL argument");
    if (int rc = check_act_args("rover_policy_value_act", n_envs, packed_policy, log_std, rng_state, env_offset, mean, actions))
        return rc;
    ROVER_CHECK(obs_stride >= kObsCols && obs_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(obs) & 15) == 0,
                "rover_policy_value_act: obs rows must be 16-byte aligned (obs_stride %% 4 == 0, got %d); allocate the "
                "observation buffer with ops.alloc_obs()", obs_stride);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(packed_value) & 127) == 0, "rover_policy_value_act: packed blob not 128B aligned");
    const SampleArgs s{log_std, reinterpret_cast<unsigned long long*>(rng_state), (uint32_t)env_offset, actions, log_prob};
    return launch_policy_forward_ws(obs, obs_stride, n_envs, packed_policy, mean, false, false, static_cast<cudaStream_t>(stream),
                                    packed_value, value, &s);
}

extern "C" int rover_policy_value_act_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed_policy,
                                           const void* packed_value, const float* log_std, int64_t* rng_state,
                                           int32_t env_offset, float* mean, float* value, float* actions, float* log_prob,
                                           void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_policy_value_act_bf16: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(obs_bf16 && packed_value && value, "rover_policy_value_act_bf16: NULL argument");
    if (int rc = check_act_args("rover_policy_value_act_bf16", n_envs, packed_policy, log_std, rng_state, env_offset, mean,
                                actions))
        return rc;
    ROVER_CHECK(stride >= kObsCols && stride % 8 == 0 && (reinterpret_cast<uintptr_t>(obs_bf16) & 15) == 0,
                "rover_policy_value_act_bf16: bf16 observation rows must be 16-byte aligned (stride %% 8 == 0, got %d)", stride);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(packed_value) & 127) == 0, "rover_policy_value_act_bf16: packed blob not 128B aligned");
    const SampleArgs s{log_std, reinterpret_cast<unsigned long long*>(rng_state), (uint32_t)env_offset, actions, log_prob};
    return launch_policy_forward_ws(obs_bf16, stride, n_envs, packed_policy, mean, false, true, static_cast<cudaStream_t>(stream),
                                    packed_value, value, &s);
}

extern "C" int rover_action_noise(int64_t* rng_state, int32_t env_offset, int32_t n_envs, float* eps_out, int32_t advance,
                                  void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_action_noise: negative n_envs");
    ROVER_CHECK(env_offset >= 0, "rover_action_noise: env_offset must be >= 0 (got %d)", env_offset);
    ROVER_CHECK(rng_state && (eps_out || n_envs == 0), "rover_action_noise: NULL argument");
    ROVER_CHECK((reinterpret_cast<uintptr_t>(rng_state) & 7) == 0 && (reinterpret_cast<uintptr_t>(eps_out) & 7) == 0,
                "rover_action_noise: rng_state and eps_out must be 8-byte aligned");
    int blocks = (n_envs + 255) / 256;
    if (blocks > 1024) blocks = 1024;
    if (blocks == 0) {
        if (!advance) return 0;
        blocks = 1;  // nothing to draw, but the step still advances
    }
    ROVER_CUDA(launch_overlapped(action_noise_kernel, dim3(blocks), dim3(256), 0, static_cast<cudaStream_t>(stream),
                                 reinterpret_cast<unsigned long long*>(rng_state), (uint32_t)env_offset, (int)n_envs, eps_out,
                                 (int)(advance != 0)));
    return check_launch("action_noise_kernel");
}

extern "C" int rover_policy_math(int32_t op, const float* a, float* out0, float* out1, int32_t n, void* stream) {
    using namespace rover;
    ROVER_CHECK(op == ROVER_POLICY_MATH_LOG || op == ROVER_POLICY_MATH_EXP || op == ROVER_POLICY_MATH_SINCOSPI,
                "rover_policy_math: op must be ROVER_POLICY_MATH_LOG, _EXP or _SINCOSPI");
    ROVER_CHECK(n >= 0, "rover_policy_math: negative n");
    if (n == 0) return 0;
    ROVER_CHECK(a && out0 && (out1 || op != ROVER_POLICY_MATH_SINCOSPI), "rover_policy_math: NULL argument");
    policy_math_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(op, a, out0, out1, n);
    return check_launch("policy_math_kernel");
}
