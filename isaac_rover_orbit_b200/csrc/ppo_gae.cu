// PPO returns and advantages over the rollout memory: skrl 1.1.0 PPO._update -> compute_gae (DESIGN.md section 2).
//
// Three launches on the caller's stream, each under programmatic dependent launch:
//   (a) recurrence      -- one thread per environment walks the T steps backwards; the loads of kChunk steps are issued
//                          before the dependent chain consumes them.  Writes returns and the raw advantages, and one fp64
//                          partial sum of the advantages per block;
//   (b) squared devs    -- every block reduces (a)'s partials to mean64 = sum / n and stores its fp64 partial of
//                          sum (a - mean64)^2 over a grid-stride share of the entries;
//   (c) normalise       -- every block reduces both partial arrays (same fixed order as in (b)) and rewrites its share of
//                          the advantages as fl32(fl32(a - mean_f) / fl32(std_f + 1e-8f)).
// Every reduction has a fixed order and there are no float atomics: results are deterministic, and the launches are
// graph-capturable.  Block counts depend on (T, N) only, never on the device.
#include "common.cuh"

namespace rover {

constexpr int kGaeThreads = 128;   // (a): environments per block
constexpr int kGaeChunk = 16;      // (a): steps whose loads are in flight together
constexpr int kFlatThreads = 256;  // (b), (c)
constexpr int kFlatItems = 4;      // (b), (c): entries per thread per loop trip
constexpr int kFlatMaxBlocks = 592;

static inline int gae_blocks(int32_t n_envs) { return (n_envs + kGaeThreads - 1) / kGaeThreads; }

static inline int flat_blocks(int64_t n) {
    const int64_t b = (n + (int64_t)kFlatThreads * kFlatItems - 1) / ((int64_t)kFlatThreads * kFlatItems);
    return (int)(b < kFlatMaxBlocks ? b : kFlatMaxBlocks);
}

// Sum of one double per thread; every thread gets the same value (xor butterfly, then the warp sums in warp order).
template <int kThreads>
__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = red[0];
#pragma unroll
    for (int w = 1; w < kThreads / 32; ++w) s += red[w];
    __syncthreads();  // red may be reused
    return s;
}

// Sum of a partial array in a fixed order (thread t: entries t, t + kThreads, ... in turn; then block_sum).
template <int kThreads>
__device__ __forceinline__ double sum_partials(const double* __restrict__ p, int count, double* red) {
    double s = 0.0;
    for (int i = threadIdx.x; i < count; i += kThreads) s += p[i];
    return block_sum<kThreads>(s, red);
}

__global__ void __launch_bounds__(kGaeThreads)
ppo_gae_recurrence_kernel(const float* __restrict__ rewards, const uint8_t* __restrict__ dones,
                          const float* __restrict__ values, const float* __restrict__ last_values, int T, int N,
                          float gamma, float lam, float* __restrict__ returns, float* __restrict__ advantages,
                          double* __restrict__ adv_partials) {
    __shared__ double red[kGaeThreads / 32];
    grid_dependency_wait();
    const int e = blockIdx.x * kGaeThreads + threadIdx.x;
    double sum = 0.0;
    if (e < N) {
        float next_value = last_values[e];
        float adv = 0.0f;  // skrl: advantage = 0, so the first lambda * advantage is lambda * 0
        for (int i0 = T - 1; i0 >= 0; i0 -= kGaeChunk) {
            float r[kGaeChunk], v[kGaeChunk];
            uint8_t d[kGaeChunk];
#pragma unroll
            for (int k = 0; k < kGaeChunk; ++k) {
                if (i0 - k >= 0) {
                    const size_t o = (size_t)(i0 - k) * N + e;
                    r[k] = rewards[o];
                    v[k] = values[o];
                    d[k] = dones[o];
                }
            }
#pragma unroll
            for (int k = 0; k < kGaeChunk; ++k) {
                if (i0 - k >= 0) {
                    // advantage = rewards[i] - values[i] + discount_factor * not_dones[i] * (nv + lambda * advantage),
                    // every operation rounded on its own, in Python's evaluation order (no contraction)
                    const float not_done = d[k] == 0 ? 1.0f : 0.0f;
                    adv = __fadd_rn(__fsub_rn(r[k], v[k]),
                                    __fmul_rn(__fmul_rn(gamma, not_done), __fadd_rn(next_value, __fmul_rn(lam, adv))));
                    const size_t o = (size_t)(i0 - k) * N + e;
                    advantages[o] = adv;
                    returns[o] = __fadd_rn(adv, v[k]);
                    sum += (double)adv;
                    next_value = v[k];
                }
            }
        }
    }
    sum = block_sum<kGaeThreads>(sum, red);
    if (threadIdx.x == 0) adv_partials[blockIdx.x] = sum;
}

__global__ void __launch_bounds__(kFlatThreads)
ppo_gae_sq_dev_kernel(const float* __restrict__ advantages, int64_t n, const double* __restrict__ adv_partials,
                      int n_adv_partials, double* __restrict__ m2_partials) {
    __shared__ double red[kFlatThreads / 32];
    grid_dependency_wait();
    const double mean = sum_partials<kFlatThreads>(adv_partials, n_adv_partials, red) / (double)n;
    const int64_t stride = (int64_t)gridDim.x * kFlatThreads;
    double m2 = 0.0;
    for (int64_t j0 = (int64_t)blockIdx.x * kFlatThreads + threadIdx.x; j0 < n; j0 += stride * kFlatItems) {
        float a[kFlatItems];
#pragma unroll
        for (int k = 0; k < kFlatItems; ++k) a[k] = j0 + k * stride < n ? advantages[j0 + k * stride] : 0.0f;
#pragma unroll
        for (int k = 0; k < kFlatItems; ++k) {
            if (j0 + k * stride < n) {
                const double dev = (double)a[k] - mean;
                m2 += dev * dev;
            }
        }
    }
    m2 = block_sum<kFlatThreads>(m2, red);
    if (threadIdx.x == 0) m2_partials[blockIdx.x] = m2;
}

__global__ void __launch_bounds__(kFlatThreads)
ppo_gae_normalise_kernel(float* __restrict__ advantages, int64_t n, const double* __restrict__ adv_partials,
                         int n_adv_partials, const double* __restrict__ m2_partials, int n_m2_partials) {
    __shared__ double red[kFlatThreads / 32];
    grid_dependency_wait();
    const double mean = sum_partials<kFlatThreads>(adv_partials, n_adv_partials, red) / (double)n;
    const double m2 = sum_partials<kFlatThreads>(m2_partials, n_m2_partials, red);
    // torch: (advantages - advantages.mean()) / (advantages.std() + 1e-8), unbiased std (NaN for n = 1)
    const float mean_f = __double2float_rn(mean);
    const float denom = __fadd_rn(__double2float_rn(sqrt(m2 / (double)(n - 1))), 1e-8f);
    const int64_t stride = (int64_t)gridDim.x * kFlatThreads;
    for (int64_t j0 = (int64_t)blockIdx.x * kFlatThreads + threadIdx.x; j0 < n; j0 += stride * kFlatItems) {
        float a[kFlatItems];
#pragma unroll
        for (int k = 0; k < kFlatItems; ++k) a[k] = j0 + k * stride < n ? advantages[j0 + k * stride] : 0.0f;
#pragma unroll
        for (int k = 0; k < kFlatItems; ++k)
            if (j0 + k * stride < n) advantages[j0 + k * stride] = __fdiv_rn(__fsub_rn(a[k], mean_f), denom);
    }
}

}  // namespace rover

extern "C" int64_t rover_ppo_gae_work_bytes(int32_t T, int32_t n_envs) {
    if (T < 0 || n_envs < 0) return -1;
    if (T == 0 || n_envs == 0) return 0;
    return 8 * ((int64_t)rover::gae_blocks(n_envs) + rover::flat_blocks((int64_t)T * n_envs));
}

extern "C" int rover_ppo_gae(const float* rewards, const uint8_t* dones, const float* values, const float* last_values,
                             int32_t T, int32_t n_envs, float discount_factor, float lambda_coefficient, float* returns,
                             float* advantages, void* work, int64_t work_bytes, void* stream) {
    using namespace rover;
    ROVER_CHECK(T >= 0 && n_envs >= 0, "rover_ppo_gae: negative sizes");
    if (T == 0 || n_envs == 0) return 0;
    ROVER_CHECK(rewards && dones && values && last_values && returns && advantages && work, "rover_ppo_gae: NULL buffer");
    const int64_t need = rover_ppo_gae_work_bytes(T, n_envs);
    ROVER_CHECK(work_bytes >= need && (reinterpret_cast<uintptr_t>(work) & 7) == 0,
                "rover_ppo_gae: work area of %lld bytes (8-byte aligned) needed, got %lld", (long long)need,
                (long long)work_bytes);
    const int64_t n = (int64_t)T * n_envs;
    const int nb_gae = gae_blocks(n_envs), nb_flat = flat_blocks(n);
    double* adv_partials = static_cast<double*>(work);
    double* m2_partials = adv_partials + nb_gae;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    ROVER_CUDA(launch_overlapped(ppo_gae_recurrence_kernel, dim3(nb_gae), dim3(kGaeThreads), 0, s, rewards, dones, values,
                                 last_values, (int)T, (int)n_envs, discount_factor, lambda_coefficient, returns, advantages,
                                 adv_partials));
    if (int rc = check_launch("ppo_gae_recurrence_kernel")) return rc;
    ROVER_CUDA(launch_overlapped(ppo_gae_sq_dev_kernel, dim3(nb_flat), dim3(kFlatThreads), 0, s,
                                 static_cast<const float*>(advantages), n, static_cast<const double*>(adv_partials), nb_gae,
                                 m2_partials));
    if (int rc = check_launch("ppo_gae_sq_dev_kernel")) return rc;
    ROVER_CUDA(launch_overlapped(ppo_gae_normalise_kernel, dim3(nb_flat), dim3(kFlatThreads), 0, s, advantages, n,
                                 static_cast<const double*>(adv_partials), nb_gae, static_cast<const double*>(m2_partials),
                                 nb_flat));
    return check_launch("ppo_gae_normalise_kernel");
}
