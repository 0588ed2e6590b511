// Counter-based random variates of the reset path, generated where they are consumed.
//
// The reference draws them with torch's global generator on the step path (reference root relative):
//   rover_envs/envs/navigation/mdp/randomizations.py:22   torch.randperm(len(spawn_locations))[:K]
//   rover_envs/envs/navigation/mdp/randomizations.py:30   torch.rand(K) * 2 * pi                      (spawn yaw)
//   .../utils/terrains/terrain_importer.py:94-95          Tensor.uniform_(-pi, pi)                    (target heading)
//   .../utils/terrains/terrain_importer.py:169            torch.rand(K) * 2 * pi, once per rejection round
// A torch generator stream cannot be reproduced inside a kernel, and four extra launches per step plus a [N, rounds]
// table in HBM are exactly what a fused step is meant to avoid.  Here every variate is a pure function of
// (seed, step, env, role): Philox4x32-10 (Salmon et al., SC'11; the generator behind curand / torch CUDA) with
//   key     = (seed_lo, seed_hi)
//   counter = (env, step_lo, step_hi, stream)      stream 0: {yaw, heading, -, -};  stream 1 + q: theta rounds 4q .. 4q+3
// and the without-replacement spawn draw is a keyed bijection of [0, n_spawns) evaluated at the ENV ID (Kensler's
// cycle-walking hash permutation: add key / multiply by an odd constant / xor-shift on the next power of two, repeated
// until the value falls inside the range), keyed by Philox(counter = (0xffffffff, step_lo, step_hi, 0xffffffff)).
// The reference assigns randperm(len)[:K] to the K reset envs in ascending order; a uniformly random permutation
// evaluated at K distinct env ids has the same distribution (K distinct, uniformly drawn rows) and needs no reset rank --
// no cross-block prefix sum in front of the reset chain.
// The same functions are compiled for the host (rover_rng_variates) so that the oracle consumes identical numbers.
//
// The policy's action noise (skrl GaussianMixin.act: torch.randn(N, 2) -> Normal.rsample) comes from the same
// generator with its own {seed, step} state and its own stream:
//   counter = (env, step_lo, step_hi, kActionStream)    -> normal2(): two N(0, 1) draws by Box-Muller
// kActionStream lies outside the reset path's streams (0 and 1 + q, q < 1024) and the spawn key's 0xffffffff.  Same
// distribution as torch's draw, not the same numbers: the same documented deviation, by design, as the spawn permutation.
// normal2 is device code only (logf / sinf / cosf of the host's libm round differently; rover_action_noise exports it).
#pragma once
#include <stdint.h>

namespace rover {

#if defined(__CUDACC__)
#define ROVER_HD __host__ __device__ __forceinline__
#else
#define ROVER_HD inline
#endif

ROVER_HD void philox_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
    hi = __umulhi(a, b);
    lo = a * b;
#else
    const uint64_t p = (uint64_t)a * (uint64_t)b;
    hi = (uint32_t)(p >> 32);
    lo = (uint32_t)p;
#endif
}

// Philox4x32-10 (Random123): 10 rounds, key schedule k += (0x9E3779B9, 0xBB67AE85)
ROVER_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                            uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0, lo0, hi1, lo1;
        philox_mulhilo(0xD2511F53u, c0, hi0, lo0);
        philox_mulhilo(0xCD9E8D57u, c2, hi1, lo1);
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0, c1 = lo1, c2 = n2, c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}

// 24 random bits -> [0, 1) on the fp32 grid torch.rand uses (multiples of 2^-24)
ROVER_HD float u01(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; }

struct RngKey {
    uint32_t seed_lo, seed_hi, step_lo, step_hi;
};

ROVER_HD RngKey make_rng_key(uint64_t seed, uint64_t step) {
    return RngKey{(uint32_t)seed, (uint32_t)(seed >> 32), (uint32_t)step, (uint32_t)(step >> 32)};
}

// the four variates of (env, stream)
ROVER_HD void rng_env_stream(const RngKey& k, uint32_t env, uint32_t stream, uint32_t (&out)[4]) {
    philox4x32_10(env, k.step_lo, k.step_hi, stream, k.seed_lo, k.seed_hi, out);
}

struct SpawnPermKey {
    uint32_t k[4];
    uint32_t mask;   // next power of two of n - 1
    uint32_t n;
};

ROVER_HD SpawnPermKey make_spawn_perm_key(const RngKey& k, uint32_t n_spawns) {
    SpawnPermKey p;
    philox4x32_10(0xffffffffu, k.step_lo, k.step_hi, 0xffffffffu, k.seed_lo, k.seed_hi, p.k);
    uint32_t m = n_spawns > 1u ? n_spawns - 1u : 1u;
    m |= m >> 1, m |= m >> 2, m |= m >> 4, m |= m >> 8, m |= m >> 16;
    p.mask = m;
    p.n = n_spawns;
    return p;
}

// row of the spawn table for env j (j < n): a bijection of [0, n), so K distinct envs draw K distinct rows
ROVER_HD uint32_t spawn_perm_at(const SpawnPermKey& p, uint32_t j) {
    const uint32_t w = p.mask;
    uint32_t x = j;
    do {  // every step below is a bijection of [0, w]; cycle-walk until the image lies in [0, n)
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            x = (x + p.k[r]) & w;
            x = (x * 0x9E3779B1u) & w;       // odd multiplier
            x ^= (x >> 5);                   // xor-shift right: invertible on any width
            x = (x * 0x85EBCA6Bu) & w;
            x ^= (x >> 3);
        }
    } while (x >= p.n);
    return x;
}

constexpr uint32_t kActionStream = 0x80000000u;

#if defined(__CUDACC__)
// Two standard-normal fp32 values of env `env`: Box-Muller on the first two words of one Philox4x32-10 call.
//   u1 = (24 bits + 1) * 2^-24 in (0, 1]   (log never sees 0)      u2 = 24 bits * 2^-24 in [0, 1)
//   r = sqrt(-2 ln u1),  z0 = r cos(2 pi u2),  z1 = r sin(2 pi u2)
// Every operation is written out with its rounding (no contraction left to the compiler).  The angle goes to
// sincospif(2 u2) = (sin, cos)(pi * 2 u2): 2 u2 is exact, so no rounded 2 pi enters, and the argument is known to be
// small -- sinf / cosf of 2 pi u2 would carry the large-argument reduction (a local-memory frame) into the forward pass.
__device__ __forceinline__ float2 normal2(const RngKey& k, uint32_t env) {
    uint32_t w[4];
    rng_env_stream(k, env, kActionStream, w);
    const float u1 = __fmul_rn((float)((w[0] >> 8) + 1u), 5.9604644775390625e-8f);
    const float u2 = __fmul_rn((float)(w[1] >> 8), 5.9604644775390625e-8f);
    const float r = __fsqrt_rn(__fmul_rn(-2.f, logf(u1)));
    float s, c;
    sincospif(__fmul_rn(2.f, u2), &s, &c);
    return make_float2(__fmul_rn(r, c), __fmul_rn(r, s));
}

// {seed, step} (device int64[2]) of a launch that draws with it.  advance: the launch takes the step once and leaves
// step + 1 behind, by the last-block pattern -- each of the n_blocks blocks takes a ticket with one atomic on the step
// word (bits 40..63 count the tickets, bits 0..39 hold the step, so step < 2^40 - 1), and the block that takes the last
// ticket writes step + 1.  One call per block, after griddepcontrol.wait (the launch in front may be the one advancing it).
constexpr int kStepTicketShift = 40;
constexpr unsigned long long kStepMask = (1ull << kStepTicketShift) - 1ull;
__device__ __forceinline__ RngKey take_step(unsigned long long* state, unsigned n_blocks, bool advance) {
    const unsigned long long seed = *reinterpret_cast<volatile unsigned long long*>(state);
    if (!advance) return make_rng_key(seed, *reinterpret_cast<volatile unsigned long long*>(state + 1) & kStepMask);
    const unsigned long long old = atomicAdd(state + 1, 1ull << kStepTicketShift);
    const unsigned long long step = old & kStepMask;
    if ((old >> kStepTicketShift) == (unsigned long long)n_blocks - 1ull) atomicExch(state + 1, step + 1ull);
    return make_rng_key(seed, step);
}
#endif

}  // namespace rover
