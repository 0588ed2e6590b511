// Fused non-physics MDP step of AAURoverEnv-v0: two launches around the (external) physics state.
//
//   mdp_pre_step_kernel   one thread per env: action manager shift, AckermannAction2 kinematics, counters,
//                         the 4 terminations, the 7 weighted rewards + episodic sums, reset flags.
//   mdp_post_step_kernel  one thread per env: rank of each reset env (block prefix + warp scan), spawn/yaw
//                         reset, manager resets + episode statistics, bounded target rejection sampling on the
//                         valid-location mask, heightmap lookup, command metrics / update, observation head.
//
// Reference lines restated (relative to the reference root):
//   rover_envs/mdp/actions/ackermann_actions.py:226-322        rover_envs/envs/navigation/mdp/rewards.py:14-137
//   rover_envs/envs/navigation/mdp/terminations.py:14-64        .../mdp/observations.py:15-32
//   .../mdp/randomizations.py:12-39                             .../utils/terrains/terrain_importer.py:74-175
//   .../utils/terrains/terrain_utils.py:62-84, 202-223          .../entrypoints/rover_env.py:61-102 (ordering)
// plus the ORBIT manager combine rules and math helpers of SURVEY.md Appendix A.1/A.2.
// fp32 arithmetic follows the reference's operation order; contraction is disabled (__f*_rn) wherever a
// value is compared against a threshold or truncated to an index.
#include "mdp_env.cuh"

namespace rover {

#ifndef ROVER_MDP_DBG
#define ROVER_MDP_DBG 0  // 1: globaltimer (ns) stamps of every block of the single-launch step (profiles/mdp_timeline.py)
#endif
#if ROVER_MDP_DBG
__device__ unsigned long long g_mdp_dbg[8][1024];
#define MDP_STAMP(slot)                                                                  \
    do {                                                                                 \
        if (threadIdx.x == 0 && blockIdx.x < 1024) {                                     \
            unsigned long long t__;                                                      \
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t__));                       \
            g_mdp_dbg[slot][blockIdx.x] = t__;                                           \
        }                                                                                \
    } while (0)
#else
#define MDP_STAMP(slot) \
    do {                \
    } while (0)
#endif


__global__ void ackermann_kernel(const float* __restrict__ actions, int n, const __grid_constant__ RoverMdpParams P,
                                 float* __restrict__ processed, float* __restrict__ jp, float* __restrict__ jv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float lin_p = __fadd_rn(__fmul_rn(actions[2 * i], P.scale_lin), P.offset_lin);
    const float ang_p = __fadd_rn(__fmul_rn(actions[2 * i + 1], P.scale_ang), P.offset_ang);
    if (processed) {
        processed[2 * i] = lin_p;
        processed[2 * i + 1] = ang_p;
    }
    ackermann_dispatch(P, lin_p, ang_p, jp + 4 * (size_t)i, jv + 6 * (size_t)i);
}

__global__ void __launch_bounds__(ROVER_MDP_BLOCK)
mdp_pre_step_kernel(const float* __restrict__ new_actions, const float* __restrict__ force, int n,
                    const __grid_constant__ RoverMdpParams P, const __grid_constant__ RoverMdpState S,
                    const __grid_constant__ RoverMdpOut O, int phases) {
    const int i = blockIdx.x * ROVER_MDP_BLOCK + threadIdx.x;
    const bool reset = pre_step_env(i, new_actions, force, n, P, S, O, phases);
    if (phases & ROVER_PRE_TERMS) {
        const int cnt = __syncthreads_count(reset);
        if (threadIdx.x == 0) O.block_reset_counts[blockIdx.x] = cnt;
    }
}


// {seed, step}: one uniform load per thread (L2 / L1 hit after the first); the step word is advanced by the last block
// of the launch, after every block has read it
template <bool kRng>
__device__ __forceinline__ RngKey load_rng_key(const VariatesDev& V) {
    if (!kRng) return make_rng_key(0ull, 0ull);
    return make_rng_key(V.rng[0], *reinterpret_cast<volatile unsigned long long*>(V.rng + 1));
}

// barrier of the ROVER_MDP_BLOCK threads that own an env (the single-launch step runs extra kinematics warps in the CTA
// that are gone by then: a named barrier with an explicit count instead of __syncthreads())
__device__ __forceinline__ void mdp_block_sync() { asm volatile("bar.sync 1, %0;" ::"n"(ROVER_MDP_BLOCK) : "memory"); }

// Hardware barriers of the split CTA (2 env warps + 2 kinematics warps = 128 threads; 0 is __syncthreads, 1 the env warps'
// own barrier above).  One side arrives, the other waits: producer / consumer hand-offs through shared memory.
enum SplitBarrier : int {
    kBarTicket = 2,      // env warps took the CTA's ticket            -> kinematics warps (launch-wide reduction if it was the last)
    kBarKinematics = 3,  // the 64 kinematics threads among themselves (publication, reduction)
    kBarSnapshot = 4,    // kinematics warps of CTA 0 read the totals they publish -> env warps (before their ticket)
    kBarHandoff = 5,     // kinematics warps: variates + would-be spawn rows       -> env warps
    kBarResetFlags = 6,  // env warps: which envs reset                              -> kinematics warps
    kBarTargets = 7,     // kinematics warps: the new targets                        -> env warps
};
template <int kId>
__device__ __forceinline__ void split_arrive() { asm volatile("bar.arrive %0, 128;" ::"n"(kId) : "memory"); }
template <int kId>
__device__ __forceinline__ void split_wait() { asm volatile("bar.sync %0, 128;" ::"n"(kId) : "memory"); }

// shared memory of one MDP CTA
struct MdpShared {
    int warp_cnt[ROVER_MDP_BLOCK / 32];
    int block_base;
    float red[ROVER_MDP_BLOCK / 4][kStats];  // 16 row groups of the last-block reduction (>= warps per block)
    double pub[kStats];
    int is_last;
    // split CTA: what the kinematics warps hand to the env warps (hardware barrier 5) -- the spawn row and the stream-0
    // variates each env WOULD use if it reset or re-drew its target this step
    int hand_idx[ROVER_MDP_BLOCK];
    float hand[5][ROVER_MDP_BLOCK];  // spawn x, y, z, yaw_u, heading_u
    // ... what the env warps tell them (barrier 6: which envs reset) and get back (barrier 7: the new target of every env that
    // resets or whose command timer ran out -- the rejection sampling, a cold miss and ~400 instructions, runs beside
    // the env warps' reward / spawn / manager-reset work)
    unsigned char reset_flag[ROVER_MDP_BLOCK];
    float target[4][ROVER_MDP_BLOCK];  // x, y, z, exhausted
};

// barrier among 64 threads on hardware barrier kId
template <int kId>
__device__ __forceinline__ void sync64() { asm volatile("bar.sync %0, 64;" ::"n"(kId) : "memory"); }

// The block's share of the 16 episode statistics -> its row of block_stats, then a ticket: the CTA that takes the last
// one owns the launch-wide reduction (sh.is_last).  Called by the ROVER_MDP_BLOCK threads that own an env.
__device__ __forceinline__ void publish_block_stats(float (&st)[kStats], MdpShared& sh, int bid, int n_blocks,
                                                    float* __restrict__ block_stats, unsigned int* __restrict__ done_counter,
                                                    bool after_snapshot = false) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    warp_stats_reduce(st, lane, sh.red[wid]);
    mdp_block_sync();
    if (threadIdx.x < kStats) {
        float v = 0.f;
        for (int w = 0; w < ROVER_MDP_BLOCK / 32; ++w) v += sh.red[w][threadIdx.x];
        block_stats[(size_t)bid * kStats + threadIdx.x] = v;
    }
    __threadfence();
    mdp_block_sync();
    MDP_STAMP(4);
    // (split CTA 0 of a multi-GPU run: its kinematics warps have read the totals they publish -- hardware barrier 4 -- before
    // this CTA's ticket can make the launch-wide reduction, which rewrites those totals, possible)
    if (after_snapshot) split_wait<kBarSnapshot>();
    if (threadIdx.x == 0) sh.is_last = (atomicAdd(done_counter, 1u) == (unsigned)n_blocks - 1u) ? 1 : 0;
}

// Launch-wide reduction by the CTA that took the last ticket; `tid` in [0, 64), the 64 callers synchronise on hardware
// barrier kBar.  Fixed summation tree (deterministic, same result for the same inputs whatever the block schedule): thread
// t owns the statistics quad c = t % 4 of the block rows g, g + 16, ... (g = t / 4): float4 loads, kUnroll of them in
// flight per thread, so the 16 KB of partials (L2) cost one or two round trips instead of a chain of them; the 16 row
// groups are then combined in order of g.
// ---- multi-GPU: store this rank's running totals `total` (threads 0..15 of the 64 callers hold one each) into the rank's
//      slot of every rank's mailbox (peer stores over NVLink).  A slot holds a sequence number and two value buffers; the
//      writer fills buffer (seq + 1) & 1 in every mailbox, fences once, then stores seq + 1 everywhere -- one system-scope
//      fence per publication, all peers in flight together.  No collective, no extra launch.
template <int kBar>
__device__ __forceinline__ void publish_totals(int tid, double total, MdpShared& sh, const StatsExchangeDev& X) {
    if (tid < kStats) sh.pub[tid] = total;
    sync64<kBar>();
    const unsigned long long seq = *X.sequence + 1ull;
    for (int e = tid; e < X.world * kStats; e += ROVER_MDP_BLOCK) {
        const int p = e / kStats, k = e % kStats;
        unsigned char* slot = static_cast<unsigned char*>(X.peer_mailbox[p]) + (size_t)X.rank * ROVER_MAILBOX_SLOT_BYTES;
        reinterpret_cast<volatile double*>(slot + 8)[(seq & 1ull) * kStats + k] = sh.pub[k];
    }
    __threadfence_system();
    sync64<kBar>();
    for (int p = tid; p < X.world; p += ROVER_MDP_BLOCK) {
        unsigned char* slot = static_cast<unsigned char*>(X.peer_mailbox[p]) + (size_t)X.rank * ROVER_MAILBOX_SLOT_BYTES;
        *reinterpret_cast<volatile unsigned long long*>(slot) = seq;
    }
    if (tid == 0) *X.sequence = seq;
}

// kPublish = false (the split single-launch step): the totals are only accumulated here; they were / will be published by
// CTA 0's kinematics warps at the START of a launch (mdp_fused_step_kernel), off the step's critical path.
template <bool kFused, bool kRng, int kBar, bool kPublish = true>
__device__ __forceinline__ void final_stats_reduce(int tid, MdpShared& sh, int n_blocks, const RoverMdpParams& P,
                                                   const VariatesDev& V, const float* __restrict__ block_stats,
                                                   unsigned int* __restrict__ done_counter, float* __restrict__ stats,
                                                   float* __restrict__ log_out, int phases, const StatsExchangeDev& X,
                                                   unsigned long long* __restrict__ lookback, unsigned epoch) {
    static_assert(ROVER_MDP_BLOCK == 64 && kStats == 16, "last-block reduction layout");
    constexpr int kGroups = ROVER_MDP_BLOCK / 4, kUnroll = 16;
    const int c4 = tid & 3, g = tid >> 2;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (unsigned b0 = g; b0 < (unsigned)n_blocks; b0 += kGroups * kUnroll) {
        float4 x[kUnroll];
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) {
            const unsigned bb = b0 + u * kGroups;
            x[u] = bb < (unsigned)n_blocks ? __ldcg(reinterpret_cast<const float4*>(block_stats + (size_t)bb * kStats) + c4)
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < kUnroll; ++u) acc.x += x[u].x, acc.y += x[u].y, acc.z += x[u].z, acc.w += x[u].w;
    }
    sync64<kBar>();  // sh.red[] is free: every thread of the CTA passed the block-level reduction
    sh.red[g][4 * c4 + 0] = acc.x, sh.red[g][4 * c4 + 1] = acc.y, sh.red[g][4 * c4 + 2] = acc.z, sh.red[g][4 * c4 + 3] = acc.w;
    sync64<kBar>();
    double total = 0.0;
    if (tid < kStats) {
        float t = 0.f;
        for (int q = 0; q < kGroups; ++q) t += sh.red[q][tid];
        stats[tid] += t;
        // extras["log"] of the ORBIT managers' reset() (A.2), refreshed only by a launch that reset something -- the
        // reference calls _reset_idx only then (rover_env.py:89-91), so the previous values stay visible otherwise:
        //   Episode Reward/<term> = mean(episode_sums[ids]) / max_episode_length_s, Episode Termination/<term> =
        //   count, Metrics/target_pose/<m> = mean over ids; [13] = number of resets, [14], [15] as in stats
        const float cnt = __shfl_sync(0xffffu, t, 13);  // the 16 statistics live in lanes 0..15 of one warp
        if (log_out != nullptr && (phases & ROVER_PHASE_MANAGERS) && cnt > 0.f) {
            float v = t;
            if (tid < ROVER_NUM_REWARD_TERMS) v = __fdiv_rn(__fdiv_rn(t, cnt), P.episode_length_s);
            else if (tid == 11 || tid == 12) v = __fdiv_rn(t, cnt);
            log_out[tid] = v;
        }
        if (tid == 0) {
            *done_counter = 0u;  // re-arm for the next launch
            if (kRng) V.rng[1] = V.rng[1] + 1ull;  // next launch = next step of the variate streams
            if (kFused && !kRng) {  // fused step, explicit variates: next launch = next epoch, tickets from 0 again
                lookback[n_blocks] = 0ull;
                lookback[n_blocks + 1] = (unsigned long long)(epoch + 1u);
            }
        }
        if (X.world > 0) {
            total = X.cumulative[tid] + (double)t;
            X.cumulative[tid] = total;
        }
    }
    if (kPublish && X.world > 0) publish_totals<kBar>(tid, total, sh, X);
}

// hardware barrier 2: the env warps of a split CTA announce the ticket (arrive), its kinematics warps wait for it (sync)
__device__ __forceinline__ void split_ticket_arrive() { split_arrive<kBarTicket>(); }
__device__ __forceinline__ void split_ticket_wait() { split_wait<kBarTicket>(); }

// kSplit (single-launch step with in-kernel variates): the statistics leave the env warps as soon as they are complete --
// after the target draw, before metrics / command update / observation head -- where the fence in front of the ticket
// finds no recent stores to wait for, and the launch-wide reduction of the last CTA is done by its kinematics warps
// while the env warps finish their envs.
template <bool kFused, bool kRng, bool kSplit = false>
__device__ __forceinline__ void post_step_block(MdpShared& sh, int bid, int n_blocks, bool reset_in, float* __restrict__ root_pos_w,
                                                float* __restrict__ root_quat_w, int n, const RoverMdpParams& P,
                                                const RoverMdpState& S, const RoverMdpOut& O, const Tables& T,
                                                const VariatesDev& V, long long* __restrict__ out_spawn_index,
                                                float* __restrict__ block_stats, unsigned int* __restrict__ done_counter,
                                                float* __restrict__ stats, float* __restrict__ log_out,
                                                float* __restrict__ obs, int obs_stride, int phases,
                                                const StatsExchangeDev& X, unsigned long long* __restrict__ lookback,
                                                unsigned epoch, const RngKey key, const SpawnEarly early = SpawnEarly()) {
    int(&warp_cnt)[ROVER_MDP_BLOCK / 32] = sh.warp_cnt;
    int& block_base = sh.block_base;
    const int i = bid * ROVER_MDP_BLOCK + threadIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const bool valid = i < n;
    const bool reset = kFused ? (valid && reset_in) : (valid && O.reset_flags[i] != 0);

    EnvRegs er;
    post_env_load<kRng>(i, valid, root_pos_w, root_quat_w, S, V, er);

    // ---- explicit variates: rank of this env among the reset envs in ascending env order (== reset_buf.nonzero() order),
    //      the index into spawn_perm (randperm(len)[:K] assigned in that order, randomizations.py:22).  The in-kernel
    //      generator needs no rank: its spawn draw is a keyed permutation of [0, n_spawns) evaluated at the ENV ID -- K
    //      distinct envs get K distinct rows, and a uniformly random permutation evaluated at K distinct points has
    //      exactly the distribution of randperm(len)[:K] -- so the cross-block prefix (a dependent load in front of the
    //      reset chain; a look-back in the single-launch step) disappears.
    int rank = 0;
    if constexpr (!kRng) {
        const unsigned ballot = __ballot_sync(0xffffffffu, reset);
        if (lane == 0) warp_cnt[wid] = __popc(ballot);
        if (!kFused) {
            if (wid == 0) {
                int acc = 0;
                for (int b = lane; b < bid; b += 32) acc += O.block_reset_counts[b];
                for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
                if (lane == 0) block_base = acc;
            }
            mdp_block_sync();
        } else {
            mdp_block_sync();
            if (wid == 0) {
                // decoupled look-back (single pass): publish this block's count, walk back over the predecessors' descriptors
                // until one carries an inclusive prefix, publish our own.  Logical block ids are tickets, so every
                // predecessor has started; descriptors are tagged with the launch epoch, so nothing is re-zeroed.
                int cnt = 0;
                for (int w = 0; w < ROVER_MDP_BLOCK / 32; ++w) cnt += warp_cnt[w];
                volatile unsigned long long* desc = lookback;
                int base = 0;
                if (bid > 0) {
                    if (lane == 0) desc[bid] = make_lookback(epoch, kDescAggregate, (unsigned)cnt);
                    int look = bid - 1;
                    while (true) {
                        const int idx = look - lane;
                        unsigned long long d = make_lookback(epoch, kDescPrefix, 0u);  // before block 0: prefix 0
                        if (idx >= 0) {
                            do {
                                d = desc[idx];
                            } while ((unsigned)(d >> 34) != (epoch & 0x3fffffffu) || ((d >> 32) & 3ull) == 0ull);
                        }
                        const bool is_prefix = ((d >> 32) & 3ull) == kDescPrefix;
                        const unsigned pmask = __ballot_sync(0xffffffffu, is_prefix);
                        const int first = pmask ? __ffs(pmask) - 1 : 32;  // closest predecessor with an inclusive prefix
                        int v = (lane <= first) ? (int)(unsigned)(d & 0xffffffffull) : 0;
                        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                        base += v;
                        if (pmask) break;
                        look -= 32;
                    }
                }
                if (lane == 0) {
                    __threadfence();
                    desc[bid] = make_lookback(epoch, kDescPrefix, (unsigned)(base + cnt));
                    block_base = base;
                }
            }
            mdp_block_sync();
        }
        rank = block_base + __popc(ballot & ((1u << lane) - 1u));
        for (int w = 0; w < wid; ++w) rank += warp_cnt[w];

    }

    float st[kStats];
    if constexpr (kSplit) {
        post_env_work<kRng>(
            i, valid, reset, rank, er, root_pos_w, root_quat_w, P, S, O, T, V, key, out_spawn_index, obs, obs_stride, phases, st,
            NoPoseHook(), early,
            [&](float(&stv)[kStats]) {
                publish_block_stats(stv, sh, bid, n_blocks, block_stats, done_counter, X.world > 0 && bid == 0);
                __threadfence_block();
                split_ticket_arrive();
            },
            [&](float& tx, float& ty, float& tz, bool& ex) {  // the targets the kinematics warps drew (barrier 7)
                split_wait<kBarTargets>();
                const int t = (int)threadIdx.x;
                tx = sh.target[0][t], ty = sh.target[1][t], tz = sh.target[2][t], ex = sh.target[3][t] != 0.f;
                return true;
            });
        MDP_STAMP(3);
        return;
    } else {
        post_env_work<kRng>(i, valid, reset, rank, er, root_pos_w, root_quat_w, P, S, O, T, V, key, out_spawn_index, obs,
                            obs_stride, phases, st, NoPoseHook(), early);
        MDP_STAMP(3);
        // ---- deterministic episode statistics: warp shuffle -> block -> last block sums the partials in order
        publish_block_stats(st, sh, bid, n_blocks, block_stats, done_counter);
        mdp_block_sync();
        MDP_STAMP(5);
        if (sh.is_last) {
            final_stats_reduce<kFused, kRng, 1>((int)threadIdx.x, sh, n_blocks, P, V, block_stats, done_counter, stats, log_out,
                                                phases, X, lookback, epoch);
            MDP_STAMP(6);
        }
    }
}

template <bool kRng>
__global__ void __launch_bounds__(ROVER_MDP_BLOCK)
mdp_post_step_kernel(float* __restrict__ root_pos_w, float* __restrict__ root_quat_w, int n,
                     const __grid_constant__ RoverMdpParams P, const __grid_constant__ RoverMdpState S,
                     const __grid_constant__ RoverMdpOut O, const __grid_constant__ Tables T,
                     const __grid_constant__ VariatesDev V, long long* __restrict__ out_spawn_index,
                     float* __restrict__ block_stats, unsigned int* __restrict__ done_counter, float* __restrict__ stats,
                     float* __restrict__ log_out, float* __restrict__ obs, int obs_stride, int phases,
                     const __grid_constant__ StatsExchangeDev X) {
    __shared__ MdpShared sh;
    grid_dependency_trigger();  // (see mdp_fused_step_kernel)
    post_step_block<false, kRng>(sh, (int)blockIdx.x, (int)gridDim.x, false, root_pos_w, root_quat_w, n, P, S, O, T, V,
                                 out_spawn_index, block_stats, done_counter, stats, log_out, obs, obs_stride, phases, X,
                                 nullptr, 0u, load_rng_key<kRng>(V));
}

// rover_mdp_step: pre-step + post-step of one env block in ONE launch (the reset rank comes from a look-back instead of a
// second launch; the pre-step's outputs of an env are consumed by the same thread).  lookback: [n_blocks] descriptors,
// then the ticket counter and the epoch (both maintained by the kernel itself, so the launch can sit in a CUDA graph).
// Logical block ids are ALWAYS tickets: the look-back spins on predecessors, which is only safe if every predecessor
// has started -- blockIdx order guarantees that on an idle GPU only, a ticket taken at block start guarantees it under
// MPS, concurrent kernels or a partitioned device as well (one atomic per block).
template <bool kRng, bool kSplit = false>
__global__ void __launch_bounds__(kSplit ? 2 * ROVER_MDP_BLOCK : ROVER_MDP_BLOCK)
mdp_fused_step_kernel(const float* __restrict__ new_actions, const float* __restrict__ force,
                      float* __restrict__ root_pos_w, float* __restrict__ root_quat_w, int n,
                      const __grid_constant__ RoverMdpParams P, const __grid_constant__ RoverMdpState S,
                      const __grid_constant__ RoverMdpOut O, const __grid_constant__ Tables T,
                      const __grid_constant__ VariatesDev V, long long* __restrict__ out_spawn_index,
                      float* __restrict__ block_stats, unsigned int* __restrict__ done_counter, float* __restrict__ stats,
                      float* __restrict__ log_out, float* __restrict__ obs, int obs_stride, int pre_phases, int phases,
                      const __grid_constant__ StatsExchangeDev X, unsigned long long* __restrict__ lookback) {
    __shared__ int s_bid;
    __shared__ unsigned s_epoch;
    __shared__ MdpShared sh;
    const int n_blocks = (int)gridDim.x;
    int bid = (int)blockIdx.x;
    unsigned epoch = 0u;
    if constexpr (!kRng) {  // (the in-kernel generator needs no reset rank, hence no look-back and no ticket)
        grid_dependency_wait();  // the ticket counter is re-armed by the previous launch of this kernel
        if (threadIdx.x == 0) {
            s_epoch = (unsigned)*reinterpret_cast<volatile unsigned long long*>(lookback + n_blocks + 1);
            s_bid = (int)atomicAdd(lookback + n_blocks, 1ull);
        }
        __syncthreads();
        bid = s_bid;
        epoch = s_epoch;
    }
    // the kernel behind this one on the stream (the height scan) may bring its CTAs up as SMs become free: it waits for
    // this grid's completion before it reads a pose (common.cuh, launch_overlapped)
    grid_dependency_trigger();
    MDP_STAMP(0);
    if constexpr (kSplit) {
        // warps 2, 3 of the CTA work beside the warps that own the envs, on everything that does not depend on an env's
        // reset decision: the variate stream / spawn row each env would use (handed over through shared memory), the
        // action term's kinematics (AckermannAction2: ~25 % of the pre-step's dependent chain, a function of the new action
        // only), on multi-GPU runs the publication of the rank's totals, and at the end the launch-wide reduction
        static_assert(kRng, "the split CTA is the in-kernel-variates step");
        if (threadIdx.x >= ROVER_MDP_BLOCK) {
            const int ht = (int)threadIdx.x - ROVER_MDP_BLOCK;
            grid_dependency_wait();
            // multi-GPU: CTA 0's kinematics warps publish the rank's running totals AS OF THE PREVIOUS LAUNCH to the peers'
            // mailboxes -- two NVLink round trips (values, fence, sequence number) that would otherwise sit between the
            // launch-wide reduction and the end of the kernel (5 us per step at 2 GPUs), here beside ~10 us of env work.
            // The mailboxes therefore run one launch behind; rover_stats_publish (P2PStats.flush) brings them up to date.
            const bool publisher = X.world > 0 && bid == 0;
            double snapshot = 0.0;
            if (publisher) {
                if (ht < kStats) snapshot = X.cumulative[ht];
                split_arrive<kBarSnapshot>();  // read before this CTA's ticket (publish_block_stats)
            }
            {   // the env's variate stream 0 and its would-be spawn row: rng state -> Philox -> keyed permutation -> row, a
                // chain of two cold misses and ~350 instructions that the env warps no longer carry
                const int hi = bid * ROVER_MDP_BLOCK + ht;
                const RngKey hkey = load_rng_key<kRng>(V);
                int idx = -1;
                float hx = 0.f, hy = 0.f, hz = 0.f, yaw_u = 0.f, heading_u = 0.f;
                if (hi < n) {
                    if (phases & ROVER_PHASE_SPAWN) {
                        idx = (int)spawn_perm_at(make_spawn_perm_key(hkey, (uint32_t)T.n_spawns), (uint32_t)hi);
                        const float* sp = T.spawn + 3 * (size_t)idx;
                        hx = __ldg(sp), hy = __ldg(sp + 1), hz = __ldg(sp + 2);
                    }
                    uint32_t w[4];
                    rng_env_stream(hkey, (uint32_t)hi, 0u, w);
                    yaw_u = u01(w[0]), heading_u = u01(w[1]);
                }
                sh.hand_idx[ht] = idx;
                sh.hand[0][ht] = hx, sh.hand[1][ht] = hy, sh.hand[2][ht] = hz, sh.hand[3][ht] = yaw_u, sh.hand[4][ht] = heading_u;
                __threadfence_block();
                split_arrive<kBarHandoff>();
                // the target draw of the envs that reset (flag from the env warps) or whose timer runs out this step:
                // the same rs_reset / rs_timer / origin rules as post_env_work, the same resample_warp
                const float tl = (hi < n && (phases & ROVER_PHASE_TIME)) ? S.time_left[hi] : 0.f;
                float ox = hx, oy = hy;
                split_wait<kBarResetFlags>();
                const bool h_reset = hi < n && sh.reset_flag[ht] != 0;
                const bool rs_reset = h_reset && (phases & ROVER_PHASE_RESAMPLE);
                const bool rs_timer = hi < n && !rs_reset && (phases & ROVER_PHASE_TIME) && __fsub_rn(tl, P.step_dt) <= 0.f;
                if ((rs_reset || rs_timer) && !(h_reset && (phases & ROVER_PHASE_SPAWN))) {
                    ox = S.env_origins[3 * (size_t)hi];
                    oy = S.env_origins[3 * (size_t)hi + 1];
                }
                float tx = 0.f, ty = 0.f, tz = 0.f;
                const bool ex = resample_warp<kRng>(hi, rs_reset || rs_timer, P, T, ox, oy, V.theta_u, hkey, V.n_rounds, tx, ty, tz);
                sh.target[0][ht] = tx, sh.target[1][ht] = ty, sh.target[2][ht] = tz, sh.target[3][ht] = ex ? 1.f : 0.f;
                __threadfence_block();
                split_arrive<kBarTargets>();
            }
            pre_step_env<kPreKinematics>(bid * ROVER_MDP_BLOCK + ht, new_actions, force, n, P, S, O, pre_phases);
            if (publisher) publish_totals<kBarKinematics>(ht, snapshot, sh, X);
            // ... then they wait for the CTA's ticket: if it was the launch's last one, the launch-wide reduction of the
            // statistics is theirs (the env warps are still busy with metrics / command update / observation head)
            split_ticket_wait();
            if (sh.is_last) {
                final_stats_reduce<true, kRng, kBarKinematics, false>(ht, sh, n_blocks, P, V, block_stats, done_counter, stats, log_out, phases,
                                                         X, lookback, 0u);
#if ROVER_MDP_DBG
                if (threadIdx.x == ROVER_MDP_BLOCK) {
                    unsigned long long t__;
                    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t__));
                    g_mdp_dbg[6][blockIdx.x] = t__;
                }
#endif
            }
            return;
        }
    }
    const int i = bid * ROVER_MDP_BLOCK + threadIdx.x;
    if (i < n) {
        // every line this env reads, requested before the first dependent use: the launch then pays ONE cold-miss latency
        // for them instead of one per stage (the compiler cannot hoist the loads over the stores in between).  First the
        // pre-step's inputs (the actions are loaded right away and lead the way) ...
        asm volatile("prefetch.global.L2 [%0];" ::"l"(S.pos_cmd_b + 3 * (size_t)i));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(S.episode_sums + ROVER_NUM_REWARD_TERMS * (size_t)i));
        {
            const float* f = force + (size_t)i * P.num_bodies * 3;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(f));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(f + P.num_bodies * 3 - 1));
        }
        if ((threadIdx.x & 15) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(S.episode_length_buf + i));
        // ... then the post-step's rank-independent inputs: in flight while the pre-step part runs
        asm volatile("prefetch.global.L2 [%0];" ::"l"(root_pos_w + 3 * (size_t)i));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(root_quat_w + 4 * (size_t)i));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(S.pos_cmd_w + 3 * (size_t)i));
        if (!kRng) asm volatile("prefetch.global.L2 [%0];" ::"l"(V.theta_u + (size_t)i * V.n_rounds));
        if ((threadIdx.x & 31) == 0) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(S.heading_cmd_w + i));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(S.time_left + i));
            if (!kRng) {
                asm volatile("prefetch.global.L2 [%0];" ::"l"(V.yaw_u + i));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(V.heading_u + i));
            }
            asm volatile("prefetch.global.L2 [%0];" ::"l"(S.err_pos + i));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(S.err_heading + i));
        }
    }
    // this launch may itself be a programmatic dependent of whatever produced the actions / root state / contacts: the
    // prefetches above carry no data, everything below reads what the predecessor wrote
    if constexpr (kRng) grid_dependency_wait();
    const RngKey key = load_rng_key<kRng>(V);  // (a cold miss: first consumed in the hook below, after the kinematics)
    SpawnEarly early;
    MDP_STAMP(1);
    const bool reset = pre_step_env<kSplit ? kPreState : kPreAll>(i, new_actions, force, n, P, S, O, pre_phases, [&]() {
        if constexpr (kRng && !kSplit) {
            if (i < n && (phases & ROVER_PHASE_SPAWN)) {  // (see SpawnEarly) consumed after the rest of the pre-step
                early.have = true;
                early.idx = (long long)spawn_perm_at(make_spawn_perm_key(key, (uint32_t)T.n_spawns), (uint32_t)i);
                const float* sp = T.spawn + 3 * (size_t)early.idx;
                early.x = __ldg(sp), early.y = __ldg(sp + 1), early.z = __ldg(sp + 2);
            }
        }
    }, [&](bool reset_now) {
        if constexpr (kSplit) {  // which envs reset -> the kinematics warps: they draw the new targets during the rewards
            sh.reset_flag[threadIdx.x] = reset_now ? 1 : 0;
            __threadfence_block();
            split_arrive<kBarResetFlags>();
        }
    });
    MDP_STAMP(2);
    if constexpr (kSplit) {  // the kinematics warps' handoff (long there by now)
        split_wait<kBarHandoff>();
        const int t = (int)threadIdx.x;
        early.have = (i < n) && (phases & ROVER_PHASE_SPAWN);
        early.idx = sh.hand_idx[t];
        early.x = sh.hand[0][t], early.y = sh.hand[1][t], early.z = sh.hand[2][t];
        early.have_variates = i < n;
        early.yaw_u = sh.hand[3][t], early.heading_u = sh.hand[4][t];
    }
    if ((pre_phases & ROVER_PRE_TERMS) && threadIdx.x == 0) O.block_reset_counts[bid] = 0;  // unused by this path
    post_step_block<true, kRng, kSplit>(sh, bid, n_blocks, reset, root_pos_w, root_quat_w, n, P, S, O, T, V, out_spawn_index, block_stats,
                                done_counter, stats, log_out, obs, obs_stride, phases, X, lookback, epoch, key, early);
}

// one block: thread (p, k) = (threadIdx.x / 16, threadIdx.x % 16) reads statistic k of rank p's slot consistently
__global__ void stats_read_kernel(const unsigned char* __restrict__ mailbox, int world, double* __restrict__ out) {
    __shared__ double v[64][kStats];
    const int p = threadIdx.x / kStats, k = threadIdx.x % kStats;
    for (int p0 = 0; p0 < world; p0 += 64) {
        const int pp = p0 + p;
        if (pp < world && p < 64) {
            const unsigned char* slot = mailbox + (size_t)pp * ROVER_MAILBOX_SLOT_BYTES;
            const volatile unsigned long long* sq = reinterpret_cast<const volatile unsigned long long*>(slot);
            const volatile double* val = reinterpret_cast<const volatile double*>(slot + 8);
            double x;
            unsigned long long s1, s2;
            do {  // buffer s1 & 1 holds the totals of sequence s1; it is rewritten only on the way to s1 + 2
                s1 = *sq;
                __threadfence_system();
                x = val[(s1 & 1ull) * kStats + k];
                __threadfence_system();
                s2 = *sq;
            } while (s1 != s2);
            v[p][k] = x;
        }
        __syncthreads();
        if (threadIdx.x < kStats) {
            double t = p0 == 0 ? 0.0 : out[threadIdx.x];
            for (int q = 0; q < min(64, world - p0); ++q) t += v[q][threadIdx.x];
            out[threadIdx.x] = t;
        }
        __syncthreads();
    }
}

}  // namespace rover

static int check_state(const RoverMdpState* s, const RoverMdpOut* o) {
    using namespace rover;
    ROVER_CHECK(s && o, "rover_mdp: NULL state/out struct");
    ROVER_CHECK(s->action && s->prev_action && s->pos_cmd_w && s->heading_cmd_w && s->pos_cmd_b && s->heading_cmd_b &&
                    s->time_left && s->command_counter && s->episode_length_buf && s->episode_sums && s->env_origins &&
                    s->err_pos && s->err_heading,
                "rover_mdp: NULL pointer in RoverMdpState");
    ROVER_CHECK(o->processed_actions && o->joint_pos && o->joint_vel && o->reward && o->term_rewards && o->terminated &&
                        o->truncated && o->term_flags && o->reset_flags && o->block_reset_counts && o->term_values,
                "rover_mdp: NULL pointer in RoverMdpOut");
    ROVER_CHECK((reinterpret_cast<uintptr_t>(o->joint_pos) & 15) == 0, "rover_mdp: joint_pos not 16B aligned");
    return 0;
}

extern "C" int rover_ackermann(const float* actions, int32_t n_envs, const RoverMdpParams* params, float* processed,
                               float* joint_pos, float* joint_vel, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_ackermann: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(actions && params && joint_pos && joint_vel, "rover_ackermann: NULL argument");
    ROVER_CHECK(params->action_variant >= 1 && params->action_variant <= 3, "rover_ackermann: action_variant must be 1, 2 or 3");
    ackermann_kernel<<<(n_envs + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(actions, n_envs, *params, processed,
                                                                                        joint_pos, joint_vel);
    return check_launch("ackermann_kernel");
}

extern "C" int rover_mdp_pre_step(const float* new_actions, const float* force_matrix_w, int32_t n_envs,
                                  const RoverMdpParams* params, const RoverMdpState* state, const RoverMdpOut* out,
                                  int32_t phases, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_mdp_pre_step: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(params && (new_actions || !(phases & ROVER_PRE_ACTIONS)) &&
                    (force_matrix_w || !(phases & ROVER_PRE_TERMS)),
                "rover_mdp_pre_step: NULL argument");
    ROVER_CHECK(params->num_bodies >= 0 && params->max_episode_length > 0, "rover_mdp_pre_step: bad params");
    if (int rc = check_state(state, out)) return rc;
    const int blocks = (n_envs + ROVER_MDP_BLOCK - 1) / ROVER_MDP_BLOCK;
    mdp_pre_step_kernel<<<blocks, ROVER_MDP_BLOCK, 0, static_cast<cudaStream_t>(stream)>>>(
        new_actions, force_matrix_w, n_envs, *params, *state, *out, phases);
    return check_launch("mdp_pre_step_kernel");
}

namespace rover {

static int make_variates(const RoverResetVariates* var, int n_envs, VariatesDev& V, const char* who) {
    ROVER_CHECK(var != nullptr, "%s: NULL RoverResetVariates", who);
    ROVER_CHECK(var->n_rounds >= 1 && var->n_rounds <= 4096, "%s: n_rounds must be in [1, 4096]", who);
    if (var->rng_state != nullptr) {
        V = VariatesDev{nullptr, nullptr, nullptr, nullptr, reinterpret_cast<unsigned long long*>(var->rng_state), var->n_rounds};
    } else {
        ROVER_CHECK(var->spawn_perm && var->yaw_u && var->heading_u && var->theta_u,
                    "%s: explicit variates need spawn_perm, yaw_u, heading_u and theta_u (or set rng_state)", who);
        V = VariatesDev{reinterpret_cast<const long long*>(var->spawn_perm), var->yaw_u, var->heading_u, var->theta_u, nullptr,
                        var->n_rounds};
    }
    (void)n_envs;
    return 0;
}

static int make_exchange(const RoverStatsExchange* xchg, StatsExchangeDev& X, const char* who) {
    X = StatsExchangeDev{nullptr, nullptr, nullptr, 0, 0};
    if (xchg != nullptr) {
        ROVER_CHECK(xchg->peer_mailbox && xchg->cumulative && xchg->sequence && xchg->world >= 1 && xchg->rank >= 0 &&
                        xchg->rank < xchg->world,
                    "%s: bad RoverStatsExchange", who);
        X = StatsExchangeDev{xchg->peer_mailbox, xchg->cumulative, reinterpret_cast<unsigned long long*>(xchg->sequence),
                             xchg->rank, xchg->world};
    }
    return 0;
}

static int check_post_args(const float* root_pos_w, const float* root_quat_w, int n_envs, const RoverMdpParams* params,
                           const RoverTerrainTables* tables, const float* stats, const float* scratch, const float* obs,
                           int obs_stride, int phases, const char* who) {
    ROVER_CHECK(root_pos_w && root_quat_w && params && tables && stats && scratch, "%s: NULL argument", who);
    ROVER_CHECK(tables->heightmap && tables->safe_mask && tables->spawn_table && tables->height > 0 &&
                    tables->width > 0 && tables->n_spawns > 0 && tables->resolution > 0.f,
                "%s: bad terrain tables", who);
    // without-replacement spawn draw: reset rank j < n_envs indexes a permutation of the table's rows
    ROVER_CHECK(!(phases & ROVER_PHASE_SPAWN) || tables->n_spawns >= n_envs,
                "%s: spawn table has %d rows for %d envs (randperm(len(spawn))[:K] needs K <= len)", who, tables->n_spawns,
                n_envs);
    // a reset resample and a time-based resample of one env share the env's variates; they never meet in one step as
    // long as a fresh command outlives the step (reference: 150 s against 0.2 s)
    ROVER_CHECK(params->resampling_time > params->step_dt, "%s: resampling_time must exceed step_dt", who);
    ROVER_CHECK((reinterpret_cast<uintptr_t>(root_quat_w) & 15) == 0, "%s: root_quat_w not 16B aligned", who);
    ROVER_CHECK(obs == nullptr || obs_stride >= 4, "%s: obs_stride < 4", who);
    return 0;
}

}  // namespace rover

extern "C" int rover_mdp_post_step(float* root_pos_w, float* root_quat_w, int32_t n_envs, const RoverMdpParams* params,
                                   const RoverMdpState* state, const RoverMdpOut* out,
                                   const RoverTerrainTables* tables, const int64_t* spawn_perm, const float* yaw_u,
                                   const float* heading_u, const float* theta_u, int32_t n_rounds,
                                   int64_t* out_spawn_index, float* stats, float* scratch, float* obs,
                                   int32_t obs_stride, int32_t phases, void* stream) {
    return rover_mdp_post_step_x(root_pos_w, root_quat_w, n_envs, params, state, out, tables, spawn_perm, yaw_u, heading_u,
                                 theta_u, n_rounds, out_spawn_index, stats, scratch, obs, obs_stride, phases, nullptr,
                                 stream);
}

extern "C" int rover_mdp_post_step_x(float* root_pos_w, float* root_quat_w, int32_t n_envs, const RoverMdpParams* params,
                                     const RoverMdpState* state, const RoverMdpOut* out,
                                     const RoverTerrainTables* tables, const int64_t* spawn_perm, const float* yaw_u,
                                     const float* heading_u, const float* theta_u, int32_t n_rounds,
                                     int64_t* out_spawn_index, float* stats, float* scratch, float* obs,
                                     int32_t obs_stride, int32_t phases, const RoverStatsExchange* xchg, void* stream) {
    const RoverResetVariates var{spawn_perm, yaw_u, heading_u, theta_u, n_rounds, 0, nullptr};
    return rover_mdp_post_step_v3(root_pos_w, root_quat_w, n_envs, params, state, out, tables, &var, out_spawn_index, stats,
                                  scratch, nullptr, obs, obs_stride, phases, xchg, stream);
}

extern "C" int rover_mdp_post_step_v3(float* root_pos_w, float* root_quat_w, int32_t n_envs, const RoverMdpParams* params,
                                      const RoverMdpState* state, const RoverMdpOut* out,
                                      const RoverTerrainTables* tables, const RoverResetVariates* variates,
                                      int64_t* out_spawn_index, float* stats, float* scratch, float* log_out, float* obs,
                                      int32_t obs_stride, int32_t phases, const RoverStatsExchange* xchg, void* stream) {
    using namespace rover;
    StatsExchangeDev X;
    if (int rc = make_exchange(xchg, X, "rover_mdp_post_step")) return rc;
    ROVER_CHECK(n_envs >= 0, "rover_mdp_post_step: negative n_envs");
    if (n_envs == 0) return 0;
    if (int rc = check_post_args(root_pos_w, root_quat_w, n_envs, params, tables, stats, scratch, obs, obs_stride, phases,
                                 "rover_mdp_post_step"))
        return rc;
    VariatesDev V;
    if (int rc = make_variates(variates, n_envs, V, "rover_mdp_post_step")) return rc;
    if (int rc = check_state(state, out)) return rc;
    Tables T{tables->heightmap, tables->safe_mask, tables->height,   tables->width,   tables->offset_x,
             tables->offset_y,  tables->resolution, tables->spawn_table, tables->n_spawns};
    const int blocks = (n_envs + ROVER_MDP_BLOCK - 1) / ROVER_MDP_BLOCK;
    // scratch layout: [blocks * 16] block partials, then one uint32 completion counter (zero-initialised by caller)
    float* block_stats = scratch;
    unsigned int* counter = reinterpret_cast<unsigned int*>(scratch + (size_t)blocks * ROVER_STATS_LEN);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (V.rng != nullptr)
        mdp_post_step_kernel<true><<<blocks, ROVER_MDP_BLOCK, 0, st>>>(
            root_pos_w, root_quat_w, n_envs, *params, *state, *out, T, V, reinterpret_cast<long long*>(out_spawn_index),
            block_stats, counter, stats, log_out, obs, obs_stride, phases, X);
    else
        mdp_post_step_kernel<false><<<blocks, ROVER_MDP_BLOCK, 0, st>>>(
            root_pos_w, root_quat_w, n_envs, *params, *state, *out, T, V, reinterpret_cast<long long*>(out_spawn_index),
            block_stats, counter, stats, log_out, obs, obs_stride, phases, X);
    return check_launch("mdp_post_step_kernel");
}

extern "C" int rover_mdp_step(const float* new_actions, const float* force_matrix_w, float* root_pos_w, float* root_quat_w,
                              int32_t n_envs, const RoverMdpParams* params, const RoverMdpState* state,
                              const RoverMdpOut* out, const RoverTerrainTables* tables, const int64_t* spawn_perm,
                              const float* yaw_u, const float* heading_u, const float* theta_u, int32_t n_rounds,
                              int64_t* out_spawn_index, float* stats, float* scratch, uint64_t* lookback, float* obs,
                              int32_t obs_stride, int32_t pre_phases, int32_t phases, const RoverStatsExchange* xchg,
                              void* stream) {
    const RoverResetVariates var{spawn_perm, yaw_u, heading_u, theta_u, n_rounds, 0, nullptr};
    return rover_mdp_step_v3(new_actions, force_matrix_w, root_pos_w, root_quat_w, n_envs, params, state, out, tables, &var,
                             out_spawn_index, stats, scratch, lookback, nullptr, obs, obs_stride, pre_phases, phases, xchg,
                             stream);
}

extern "C" int rover_mdp_step_v3(const float* new_actions, const float* force_matrix_w, float* root_pos_w,
                                 float* root_quat_w, int32_t n_envs, const RoverMdpParams* params,
                                 const RoverMdpState* state, const RoverMdpOut* out, const RoverTerrainTables* tables,
                                 const RoverResetVariates* variates, int64_t* out_spawn_index, float* stats, float* scratch,
                                 uint64_t* lookback, float* log_out, float* obs, int32_t obs_stride, int32_t pre_phases,
                                 int32_t phases, const RoverStatsExchange* xchg, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_mdp_step: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(params && (new_actions || !(pre_phases & ROVER_PRE_ACTIONS)) &&
                    (force_matrix_w || !(pre_phases & ROVER_PRE_TERMS)) && variates &&
                    (lookback || variates->rng_state),
                "rover_mdp_step: NULL argument (lookback is needed with explicit variates)");
    ROVER_CHECK(params->num_bodies >= 0 && params->max_episode_length > 0, "rover_mdp_step: bad params");
    if (int rc = check_post_args(root_pos_w, root_quat_w, n_envs, params, tables, stats, scratch, obs, obs_stride, phases,
                                 "rover_mdp_step"))
        return rc;
    VariatesDev V;
    if (int rc = make_variates(variates, n_envs, V, "rover_mdp_step")) return rc;
    if (int rc = check_state(state, out)) return rc;
    StatsExchangeDev X;
    if (int rc = make_exchange(xchg, X, "rover_mdp_step")) return rc;
    Tables T{tables->heightmap, tables->safe_mask, tables->height,   tables->width,   tables->offset_x,
             tables->offset_y,  tables->resolution, tables->spawn_table, tables->n_spawns};
    const int blocks = (n_envs + ROVER_MDP_BLOCK - 1) / ROVER_MDP_BLOCK;
    float* block_stats = scratch;
    unsigned int* counter = reinterpret_cast<unsigned int*>(scratch + (size_t)blocks * ROVER_STATS_LEN);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // ROVER_MDP_SPLIT=0: the in-kernel-variates step without the kinematics warps (A/B timing, profiles/r02_step.md)
    static const bool split = !(std::getenv("ROVER_MDP_SPLIT") && std::getenv("ROVER_MDP_SPLIT")[0] == '0');
    if (V.rng != nullptr && split)
        ROVER_CUDA(launch_overlapped(mdp_fused_step_kernel<true, true>, dim3(blocks), dim3(2 * ROVER_MDP_BLOCK), 0, st, new_actions,
                                     force_matrix_w, root_pos_w, root_quat_w, (int)n_envs, *params, *state, *out, T, V,
                                     reinterpret_cast<long long*>(out_spawn_index), block_stats, counter, stats, log_out, obs,
                                     (int)obs_stride, (int)pre_phases, (int)phases, X,
                                     reinterpret_cast<unsigned long long*>(lookback)));
    else if (V.rng != nullptr)
        ROVER_CUDA(launch_overlapped(mdp_fused_step_kernel<true>, dim3(blocks), dim3(ROVER_MDP_BLOCK), 0, st, new_actions,
                                     force_matrix_w, root_pos_w, root_quat_w, (int)n_envs, *params, *state, *out, T, V,
                                     reinterpret_cast<long long*>(out_spawn_index), block_stats, counter, stats, log_out, obs,
                                     (int)obs_stride, (int)pre_phases, (int)phases, X,
                                     reinterpret_cast<unsigned long long*>(lookback)));
    else
        ROVER_CUDA(launch_overlapped(mdp_fused_step_kernel<false>, dim3(blocks), dim3(ROVER_MDP_BLOCK), 0, st, new_actions,
                                     force_matrix_w, root_pos_w, root_quat_w, (int)n_envs, *params, *state, *out, T, V,
                                     reinterpret_cast<long long*>(out_spawn_index), block_stats, counter, stats, log_out, obs,
                                     (int)obs_stride, (int)pre_phases, (int)phases, X,
                                     reinterpret_cast<unsigned long long*>(lookback)));
    return check_launch("mdp_fused_step_kernel");
}

// The variates the kernels generate in registers, evaluated on the HOST by the same functions (rng.cuh): the oracle is
// fed these, the kernel generates its own, and the two must agree bit for bit (tests/test_gpu_rng.py).
extern "C" int rover_rng_variates(uint64_t seed, uint64_t step, int32_t n_envs, int32_t n_rounds, int32_t n_spawns,
                                  int64_t* spawn_by_env, float* yaw_u, float* heading_u, float* theta_u) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0 && n_rounds >= 1 && n_spawns >= 1, "rover_rng_variates: bad sizes");
    const RngKey key = make_rng_key(seed, step);
    if (spawn_by_env != nullptr) {
        const SpawnPermKey pk = make_spawn_perm_key(key, (uint32_t)n_spawns);
        const int k = n_envs < n_spawns ? n_envs : n_spawns;
        for (int i = 0; i < k; ++i) spawn_by_env[i] = (int64_t)spawn_perm_at(pk, (uint32_t)i);
    }
    for (int i = 0; i < n_envs; ++i) {
        uint32_t w[4];
        rng_env_stream(key, (uint32_t)i, 0u, w);
        if (yaw_u) yaw_u[i] = u01(w[0]);
        if (heading_u) heading_u[i] = u01(w[1]);
        if (theta_u) {
            for (int r0 = 0; r0 < n_rounds; r0 += 4) {
                rng_env_stream(key, (uint32_t)i, 1u + (uint32_t)(r0 / 4), w);
                for (int k = 0; k < 4 && r0 + k < n_rounds; ++k) theta_u[(size_t)i * n_rounds + r0 + k] = u01(w[k]);
            }
        }
    }
    return 0;
}

extern "C" int rover_philox4x32_10(const uint32_t counter[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t o[4];
    rover::philox4x32_10(counter[0], counter[1], counter[2], counter[3], key[0], key[1], o);
    for (int k = 0; k < 4; ++k) out[k] = o[k];
    return 0;
}

// The step's three functions that are not correctly rounded (atan2f, sinf, cosf), evaluated elementwise by the device code
// the step kernels run (this translation unit's flags and libdevice): an fp32 model of the step takes them from here.
__global__ void mdp_math_kernel(int op, const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                                int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float x = a[i];
    out[i] = op == ROVER_MDP_MATH_ATAN2 ? atan2f(x, b[i]) : (op == ROVER_MDP_MATH_SIN ? sinf(x) : cosf(x));
}

extern "C" int rover_mdp_math(int32_t op, const float* a, const float* b, float* out, int32_t n, void* stream) {
    using namespace rover;
    ROVER_CHECK(op == ROVER_MDP_MATH_ATAN2 || op == ROVER_MDP_MATH_SIN || op == ROVER_MDP_MATH_COS,
                "rover_mdp_math: op must be ROVER_MDP_MATH_ATAN2, _SIN or _COS");
    ROVER_CHECK(n >= 0, "rover_mdp_math: negative n");
    if (n == 0) return 0;
    ROVER_CHECK(a && out && (b || op != ROVER_MDP_MATH_ATAN2), "rover_mdp_math: NULL argument");
    mdp_math_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(op, a, b, out, n);
    return check_launch("mdp_math_kernel");
}

__global__ void __launch_bounds__(ROVER_MDP_BLOCK) stats_publish_kernel(const __grid_constant__ rover::StatsExchangeDev X) {
    __shared__ rover::MdpShared sh;
    const int tid = (int)threadIdx.x;
    rover::publish_totals<1>(tid, tid < rover::kStats ? X.cumulative[tid] : 0.0, sh, X);
}

extern "C" int rover_stats_publish(const RoverStatsExchange* xchg, void* stream) {
    using namespace rover;
    StatsExchangeDev X;
    if (int rc = make_exchange(xchg, X, "rover_stats_publish")) return rc;
    ROVER_CHECK(X.world > 0, "rover_stats_publish: xchg is NULL");
    stats_publish_kernel<<<1, ROVER_MDP_BLOCK, 0, static_cast<cudaStream_t>(stream)>>>(X);
    return check_launch("stats_publish_kernel");
}

extern "C" int rover_stats_read(const void* mailbox_local, int32_t world, double* out, void* stream) {
    using namespace rover;
    ROVER_CHECK(mailbox_local && out && world >= 1, "rover_stats_read: bad arguments");
    stats_read_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const unsigned char*>(mailbox_local), world,
                                                                        out);
    return check_launch("stats_read_kernel");
}

extern "C" int rover_p2p_alloc(void** out_ptr, int64_t bytes) {
    using namespace rover;
    ROVER_CHECK(out_ptr && bytes > 0, "rover_p2p_alloc: bad arguments");
    ROVER_CUDA(cudaMalloc(out_ptr, (size_t)bytes));
    ROVER_CUDA(cudaMemset(*out_ptr, 0, (size_t)bytes));
    ROVER_CUDA(cudaDeviceSynchronize());
    return 0;
}
extern "C" int rover_p2p_free(void* ptr) {
    using namespace rover;
    ROVER_CUDA(cudaFree(ptr));
    return 0;
}
extern "C" int rover_p2p_export(void* ptr, uint8_t handle_out[64]) {
    using namespace rover;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    ROVER_CUDA(cudaIpcGetMemHandle(&h, ptr));
    memcpy(handle_out, &h, 64);
    return 0;
}
extern "C" int rover_p2p_open(const uint8_t handle[64], void** out_ptr) {
    using namespace rover;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    ROVER_CUDA(cudaIpcOpenMemHandle(out_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}
extern "C" int rover_p2p_close(void* ptr) {
    using namespace rover;
    ROVER_CUDA(cudaIpcCloseMemHandle(ptr));
    return 0;
}

#if ROVER_MDP_DBG
extern "C" int rover_debug_mdp_timeline(unsigned long long* host_dst) {
    return (int)cudaMemcpyFromSymbol(host_dst, rover::g_mdp_dbg, sizeof(rover::g_mdp_dbg));
}
#endif
