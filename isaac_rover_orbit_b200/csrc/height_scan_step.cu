// The whole non-physics step in ONE launch: the fused MDP step runs INSIDE the persistent height-scan kernel.
//
// Replaces, per environment step (reference root relative; the same lines as rover_mdp_step_v3 + rover_height_scan):
//   rover_envs/envs/navigation/entrypoints/rover_env.py:61-102    everything RoverEnv.step does outside PhysX
//   rover_envs/mdp/actions/ackermann_actions.py:226-322            .../mdp/rewards.py:14-137   .../mdp/terminations.py:14-64
//   .../mdp/randomizations.py:12-39   .../utils/terrains/terrain_importer.py:74-175   .../mdp/observations.py:15-45
// Why: at 16384 envs the step was two launches, 24 us (MDP: once-through code, three dependent cold misses, 10 % issue
// active -- profiles/r02_ncu_full.md) + 55 us (scan), strictly one after the other, although only the ~5 % of envs that
// reset change the pose the scan reads.  With the reset variates drawn in the kernel the MDP work of an env depends on
// nothing but that env (no reset rank), so any thread can do it: here warps of every scan CTA run it for the CTA's own
// envs, 32 at a time, ahead of the scan; an env's final pose is handed to the scan's producer warp through
// shared memory as soon as it is known (right after the spawn, before the target rejection sampling and the stores).
// The MDP step's latency chain hides behind the scan of the previous batch; only the first batch's (~4 us) is exposed.
//
// One MDP warp per CTA is not enough: a batch of 32 envs is ~2800 dependent instructions + 3 cold misses, ~25 us in a
// single warp, against the ~14 us the scan needs for 32 envs (first version: 104 us per step against 81 us for the two
// launches).  So warps 1-4 are MDP warps: batch b goes to warp 1 + b % 4, each with its own pose buffer, and an MDP warp
// that is ahead of the scan front JOINS THE SCAN CONSUMERS (work units come from a shared counter) until its next batch
// is due.  Roles: warp 0 scan producer (variant 5's, poses from shared memory), warps 1-15 workers.  Statistics: per-warp
// partials (batches in order, fixed shuffle tree) -> CTA partial -> combined in CTA order by the last CTA, which also
// writes the episode log, advances the variate step and publishes to the P2P mailboxes.
#include "mdp_env.cuh"
#include "scan_paired.cuh"

namespace rover {

constexpr int kStepWorkerWarps = 15;  // warps 1..15: scan consumers; the first kStepMdpWarps of them run the MDP step first
constexpr int kStepMdpWarps = 4;      // batches of 32 envs are dealt to them round-robin (batch b -> worker b % 4)
constexpr int kStepThreads = 32 * (1 + kStepWorkerWarps);
constexpr int kStepLead = 96;         // an MDP batch is started when the scan front is within this many envs of it
static_assert(kStepThreads == 512, "16 warps x 128 registers = the register file");
static_assert(kPairFullBars >= kStepWorkerWarps + kPairStages, "full barriers: phase-aliasing note in scan_paired.cuh");

struct StepSmem {
    PairStage stage[kPairStages];
    float vx[kPairMaxRays], vy[kPairMaxRays], vz[kPairMaxRays];
    LinePair2 xpair[kPairMaxLines], ypair[kPairMaxLines];
    unsigned long long full_bar[kPairFullBars];
    unsigned long long empty_bar[kPairStages];
    unsigned long long pose_full[kStepMdpWarps], pose_empty[kStepMdpWarps];
    float pose[kStepMdpWarps][32][8];  // final root pose of a batch of 32 envs: px, py, pz, qw, qx, qy, qz, -
    float part[kStepMdpWarps][ROVER_STATS_LEN];  // statistics partials of the MDP warps
    int next_chunk;
    int mdp_done;
};
static_assert(sizeof(StepSmem) <= 227 * 1024, "StepSmem exceeds the shared memory of one SM");
__device__ __forceinline__ float sm_vz(const StepSmem& sm, int slot) { return sm.vz[slot]; }

struct PoseToScan {
    float* slot;               // this lane's row of the batch's pose buffer
    unsigned long long* full;  // the buffer's `pose_full` barrier (32 arrivals)
    unsigned long long* empty; // ... and `pose_empty` (the producer took the previous batch that used the buffer)
    int wait_parity;           // < 0: first use of the buffer, nothing to wait for
    __device__ __forceinline__ void operator()(float px, float py, float pz, const float4& q) const {
        if (wait_parity >= 0) bar_wait(empty, (uint32_t)wait_parity);
        slot[0] = px, slot[1] = py, slot[2] = pz;
        slot[3] = q.x, slot[4] = q.y, slot[5] = q.z, slot[6] = q.w;  // (w, x, y, z)
        bar_arrive(full);  // release: the producer may read this row
    }
};

__global__ void __launch_bounds__(kStepThreads, 1)
height_scan_step_kernel(const float* __restrict__ new_actions, const float* __restrict__ force,
                        float* __restrict__ root_pos_w, float* __restrict__ root_quat_w, int n_envs,
                        const __grid_constant__ RoverMdpParams P, const __grid_constant__ RoverMdpState S,
                        const __grid_constant__ RoverMdpOut O, const __grid_constant__ Tables T,
                        const __grid_constant__ VariatesDev V, long long* __restrict__ out_spawn_index,
                        float* __restrict__ cta_stats, unsigned int* __restrict__ done_counter, float* __restrict__ stats,
                        float* __restrict__ log_out, int pre_phases, int phases, const __grid_constant__ StatsExchangeDev X,
                        const float* __restrict__ ray_local, int n_rays, const __grid_constant__ ScanGridDev g,
                        const __grid_constant__ PlaneCellsDev pc, const __grid_constant__ CUtensorMap tmap,
                        float pattern_radius, float max_d, float base_offset, float* __restrict__ obs, int obs_stride) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    StepSmem& sm = *reinterpret_cast<StepSmem*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_iter = (n_envs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;  // envs of this CTA
    const int n_batches = (n_iter + 31) / 32;
    const int n_chunks = (n_rays + kPairChunk - 1) / kPairChunk;
    const bool lines_in_smem = (pc.nx <= kPairMaxLines) && (pc.ny <= kPairMaxLines);
    float* __restrict__ out = obs + 4;  // heights behind the observation head
    const int out_stride = obs_stride;

    // ---- prologue: barriers (warp 0), pattern + line tables (worker warps, loads before stores)
    int my_flat_z = 1;
    if (warp == 0) {
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap)) : "memory");
            for (int s = 0; s < kPairFullBars; ++s) bar_init(&sm.full_bar[s], 2);  // TMA bytes + header published
            for (int s = 0; s < kPairStages; ++s) bar_init(&sm.empty_bar[s], (uint32_t)n_chunks);
            for (int s = 0; s < kStepMdpWarps; ++s) {
                bar_init(&sm.pose_full[s], 32);  // one arrival per lane of the MDP warp
                bar_init(&sm.pose_empty[s], 1);  // the producer has read the batch
            }
            sm.next_chunk = 0;
            sm.mdp_done = 0;
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    } else {
        constexpr int kFill = 32 * kStepWorkerWarps;
        constexpr int kPatLoads = (3 * kPairMaxRays + kFill - 1) / kFill;
        constexpr int kLineLoads = (kPairMaxLines + kFill - 1) / kFill;
        const int ct = threadIdx.x - 32;
        float* pat_flat = sm.vx;  // vx, vy, vz contiguous
        float pat[kPatLoads], xl[kLineLoads], xh[kLineLoads], yl[kLineLoads], yh[kLineLoads];
        const float vz0 = __ldg(ray_local + 2);
#pragma unroll
        for (int k = 0; k < kPatLoads; ++k) {
            const int i = ct + k * kFill;
            const int comp = i / kPairMaxRays, r = ray_of_slot(i - comp * kPairMaxRays);
            pat[k] = (i < 3 * kPairMaxRays && r < n_rays) ? __ldg(ray_local + 3 * r + comp) : 0.f;
            if (comp == 2 && r < n_rays && pat[k] != vz0) my_flat_z = 0;
        }
#pragma unroll
        for (int k = 0; k < kLineLoads; ++k) {
            const int i = ct + k * kFill;
            const bool okx = lines_in_smem && i < pc.nx, oky = lines_in_smem && i < pc.ny;
            xl[k] = okx ? __ldg(pc.xs + i) : 0.f;
            xh[k] = okx ? __ldg(pc.xs + i + 1) : 0.f;
            yl[k] = oky ? __ldg(pc.ys + i) : 0.f;
            yh[k] = oky ? __ldg(pc.ys + i + 1) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < kPatLoads; ++k) {
            const int i = ct + k * kFill;
            if (i < 3 * kPairMaxRays) pat_flat[i] = pat[k];
        }
#pragma unroll
        for (int k = 0; k < kLineLoads; ++k) {
            const int i = ct + k * kFill;
            if (lines_in_smem && i < pc.nx) sm.xpair[i] = {xl[k], xh[k]};
            if (lines_in_smem && i < pc.ny) sm.ypair[i] = {yl[k], yh[k]};
        }
    }
    const bool flat_z = __syncthreads_and(my_flat_z) != 0;

    if (warp == 0) {
        // =============================== scan producer: variant 5's, poses from the MDP warps ===============================
        ProducerEnv cur;
        for (int b = 0; b < n_batches; ++b) {
            const int base = b * 32, pb = b % kStepMdpWarps;
            bar_wait(&sm.pose_full[pb], (uint32_t)(b / kStepMdpWarps) & 1u);
            {
                const float* row = &sm.pose[pb][lane][0];
                cur.have = base + lane < n_iter;
#pragma unroll
                for (int k = 0; k < 3; ++k) cur.pv[k] = cur.have ? row[k] : 0.f;
#pragma unroll
                for (int k = 0; k < 4; ++k) cur.qv[k] = cur.have ? row[3 + k] : (k == 0 ? 1.f : 0.f);
                cur.px = cur.pv[0], cur.py = cur.pv[1], cur.pz = cur.pv[2];
            }
            __syncwarp();
            if (lane == 0) bar_arrive(&sm.pose_empty[pb]);
            producer_window(cur, pc, pattern_radius);
            producer_frame(cur);
            producer_verdict(cur, sm, pc, pattern_radius, lines_in_smem);
            const int n_here = min(32, n_iter - base);
            for (int k = 0; k < n_here; ++k) {
                if (lane == k) {
                    const int it = base + k;
                    const int s = it % kPairStages;
                    unsigned long long* full = &sm.full_bar[it % kPairFullBars];
                    PairStage& st = sm.stage[s];
                    if (it >= kPairStages) bar_wait(&sm.empty_bar[s], ((uint32_t)(it / kPairStages) & 1u) ^ 1u);  // stage drained
                    if (cur.ok) {
                        bar_arrive_expect_tx(full, kPairStageBytes);
                        tma_load_window_planar(st.p, &tmap, cur.ic0, cur.jr0, full);
                    } else {
                        bar_arrive(full);
                    }
                    st.hdr = {cur.cw, cur.sz, cur.px, cur.py, cur.pz, cur.ic0, cur.jr0, cur.ncols, cur.nrows, cur.ok ? 1 : 0, 0, 0};
                    bar_arrive(full);  // header published (release)
                }
                __syncwarp();  // environments are issued strictly in order (phase-aliasing argument of variant 5)
            }
        }
    } else {
        // =============================== workers: scan consumers; workers 0..3 run the MDP step of their batches first =========
        // Work units of the scan are handed out in order from a shared counter (so that an MDP warp can join and leave the
        // pool); an MDP warp starts its next batch when the scan front comes within kStepLead envs of it, and in any case
        // before it touches a chunk of an env at or behind that batch (its own pending batch can never be what it waits for).
        const int w = warp - 1;
        const bool mdp_warp = w < kStepMdpWarps;
        const int n_mdp_active = min(kStepMdpWarps, n_batches);
        int my_next = mdp_warp ? w : n_batches;  // next batch this warp owes
        RngKey key = make_rng_key(0ull, 0ull);
        if (mdp_warp) key = make_rng_key(V.rng[0], *reinterpret_cast<volatile unsigned long long*>(V.rng + 1));
        float acc = 0.f;  // lane k < 16 accumulates statistic k over this warp's batches (in order)
        bool have_chunk = false, draining = false;
        int it = 0, c = 0;
        while (true) {
            bool run_mdp = false;
            if (my_next < n_batches) {
                if (draining) run_mdp = true;
                else if (have_chunk) run_mdp = my_next <= it / 32 + 1;
                else run_mdp = my_next * 32 <= *reinterpret_cast<volatile int*>(&sm.next_chunk) / n_chunks + kStepLead;
            }
            if (run_mdp) {
                // ------------------------------------------------ the MDP step of batch my_next: one env per lane
                const int b = my_next;
                const int eit = b * 32 + lane;
                const bool valid = eit < n_iter;
                const int i = valid ? (int)blockIdx.x + eit * (int)gridDim.x : n_envs;  // (n_envs: skipped by the i < n guards)
                if (valid) {  // the post-step's inputs: in flight while the pre-step part runs
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(root_pos_w + 3 * (size_t)i));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(root_quat_w + 4 * (size_t)i));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(S.pos_cmd_w + 3 * (size_t)i));
                }
                const bool reset = pre_step_env(i, new_actions, force, n_envs, P, S, O, pre_phases);
                EnvRegs er;
                post_env_load<true>(i, valid, root_pos_w, root_quat_w, S, V, er);
                float st[kStats];
                const int use = b / kStepMdpWarps;  // w owns pose buffer w: use 0, 1, 2, ...
                const PoseToScan hook{&sm.pose[w][lane][0], &sm.pose_full[w], &sm.pose_empty[w], use > 0 ? ((use - 1) & 1) : -1};
                if (!valid) hook(0.f, 0.f, 0.f, make_float4(1.f, 0.f, 0.f, 0.f));  // a lane without an env still arrives
                post_env_work<true>(i, valid, valid && reset, 0, er, root_pos_w, root_quat_w, P, S, O, T, V, key, out_spawn_index,
                                    obs, obs_stride, phases, st, hook);
                // the batch's statistics: fixed shuffle tree, then lane k keeps statistic k
#pragma unroll
                for (int k = 0; k < kStats; ++k) {
                    float v = st[k];
                    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
                    v = __shfl_sync(0xffffffffu, v, 0);
                    if (lane == k) acc += v;
                }
                my_next += kStepMdpWarps;
                if (my_next >= n_batches) {
                    // ---- this warp's MDP work is done: its partial -> shared; the last MDP warp of the CTA combines them
                    //      (fixed order) -> global; the last CTA combines the CTA partials in CTA order (deterministic),
                    //      writes the log, advances the variate step and publishes to the other ranks' mailboxes
                    if (lane < kStats) sm.part[w][lane] = acc;
                    __threadfence_block();
                    __syncwarp();
                    int done = 0;
                    if (lane == 0) done = atomicAdd(&sm.mdp_done, 1);
                    done = __shfl_sync(0xffffffffu, done, 0);
                    if (done == n_mdp_active - 1) {
                        __threadfence_block();
                        float cta = 0.f;
                        if (lane < kStats)
                            for (int q = 0; q < n_mdp_active; ++q) cta += *reinterpret_cast<volatile float*>(&sm.part[q][lane]);
                        if (lane < kStats) cta_stats[(size_t)blockIdx.x * kStats + lane] = cta;
                        __threadfence();
                        __syncwarp();
                        unsigned ticket = 0;
                        if (lane == 0) ticket = atomicAdd(done_counter, 1u);
                        ticket = __shfl_sync(0xffffffffu, ticket, 0);
                        if (ticket == gridDim.x - 1u) {
                            __threadfence();
                            float t = 0.f;
                            if (lane < kStats)
                                for (unsigned cc = 0; cc < gridDim.x; ++cc) t += __ldcg(cta_stats + (size_t)cc * kStats + lane);
                            const float cnt = __shfl_sync(0xffffffffu, t, 13);
                            double total = 0.0;
                            if (lane < kStats) {
                                stats[lane] += t;
                                if (log_out != nullptr && (phases & ROVER_PHASE_MANAGERS) && cnt > 0.f) {  // ORBIT manager.reset() log
                                    float v = t;
                                    if (lane < ROVER_NUM_REWARD_TERMS) v = __fdiv_rn(__fdiv_rn(t, cnt), P.episode_length_s);
                                    else if (lane == 11 || lane == 12) v = __fdiv_rn(t, cnt);
                                    log_out[lane] = v;
                                }
                                if (X.world > 0) {
                                    total = X.cumulative[lane] + (double)t;
                                    X.cumulative[lane] = total;
                                }
                            }
                            if (lane == 0) {
                                *done_counter = 0u;          // re-arm for the next launch
                                V.rng[1] = V.rng[1] + 1ull;  // next launch = next step of the variate streams
                            }
                            if (X.world > 0) {  // P2P mailboxes: values into the idle buffer of every slot, one fence, then the sequence
                                const unsigned long long seq = *X.sequence + 1ull;
                                for (int e0 = 0; e0 < X.world * kStats; e0 += 32) {
                                    const int e = e0 + lane;
                                    const double v = __shfl_sync(0xffffffffu, total, e % kStats);
                                    if (e < X.world * kStats) {
                                        unsigned char* slot = static_cast<unsigned char*>(X.peer_mailbox[e / kStats]) +
                                                              (size_t)X.rank * ROVER_MAILBOX_SLOT_BYTES;
                                        reinterpret_cast<volatile double*>(slot + 8)[(seq & 1ull) * kStats + (e % kStats)] = v;
                                    }
                                }
                                __threadfence_system();
                                __syncwarp();
                                for (int p = lane; p < X.world; p += 32) {
                                    unsigned char* slot = static_cast<unsigned char*>(X.peer_mailbox[p]) + (size_t)X.rank * ROVER_MAILBOX_SLOT_BYTES;
                                    *reinterpret_cast<volatile unsigned long long*>(slot) = seq;
                                }
                                __syncwarp();
                                if (lane == 0) *X.sequence = seq;
                            }
                        }
                    }
                }
                continue;
            }
            if (draining) break;
            if (!have_chunk) {
                int k = 0;
                if (lane == 0) k = atomicAdd(&sm.next_chunk, 1);
                k = __shfl_sync(0xffffffffu, k, 0);
                it = k / n_chunks;
                c = k - it * n_chunks;
                if (it >= n_iter) {  // the scan is handed out; an MDP batch still owed (cannot be needed any more) is run, then out
                    draining = true;
                    continue;
                }
                have_chunk = true;
                continue;  // re-check the MDP duty against the env just drawn
            }
            have_chunk = false;
            // ------------------------------------------------ one 256-ray chunk of env `it` (variant 5's consumer body)
            const int env = (int)blockIdx.x + it * (int)gridDim.x;
            const int s = it % kPairStages;
            const PairStage& st = sm.stage[s];
            bar_wait(&sm.full_bar[it % kPairFullBars], (uint32_t)(it / kPairFullBars) & 1u);
            const PairHeader h = st.hdr;
            float* __restrict__ out_row = out + (size_t)env * out_stride;
            const int r_begin = c * kPairChunk, r_end = min(r_begin + kPairChunk, n_rays);
            if (h.mode == 1) {
                const float sz2 = __fmul_rn(h.sz, 2.f);
                const PairCtx cx = make_pair_ctx(h, sm, st, smem_raw, pc.inv_dx, pc.inv_dy, base_offset, max_d, sm.vz[0],
                                                 n_envs >> 31);
                for (int b0 = r_begin; b0 < r_end; b0 += kPairBatch) {
                    const int r = b0 + lane;  // rays r, r + 64 (slot 0) and r + 32, r + 96 (slot 1)
                    float* __restrict__ o = out_row + r;
                    unsigned defer;
                    if (flat_z && b0 + kPairBatch <= n_rays) {
                        defer = resolve_pair<true, true, false>(smem_raw, sm, cx, b0 + 2 * lane, r, n_rays, o, nullptr);
                        defer |= resolve_pair<true, true, false>(smem_raw, sm, cx, b0 + 64 + 2 * lane, r + 32, n_rays, o + 32, nullptr) << 2;
                    } else {
                        defer = resolve_pair<false, false, false>(smem_raw, sm, cx, b0 + 2 * lane, r, n_rays, o, nullptr);
                        defer |= resolve_pair<false, false, false>(smem_raw, sm, cx, b0 + 64 + 2 * lane, r + 32, n_rays, o + 32, nullptr) << 2;
                    }
                    if (defer != 0u) {  // rare: cell guess off by one, ray on the closed far border / outside, general cell
                        for (int u = 0; u < 4; ++u) {
                            if (!((defer >> u) & 1u)) continue;
                            const int rr = r + (u >> 1) * 32 + (u & 1) * 64;
                            const int sl = b0 + (u >> 1) * 64 + 2 * lane + (u & 1);
                            const float vx = sm.vx[sl], vy = sm.vy[sl];
                            const float tx = -__fmul_rn(sz2, vy), ty = __fmul_rn(sz2, vx);
                            const float X0 = __fadd_rn(__fadd_rn(__fadd_rn(vx, __fmul_rn(h.cw, tx)), -__fmul_rn(h.sz, ty)), h.px);
                            const float Y0 = __fadd_rn(__fadd_rn(__fadd_rn(vy, __fmul_rn(h.cw, ty)), __fmul_rn(h.sz, tx)), h.py);
                            pair_resolve_deferred_ray(&sm, &st, g, pc.inv_dx, pc.inv_dy, X0, Y0, __fadd_rn(sm.vz[sl], h.pz), h.pz,
                                                      max_d, base_offset, out_row + rr, nullptr);
                        }
                    }
                }
            } else {
                pair_resolve_chunk_from_global(&sm, lane, r_begin, r_end, h, g, pc, max_d, base_offset, out_row, nullptr);
            }
            __syncwarp();
            if (lane == 0) bar_arrive(&sm.empty_bar[s]);  // this chunk no longer reads the stage
        }
    }
}

int make_dev_grid(const RoverScanGrid* grid, ScanGridDev& g);  // height_scan.cu

}  // namespace rover

extern "C" int rover_step_fused(const float* new_actions, const float* force_matrix_w, float* root_pos_w, float* root_quat_w,
                                int32_t n_envs, const RoverMdpParams* params, const RoverMdpState* state,
                                const RoverMdpOut* out, const RoverTerrainTables* tables, uint64_t* rng_state,
                                int32_t n_rounds, int64_t* out_spawn_index, float* stats, float* scratch,
                                int32_t scratch_floats, float* log_out, float* obs, int32_t obs_stride, int32_t pre_phases,
                                int32_t phases, const RoverStatsExchange* xchg, const float* ray_starts_local, int32_t n_rays,
                                const float* pattern_box, const RoverScanGrid* grid, const RoverPlaneCells* cells,
                                float max_distance, float base_offset, void* stream) {
    using namespace rover;
    ROVER_CHECK(n_envs >= 0, "rover_step_fused: negative n_envs");
    if (n_envs == 0) return 0;
    ROVER_CHECK(params && state && out && tables && rng_state && stats && scratch && obs && root_pos_w && root_quat_w &&
                    ray_starts_local && pattern_box && grid && cells,
                "rover_step_fused: NULL argument");
    ROVER_CHECK((new_actions || !(pre_phases & ROVER_PRE_ACTIONS)) && (force_matrix_w || !(pre_phases & ROVER_PRE_TERMS)),
                "rover_step_fused: NULL actions / contact forces");
    ROVER_CHECK(params->num_bodies >= 0 && params->max_episode_length > 0 && n_rounds >= 1 && n_rounds <= 4096,
                "rover_step_fused: bad params");
    ROVER_CHECK(params->resampling_time > params->step_dt, "rover_step_fused: resampling_time must exceed step_dt");
    ROVER_CHECK(tables->heightmap && tables->safe_mask && tables->spawn_table && tables->height > 0 && tables->width > 0 &&
                    tables->n_spawns >= n_envs && tables->resolution > 0.f,
                "rover_step_fused: bad terrain tables (the spawn table needs >= n_envs rows)");
    ROVER_CHECK((reinterpret_cast<uintptr_t>(root_quat_w) & 15) == 0, "rover_step_fused: root_quat_w not 16B aligned");
    ROVER_CHECK(n_rays >= 1 && n_rays <= kPairMaxRays, "rover_step_fused: pattern of %d rays (1..%d supported)", n_rays, kPairMaxRays);
    ROVER_CHECK(obs_stride >= 4 + n_rays, "rover_step_fused: obs_stride %d < 4 + n_rays", obs_stride);
    ROVER_CHECK(cells->xs && cells->ys && cells->entries && cells->entries_planar && cells->nx > 0 && cells->ny > 0,
                "rover_step_fused: needs the plane-cell table with its planar copy");
    ROVER_CHECK(state->action && state->prev_action && state->pos_cmd_w && state->heading_cmd_w && state->pos_cmd_b &&
                    state->heading_cmd_b && state->time_left && state->command_counter && state->episode_length_buf &&
                    state->episode_sums && state->env_origins && state->err_pos && state->err_heading,
                "rover_step_fused: NULL pointer in RoverMdpState");
    ROVER_CHECK(out->processed_actions && out->joint_pos && out->joint_vel && out->reward && out->term_rewards &&
                    out->terminated && out->truncated && out->term_flags && out->reset_flags && out->term_values,
                "rover_step_fused: NULL pointer in RoverMdpOut");
    static int n_sms = 0;
    if (n_sms == 0) {
        int dev = 0;
        ROVER_CUDA(cudaGetDevice(&dev));
        ROVER_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
        ROVER_CUDA(cudaFuncSetAttribute(height_scan_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(StepSmem)));
    }
    const int grid_dim = n_envs < n_sms ? n_envs : n_sms;
    ROVER_CHECK(scratch_floats >= grid_dim * ROVER_STATS_LEN + 1, "rover_step_fused: scratch needs %d floats", grid_dim * ROVER_STATS_LEN + 1);
    StatsExchangeDev X{nullptr, nullptr, nullptr, 0, 0};
    if (xchg != nullptr) {
        ROVER_CHECK(xchg->peer_mailbox && xchg->cumulative && xchg->sequence && xchg->world >= 1 && xchg->rank >= 0 &&
                        xchg->rank < xchg->world,
                    "rover_step_fused: bad RoverStatsExchange");
        X = StatsExchangeDev{xchg->peer_mailbox, xchg->cumulative, reinterpret_cast<unsigned long long*>(xchg->sequence),
                             xchg->rank, xchg->world};
    }
    Tables T{tables->heightmap, tables->safe_mask, tables->height,   tables->width,   tables->offset_x,
             tables->offset_y,  tables->resolution, tables->spawn_table, tables->n_spawns};
    VariatesDev V{nullptr, nullptr, nullptr, nullptr, reinterpret_cast<unsigned long long*>(rng_state), n_rounds};
    ScanGridDev g;
    if (int rc = make_dev_grid(grid, g)) return rc;
    alignas(64) CUtensorMap tmap;
    if (const int rc = encode_planar_tensor_map(&tmap, cells, kPairPitch, kPairWin, "rover_step_fused")) return rc;
    PlaneCellsDev pc{cells->xs, cells->ys, reinterpret_cast<const float4*>(cells->entries), cells->nx, cells->ny,
                     cells->inv_dx, cells->inv_dy};
    const float rx = fmaxf(fabsf(pattern_box[0]), fabsf(pattern_box[1])), ry = fmaxf(fabsf(pattern_box[2]), fabsf(pattern_box[3]));
    const float radius = sqrtf(rx * rx + ry * ry) * 1.0001f + 1.0e-3f;
    // scratch: [grid_dim * 16] CTA partials, then one uint32 completion counter at the END of the buffer (zeroed once by the
    // caller, re-armed by the kernel; a buffer of its own -- not the block kernels' scratch)
    unsigned int* counter = reinterpret_cast<unsigned int*>(scratch + scratch_floats - 1);
    height_scan_step_kernel<<<grid_dim, kStepThreads, sizeof(StepSmem), static_cast<cudaStream_t>(stream)>>>(
        new_actions, force_matrix_w, root_pos_w, root_quat_w, n_envs, *params, *state, *out, T, V,
        reinterpret_cast<long long*>(out_spawn_index), scratch, counter, stats, log_out, pre_phases, phases, X,
        ray_starts_local, n_rays, g, pc, tmap, radius, max_distance, base_offset, obs, obs_stride);
    return check_launch("height_scan_step_kernel");
}
