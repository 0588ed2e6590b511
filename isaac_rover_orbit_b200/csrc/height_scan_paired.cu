// Persistent, warp-specialised plane-cell height scan with packed-fp32 ray pairs -- variant 5.
//
// Why (ncu on variant 4, profiles/r01_scan_v4*.md + r01_scan_v9 source page): the kernel is issue-bound, not HBM-bound.
//   * 13 % of the warp time was the serial table fill in the prologue (3 dependent cold misses per thread),
//   * 26 % was consumers waiting on the first windows (the producer started only after that prologue),
//   * 5 x 224 thread slots per 961-ray environment left 14 % of the lanes predicated off, the two 7-warp groups ended
//     up to one environment apart, and the per-ray store path recomputed a 64-bit address and a double select.
//
// What changes (same producer / mbarrier ring / 2-D tensor-map TMA loads as variant 4):
//   * Work unit = chunk of 256 consecutive rays of one environment; the 15 consumer warps take chunks round-robin over
//     the CTA's whole run (chunk K -> warp K mod 15), so lanes are 94 % used at 961 rays and every warp gets the same
//     number of chunks; a stage's `empty` barrier counts one arrival per chunk.
//   * A lane resolves ray PAIRS (2k, 2k+1): the ray pattern sits in shared memory as three float arrays, so one LDS.64
//     yields the same coordinate of both rays, and the whole ORBIT rotation chain, the window-relative cell coordinate
//     and the reference's result rounding chain run on FADD2 / FMUL2 (add/mul.rn.f32x2 -- per-lane IEEE fp32, so the
//     roundings are exactly those of the scalar chain) -- half the issue slots of the scalar code.
//   * floor() to a cell index is one FADD2.RM against 1.5 * 2^23 (the integer lands in the mantissa) instead of two
//     F2I on the quarter-rate XU pipe; clamping is done on the raw bits.
//   * Grid-line pairs for the whole table live in shared memory once per SM (no per-stage copies by the producer);
//     the prologue issues all of its global loads before the first store (one cold-miss latency instead of three).
// Rays in general cells, cell guesses that miss, windows that do not fit or do not cover (non-uniform lattices) take
// the same out-of-line global-memory helpers as variant 4, so the staging can never change a result.
#include "scan_paired.cuh"

#ifndef ROVER_PAIR_CTX_FROM_PRODUCER
#define ROVER_PAIR_CTX_FROM_PRODUCER 0  // 1: the producer publishes the consumers' per-environment constants (PairCtx) with
                                        // the header and a consumer loads them (ten LDS.128) instead of rebuilding them per
                                        // chunk (~13 % of an environment's instructions).  Measured on a B200 (round 2, same
                                        // box): SLOWER, 25.4 / 63.4 / 209.8 us against 22.5 / 59.4 / 200.7 us at 4096 / 16384 /
                                        // 65536 envs -- the loads sit on the chunk's critical path right after the barrier
                                        // wait and the 40 live registers push the loop to 128 registers with spills.
#endif
#ifndef ROVER_PAIR_DYNAMIC
#define ROVER_PAIR_DYNAMIC 0  // 1: work units handed out from a shared counter instead of the static round-robin deal.
                              // Measured on a B200 (round 2, same box, profiles/time_scan_sizes.py): 22.5 / 59.4 / 200.7 us at
                              // 4096 / 16384 / 65536 envs against 22.5 / 57.0 / 190.0 us for the static deal -- the atomic +
                              // shuffle per unit costs more than the ~1 us of imbalance it removes, so the static deal stays.
#endif

namespace rover {

// kBf16: rover_height_scan_obs -- `out` points at column head_cols of the fp32 observation rows; the kernel also
// writes the bf16 mirror obs_bf16[env, 0 : head_cols + n_rays] (head columns converted from the fp32 row, heights
// rounded from the values it stores).
// kBf16 = 2: the same, but the fp32 heights are NOT stored (the fp32 rows are only read for their head columns): an
// inference loop whose only consumer of the heights is the bf16 policy forward (rover_height_scan_obs_bf16).
template <int kBf16>
__global__ void __launch_bounds__(kPairThreads, 1)
height_scan_paired_kernel(const float* __restrict__ pos_w, const float* __restrict__ quat_w, int n_envs,
                          const float* __restrict__ ray_local, int n_rays, const __grid_constant__ ScanGridDev g,
                          const __grid_constant__ PlaneCellsDev pc, const __grid_constant__ CUtensorMap tmap,
                          float pattern_radius, float max_d, float base_offset, float* __restrict__ out,
                          int out_stride, __nv_bfloat16* __restrict__ obs_bf16, int bf16_stride, int head_cols) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    PairSmem& sm = *reinterpret_cast<PairSmem*>(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_iter = (n_envs - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;  // envs of this CTA
    const int n_chunks = (n_rays + kPairChunk - 1) / kPairChunk;                          // chunks per env
    const bool lines_in_smem = (pc.nx <= kPairMaxLines) && (pc.ny <= kPairMaxLines);
#if ROVER_SCAN_DBG == 3
    const long long dbg_t0 = clock64();
    if (threadIdx.x == 0 && blockIdx.x < 256) {
        g_scan_cta[0][blockIdx.x] = dbg_globaltimer();
        g_scan_cta[1][blockIdx.x] = 0;
    }
#endif

    // ---- prologue.  Producer warp: barriers, then -- lane-parallel, one environment per lane -- positions, table
    // windows and the first ring pass of TMA loads (a window needs the position only), then the sensor frames.
    // Consumer warps: pattern + line tables, every global load issued before the first shared store.
    ProducerEnv cur, nxt;
    int my_flat_z = 1;
    grid_dependency_trigger();  // the policy kernel behind this one sets itself up on SMs as this grid's CTAs retire
    // The launch may overlap the tail of the kernel in front of it on the stream (the MDP step that moves reset envs:
    // common.cuh, launch_overlapped): everything up to grid_dependency_wait() reads only launch-invariant data (barriers,
    // tensor map, ray pattern, lattice lines); the poses are read after it.
    if (warp == 0) {
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap)) : "memory");
            for (int s = 0; s < kPairFullBars; ++s) bar_init(&sm.full_bar[s], 2);  // TMA bytes + header published
            for (int s = 0; s < kPairStages; ++s) bar_init(&sm.empty_bar[s], (uint32_t)n_chunks);
            sm.next_chunk = 0;
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        grid_dependency_wait();
        producer_load(cur, lane, n_iter, pos_w, quat_w);  // cold misses
        __syncwarp();
        producer_window(cur, pc, pattern_radius);
        if (lane < n_iter && lane < kPairEarly && ROVER_SCAN_DBG != 4) {
            // the box is always kPairPitch x kPairWin cells; cells beyond the table are zero-filled and never read;
            // a window that later turns out not to fit / not to cover is loaded all the same and simply not used
            bar_arrive_expect_tx(&sm.full_bar[lane], kPairStageBytes);
            tma_load_window_planar(sm.stage[lane].p, &tmap, cur.ic0, cur.jr0, &sm.full_bar[lane]);
            DBG_STAMP_ANY(16 + lane);
        }
        producer_frame(cur);
        DBG_STAMP(1);
    } else {
        constexpr int kFill = 32 * kPairConsumerWarps;
        constexpr int kPatLoads = (3 * kPairMaxRays + kFill - 1) / kFill;
        constexpr int kLineLoads = (kPairMaxLines + kFill - 1) / kFill;
        const int ct = threadIdx.x - 32;
        static_assert(offsetof(PairSmem, vy) == offsetof(PairSmem, vx) + 4 * kPairMaxRays &&
                          offsetof(PairSmem, vz) == offsetof(PairSmem, vx) + 8 * kPairMaxRays,
                      "vx, vy, vz are filled as one array");
        float* pat_flat = sm.vx;
        float pat[kPatLoads], xl[kLineLoads], xh[kLineLoads], yl[kLineLoads], yh[kLineLoads];
        const float vz0 = __ldg(ray_local + 2);
#pragma unroll
        for (int k = 0; k < kPatLoads; ++k) {  // i = component * kPairMaxRays + slot (vx, vy, vz are contiguous)
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
    if (warp == 1) DBG_STAMP(3);
    if (warp != 0) grid_dependency_wait();  // (the consumers' stores into `out` come after the producer's anyway)
    const bool flat_z = __syncthreads_and(my_flat_z) != 0;  // also publishes the tables / barriers to every warp
    if (warp == 0) DBG_STAMP(0);

    if (warp == 0) {
        // =============================== producer ===============================
        // One lane owns one environment of the current batch of 32: it already holds frame, window and verdict, so the
        // per-environment critical path is wait(empty) -> header -> TMA issue.  (A serial loop that derived the window
        // per iteration took ~850 cycles alone and ~2000 beside busy consumers -- it, not the TMA, starved them.)
        for (int base = 0; base < n_iter; base += 32) {
            if (base > 0) cur = nxt;
            producer_verdict(cur, sm, pc, pattern_radius, lines_in_smem);
            const int n_here = min(32, n_iter - base);
            for (int k = 0; k < n_here; ++k) {
                if (k == kPairStages && base + 32 < n_iter) {  // next batch, computed while the ring is full
                    producer_load(nxt, base + 32 + lane, n_iter, pos_w, quat_w);
                    producer_window(nxt, pc, pattern_radius);
                    producer_frame(nxt);
                }
                if (lane == k) {
                    const int it = base + k;
                    const int s = it % kPairStages;
                    unsigned long long* full = &sm.full_bar[it % kPairFullBars];
                    PairStage& st = sm.stage[s];
                    const bool first_pass = it < kPairEarly && ROVER_SCAN_DBG != 4;  // loaded in the prologue
                    if (!first_pass) {
                        bar_wait(&sm.empty_bar[s], ((uint32_t)(it / kPairStages) & 1u) ^ 1u);  // stage drained
                        if (cur.ok && ROVER_SCAN_DBG != 2) {
                            bar_arrive_expect_tx(full, kPairStageBytes);
                            tma_load_window_planar(st.p, &tmap, cur.ic0, cur.jr0, full);
                        } else {
                            bar_arrive(full);
                        }
                        DBG_STAMP_ANY(16 + it);
                    }
                    st.hdr = {cur.cw, cur.sz, cur.px, cur.py, cur.pz, cur.ic0, cur.jr0, cur.ncols, cur.nrows,
                              cur.ok ? 1 : 0, 0, 0};
                    // the consumers' per-environment constants, ready to load (a staged window implies that the line
                    // tables are in shared memory; vz[0] stands for every ray's z on flat patterns, the only users)
#if ROVER_PAIR_CTX_FROM_PRODUCER
                    if (cur.ok)
                        st.ctx = make_pair_ctx(st.hdr, sm, st, smem_raw, pc.inv_dx, pc.inv_dy, base_offset, max_d, sm.vz[0],
                                               n_envs >> 31);
#endif
                    bar_arrive(full);  // header + context published (release)
                }
                // environments must be issued IN ORDER (the phase-aliasing argument above relies on it): without this
                // the lanes run ahead independently and a later environment whose stage drains first overtakes
                __syncwarp();
            }
        }
        DBG_STAMP(2);
    } else {
        // =============================== consumers ===============================
        // Work units (environment, chunk): chunk K of the CTA's run goes to warp K mod 15 (static deal).  With
        // ROVER_PAIR_DYNAMIC they are handed out in order from a shared counter instead; the phase-aliasing argument in
        // scan_paired.cuh holds either way.
#if ROVER_PAIR_DYNAMIC
        int it = 0, c = 0;
        auto next_unit = [&]() {
            int k = 0;
            if (lane == 0) k = atomicAdd(&sm.next_chunk, 1);
            k = __shfl_sync(0xffffffffu, k, 0);
            it = k / n_chunks;
            c = k - it * n_chunks;
        };
        next_unit();
#else
        const int w = warp - 1;
        const int step_it = kPairConsumerWarps / n_chunks, step_c = kPairConsumerWarps % n_chunks;
        int it = w / n_chunks, c = w % n_chunks;
#endif
#if ROVER_SCAN_DBG == 3
        int dbg_j = 0;
#endif
        while (it < n_iter) {
            const int env = (int)blockIdx.x + it * (int)gridDim.x;
            const int s = it % kPairStages;
            const PairStage& st = sm.stage[s];
#if ROVER_SCAN_DBG == 3
            const int dbg_slot = (w == 0 ? 64 : w == 13 ? 128 : w == 6 ? 192 : 100000) + 4 * dbg_j;
            ++dbg_j;
#endif
            DBG_STAMP(dbg_slot);
            bar_wait(&sm.full_bar[it % kPairFullBars], (uint32_t)(it / kPairFullBars) & 1u);
            DBG_STAMP(dbg_slot + 1);
            const PairHeader h = st.hdr;
            float* __restrict__ out_row = out + (size_t)env * out_stride;
            __nv_bfloat16* __restrict__ bf_row = kBf16 ? obs_bf16 + (size_t)env * bf16_stride + head_cols : nullptr;
            const int r_begin = c * kPairChunk, r_end = min(r_begin + kPairChunk, n_rays);
            if (kBf16 && c == 0 && lane < head_cols)  // the head of the observation (written by the post-step kernel)
                bf_row[lane - head_cols] = __float2bfloat16_rn(out_row[lane - head_cols]);
            if (ROVER_SCAN_DBG == 1) {
            } else if (h.mode == 1) {
#if ROVER_PAIR_CTX_FROM_PRODUCER
                const PairCtx cx = st.ctx;  // ten LDS.128: built once per environment by the producer
#else
                const PairCtx cx = make_pair_ctx(h, sm, st, smem_raw, pc.inv_dx, pc.inv_dy, base_offset, max_d, sm.vz[0],
                                                 n_envs >> 31);
#endif
                const float sz2 = __fmul_rn(h.sz, 2.f);
                for (int b0 = r_begin; b0 < r_end; b0 += kPairBatch) {
                    const int r = b0 + lane;  // rays r, r + 64 (slot 0) and r + 32, r + 96 (slot 1)
                    float* __restrict__ o = out_row + r;
                    __nv_bfloat16* __restrict__ ob = kBf16 ? bf_row + r : nullptr;
                    unsigned defer;
                    if (flat_z && b0 + kPairBatch <= n_rays) {
                        defer = resolve_pair<true, true, kBf16>(smem_raw, sm, cx, b0 + 2 * lane, r, n_rays, o, ob);
                        defer |= resolve_pair<true, true, kBf16>(smem_raw, sm, cx, b0 + 64 + 2 * lane, r + 32, n_rays, o + 32,
                                                                 ob + 32) << 2;
                    } else {
                        defer = resolve_pair<false, false, kBf16>(smem_raw, sm, cx, b0 + 2 * lane, r, n_rays, o, ob);
                        defer |= resolve_pair<false, false, kBf16>(smem_raw, sm, cx, b0 + 64 + 2 * lane, r + 32, n_rays, o + 32,
                                                                   ob + 32) << 2;
                    }
                    // rare: cell guess off by one, ray on the closed far border or outside the grid, general cell
                    if (defer != 0u) {
                        for (int u = 0; u < 4; ++u) {
                            if (!((defer >> u) & 1u)) continue;
                            const int rr = r + (u >> 1) * 32 + (u & 1) * 64;
                            const int sl = b0 + (u >> 1) * 64 + 2 * lane + (u & 1);
                            const float vx = sm.vx[sl], vy = sm.vy[sl];
                            const float tx = -__fmul_rn(sz2, vy), ty = __fmul_rn(sz2, vx);
                            const float X = __fadd_rn(__fadd_rn(__fadd_rn(vx, __fmul_rn(h.cw, tx)), -__fmul_rn(h.sz, ty)), h.px);
                            const float Y = __fadd_rn(__fadd_rn(__fadd_rn(vy, __fmul_rn(h.cw, ty)), __fmul_rn(h.sz, tx)), h.py);
                            pair_resolve_deferred_ray(&sm, &st, g, pc.inv_dx, pc.inv_dy, X, Y, __fadd_rn(sm.vz[sl], h.pz),
                                                      h.pz, max_d, base_offset, kBf16 == 2 ? nullptr : out_row + rr,
                                                      kBf16 ? bf_row + rr : nullptr);
                        }
                    }
                }
            } else {
                pair_resolve_chunk_from_global(&sm, lane, r_begin, r_end, h, g, pc, max_d, base_offset,
                                               kBf16 == 2 ? nullptr : out_row, bf_row);
            }
            __syncwarp();
            DBG_STAMP(dbg_slot + 2);
            if (lane == 0) bar_arrive(&sm.empty_bar[s]);  // this chunk no longer reads the stage
#if ROVER_PAIR_DYNAMIC
            next_unit();
#else
            it += step_it;
            c += step_c;
            if (c >= n_chunks) {
                c -= n_chunks;
                ++it;
            }
#endif
        }
    }
#if ROVER_SCAN_DBG == 3
    if (lane == 0 && blockIdx.x < 256) atomicMax(&g_scan_cta[1][blockIdx.x], dbg_globaltimer());
#endif
}

int launch_height_scan_pipelined(const float* pos_w, const float* quat_w, int n_envs, const float* ray_local,
                                 int n_rays, const ScanGridDev& g, const RoverPlaneCells* cells, float4 pattern_box,
                                 float max_d, float base_offset, float* out, int out_stride, float* hits,
                                 cudaStream_t stream);

// obs_bf16 != nullptr: `out` is column head_cols of the fp32 observation rows and the bf16 mirror is written as well
// (rover_height_scan_obs); the caller has checked that variant 5 can run (planar table, pattern size, no hit output).
int launch_height_scan_paired(const float* pos_w, const float* quat_w, int n_envs, const float* ray_local, int n_rays,
                              const ScanGridDev& g, const RoverPlaneCells* cells, float4 pattern_box, float max_d,
                              float base_offset, float* out, int out_stride, float* hits, uint16_t* obs_bf16,
                              int bf16_stride, int head_cols, cudaStream_t stream, bool bf16_only) {
    // hit positions are a debugging / test output: served by variant 4's kernel (same heights, same table); so is a
    // table without the planar copy
    if (obs_bf16 == nullptr && (hits != nullptr || cells->entries_planar == nullptr))
        return launch_height_scan_pipelined(pos_w, quat_w, n_envs, ray_local, n_rays, g, cells, pattern_box, max_d,
                                            base_offset, out, out_stride, hits, stream);
    ROVER_CHECK(n_rays >= 1 && n_rays <= kPairMaxRays, "height_scan_paired: pattern of %d rays (1..%d supported)", n_rays,
                kPairMaxRays);
    ROVER_CHECK(cells->entries_planar != nullptr && hits == nullptr, "height_scan_paired: bf16 mirror needs the planar table");
    ROVER_CHECK(head_cols >= 0 && head_cols <= 32, "height_scan_paired: head_cols %d out of range", head_cols);
    static int n_sms = 0;
    static bool configured = false;
    if (!configured) {
        int dev = 0;
        ROVER_CUDA(cudaGetDevice(&dev));
        ROVER_CUDA(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev));
        ROVER_CUDA(cudaFuncSetAttribute(height_scan_paired_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)sizeof(PairSmem)));
        ROVER_CUDA(cudaFuncSetAttribute(height_scan_paired_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)sizeof(PairSmem)));
        ROVER_CUDA(cudaFuncSetAttribute(height_scan_paired_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)sizeof(PairSmem)));
        configured = true;
    }
    alignas(64) CUtensorMap tmap;
    if (const int rc = encode_planar_tensor_map(&tmap, cells, kPairPitch, kPairWin, "height_scan_paired")) return rc;
    PlaneCellsDev pc{cells->xs, cells->ys, reinterpret_cast<const float4*>(cells->entries), cells->nx, cells->ny,
                     cells->inv_dx, cells->inv_dy};
    // every ray origin lies within this distance of the sensor position (the yaw rotation preserves norms)
    const float rx = fmaxf(fabsf(pattern_box.x), fabsf(pattern_box.y)), ry = fmaxf(fabsf(pattern_box.z), fabsf(pattern_box.w));
    const float radius = sqrtf(rx * rx + ry * ry) * 1.0001f + 1.0e-3f;
    const int grid = n_envs < n_sms ? n_envs : n_sms;
    ROVER_CHECK(!bf16_only || obs_bf16 != nullptr, "height_scan_paired: bf16-only output needs the bf16 buffer");
    if (obs_bf16 != nullptr && bf16_only)
        ROVER_CUDA(launch_overlapped(height_scan_paired_kernel<2>, dim3(grid), dim3(kPairThreads), sizeof(PairSmem), stream,
                                     pos_w, quat_w, n_envs, ray_local, n_rays, g, pc, tmap, radius, max_d, base_offset, out,
                                     out_stride, reinterpret_cast<__nv_bfloat16*>(obs_bf16), bf16_stride, head_cols));
    else if (obs_bf16 != nullptr)
        ROVER_CUDA(launch_overlapped(height_scan_paired_kernel<1>, dim3(grid), dim3(kPairThreads), sizeof(PairSmem), stream,
                                     pos_w, quat_w, n_envs, ray_local, n_rays, g, pc, tmap, radius, max_d, base_offset, out,
                                     out_stride, reinterpret_cast<__nv_bfloat16*>(obs_bf16), bf16_stride, head_cols));
    else
        ROVER_CUDA(launch_overlapped(height_scan_paired_kernel<0>, dim3(grid), dim3(kPairThreads), sizeof(PairSmem), stream,
                                     pos_w, quat_w, n_envs, ray_local, n_rays, g, pc, tmap, radius, max_d, base_offset, out,
                                     out_stride, nullptr, 0, 0));
    return check_launch("height_scan_paired_kernel");
}

}  // namespace rover

#if ROVER_SCAN_DBG == 3
extern "C" int rover_debug_scan_timeline(unsigned long long* host_dst) {
    return (int)cudaMemcpyFromSymbol(host_dst, rover::g_scan_dbg, sizeof(rover::g_scan_dbg));
}
extern "C" int rover_debug_scan_ctas(unsigned long long* host_dst) {
    return (int)cudaMemcpyFromSymbol(host_dst, rover::g_scan_cta, sizeof(rover::g_scan_cta));
}
#endif
