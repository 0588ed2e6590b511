/* rover_b200.h -- C ABI of the B200-native non-physics MDP hot path of AAURoverEnv-v0.
 *
 * The reference (abmoRobotics/isaac_rover_orbit) is pure Python on top of ORBIT / warp / skrl and has NO
 * FFI of its own; the boundary it offers is ORBIT's manager-term plugin API (SURVEY.md section 8b).  This
 * library sits UNDER those Python callables: each entry point below names the reference interface
 * (file:line under the reference root) whose per-step work it replaces.  The Python mirror of the
 * manager-term API that calls these lives in isaac_rover_orbit_b200/ (ctypes; see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is DEVICE memory (cudaMalloc / torch CUDA tensor .data_ptr()) unless it says "host";
 *   - tensors are dense row-major fp32 unless stated; quaternions are (w, x, y, z);
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued on it, nothing synchronises;
 *   - every function returns 0 on success, non-zero on error; rover_last_error() gives the message
 *     (thread-local).  No function falls back to a CPU path;
 *   - the step kernels (MDP step, height scan, policy forward, Gaussian act) are launched with programmatic stream
 *     serialisation: one of them may begin while the kernel in front of it on the stream retires, and waits for that
 *     kernel's completion before it reads the per-step inputs.  Launch-invariant inputs -- ray pattern, scan tables,
 *     packed network weights -- are read before that wait: do not let the kernel that writes them be the one directly
 *     in front of a step call on the same stream (synchronise once after building them).  ROVER_PDL=0 disables it.
 */
#ifndef ROVER_B200_H
#define ROVER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ROVER_B200_ABI_VERSION 5
#define ROVER_MAX_LEVELS 12
#define ROVER_NUM_REWARD_TERMS 7
#define ROVER_NUM_TERMINATION_TERMS 4
#define ROVER_STATS_LEN 16

int rover_abi_version(void);
const char* rover_last_error(void);

/* ---------------------------------------------------------------------------------------------------
 * Height scan.  Replaces ORBIT RayCaster._update_buffers_impl -> raycast_mesh -> warp mesh_query_ray
 * (third-party; wired at rover_envs/envs/navigation/rover_env_cfg.py:78-86) fused with
 * height_scan_rover (rover_envs/envs/navigation/mdp/observations.py:35-45).
 * ------------------------------------------------------------------------------------------------- */
typedef struct RoverScanLevel {
    float ox, oy;        /* grid origin of this level                                   */
    float cell;          /* cell size (level-0 size * 2^level)                           */
    float inv_cell;      /* 1 / cell, the value the builder used                         */
    int32_t ncx, ncy;    /* grid extent                                                  */
    int32_t start_offset;/* offset of this level's (ncx*ncy+1) entries inside cell_start */
    int32_t reserved;
} RoverScanLevel;

typedef struct RoverScanGrid {
    int32_t n_levels;
    int32_t span;                 /* a ray in cell (i,j) tests homes (i-span..i, j-span..j)  */
    RoverScanLevel level[ROVER_MAX_LEVELS];
    const int32_t* cell_start;    /* record index ranges per home cell, all levels concatenated */
    const float* records;         /* n_records x 12 floats, 16-byte aligned                   */
    int32_t n_records;
    int32_t reserved;
} RoverScanGrid;

/* Plane-cell table (plane_cells.py): rectilinear grid whose cells carry the closed-form surface
 * z = a*lx + b*ly + c + k*min(A*lx + B*ly + C, 0); entry = {a,b,c,k | A,B,C,tag}; tag != 0 -> general cell,
 * the ray falls back to the home-grid walk.  Used by variant 2. */
typedef struct RoverPlaneCells {
    const float* xs;       /* [nx+1] grid lines, strictly increasing */
    const float* ys;       /* [ny+1] */
    const float* entries;  /* [ny, nx, 8], 16-byte aligned */
    int32_t nx, ny;
    float inv_dx, inv_dy;  /* nx / (xs[nx]-xs[0]), ny / (ys[ny]-ys[0]): first guess of the cell */
    const float* entries_planar; /* optional (may be NULL): the same table as two planes [2, ny, nx, 4] -- plane 0 the
                                    first, plane 1 the second float4 of every entry; 16-byte aligned.  Variant 5 stages
                                    windows from it (16-byte plane entries with an odd row pitch in shared memory make
                                    the per-ray LDS.128 bank-conflict free); without it variant 5 runs as variant 4. */
} RoverPlaneCells;

/* pos_w [n_envs,3], quat_w [n_envs,4]: sensor (body) pose, sensor.data.pos_w / quat_w.
 * ray_starts_local [n_rays,3]: ORBIT RayCaster.ray_starts (grid_pattern + offset.pos), env frame.
 * out_heights [n_envs,n_rays]: pos_w.z - hit.z - base_offset; a miss (no hit with 0 <= t < max_dist) is -inf.
 * out_hits_w [n_envs,n_rays,3] (optional, may be NULL): sensor.data.ray_hits_w, +inf on a miss.
 * pattern_box (HOST, 4 floats: xmin, xmax, ymin, ymax of ray_starts_local; required by variants 4 and 5).
 * cells (HOST struct, device pointers inside; required by variants 2, 4, 5, may be NULL otherwise).
 * variant: 0 = direct home-grid walk (any mesh), 2 = plane-cell fast path with home-grid fallback for general cells,
 * 4 = persistent warp-specialised pipeline (producer warp + 8-stage ring of 2-D tensor-map TMA loads on mbarriers +
 * consumer warps; also serves out_hits_w), 5 = variant 4's pipeline with 256-ray chunks dealt round-robin to the
 * consumer warps and ray pairs resolved with packed fp32 (FADD2 / FMUL2) -- the default of the Python binding.
 * (1 and 3 were measured slower in round 1 and are retired: the call fails for them.)
 * All variants produce the same heights. */
int rover_height_scan(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                      int32_t n_rays, const float* pattern_box /* host */, const RoverScanGrid* grid /* host */,
                      const RoverPlaneCells* cells /* host */, float max_distance, float base_offset,
                      float* out_heights, int32_t out_stride, float* out_hits_w, int32_t variant, void* stream);

/* The height scan with rays in any direction: ORBIT RayCasterCfg.attach_yaw_only and GridPatternCfg.direction honoured.
 * Replaces the same reference lines as rover_height_scan (rover_env_cfg.py:78-86 + observations.py:35-45, via ORBIT
 * RayCaster._update_buffers_impl), both branches of the frame:
 *   attach_yaw_only != 0: starts_w = quat_apply_yaw(q, starts) + p (the vertical kernels' starts bit for bit), dirs_w = dirs;
 *   attach_yaw_only == 0: starts_w = quat_apply(q, starts) + p, dirs_w = quat_apply(q, dirs), q as given (not normalised).
 * ray_dirs_local [n_rays,3]: per-ray directions, used as given (not normalised): the hit is the first P(t) = S + t * D on
 * the mesh with 0 <= t < max_distance, t in units of |D|; D == 0 misses.  Surfaces are double-sided.
 * out_heights / out_hits_w / out_stride / base_offset as in rover_height_scan (hit = S + t * D, one rounding per component;
 * a miss is -inf / +inf).  For D = (0, 0, -1) with attach_yaw_only the result equals variant 2 bit for bit.
 * cells is required, and grid must hold the home grid when the table has general cells (the rule of variant 2).
 * Deviation: faces with zero XY area (vertical walls) are in neither table, so a tilted ray passes through them where
 * mesh_query_ray would hit (DESIGN.md section 2, (iii)); DEM lattices have no such faces. */
int rover_ray_cast(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                   const float* ray_dirs_local, int32_t n_rays, int32_t attach_yaw_only, const RoverScanGrid* grid /* host */,
                   const RoverPlaneCells* cells /* host */, float max_distance, float base_offset, float* out_heights,
                   int32_t out_stride, float* out_hits_w, void* stream);

/* The height scan for a caller whose poses and heights live in HOST memory (a CPU-side simulator; bench.py's `e2e`):
 * pos_host [n_envs,3], quat_host [n_envs,4] and out_host [n_envs,out_stride] are host pointers (page-locked for the
 * copies to be asynchronous), everything else as in rover_height_scan.  The poses are copied in, the environments are
 * scanned in `n_slices` slices on `stream`, and slice k's heights travel to the host on an internal copy stream while
 * slice k + 1 is scanned; `stream` is complete when all heights are in out_host.  (On a B200 behind PCIe Gen5 the step is
 * the 15.7 MB device-to-host copy -- 300 of 340 us at cfg-2 -- and slicing does not pay: 1 slice 344.6 us, 8 slices 357 us,
 * profiles/time_e2e_slices.py; n_slices = 1 runs everything on `stream`.)  `work`: device scratch of
 * rover_height_scan_host_work_bytes(n_envs, out_stride) bytes, 256-byte aligned.  Replaces the same reference lines as
 * rover_height_scan (rover_env_cfg.py:78-86 + observations.py:35-45) plus the .cpu() / .to(device) round trip around them. */
int64_t rover_height_scan_host_work_bytes(int32_t n_envs, int32_t out_stride);
int rover_height_scan_host(const float* pos_host, const float* quat_host, int32_t n_envs, const float* ray_starts_local,
                           int32_t n_rays, const float* pattern_box, const RoverScanGrid* grid, const RoverPlaneCells* cells,
                           float max_distance, float base_offset, float* out_host, int32_t out_stride, void* work,
                           int64_t work_bytes, int32_t n_slices, int32_t variant, void* stream);
/* The observation variant of the height scan (B200-native addition, no counterpart in the reference): obs is the fp32
 * observation buffer [n_envs, obs_stride] whose columns [0, head_cols) were written by rover_mdp_post_step; the heights
 * go to columns [head_cols, head_cols + n_rays), and obs_bf16 [n_envs, bf16_stride] receives the bf16 (round to nearest
 * even) mirror of columns [0, head_cols + n_rays) -- the operand of rover_policy_forward_bf16 / rover_value_forward_bf16.
 * Runs as variant 5 with the extra stores when the table has a planar copy and n_rays <= 1024, else as the best
 * applicable variant followed by one conversion pass.  Heights are exactly those of rover_height_scan. */
int rover_height_scan_obs(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                          int32_t n_rays, const float* pattern_box /* host */, const RoverScanGrid* grid /* host */,
                          const RoverPlaneCells* cells /* host */, float max_distance, float base_offset, float* obs,
                          int32_t obs_stride, int32_t head_cols, uint16_t* obs_bf16, int32_t bf16_stride, void* stream);
/* The same with ONLY the bf16 observation written: for a loop in which the policy forward on bf16 observations
 * (rover_policy_forward_bf16) is the heights' only consumer.  `obs_head` is the fp32 observation buffer, read for its
 * head columns (written by the MDP step) and otherwise left alone on the variant-5 path -- its height columns keep
 * whatever they held (a general table falls back to scan + conversion and does write them).  The policy rounds fp32
 * observations to these very bf16 values, so means, actions and the whole trajectory are bit-identical to the fp32 loop;
 * what is saved is the 3844 B/env fp32 store and the 3860 B/env fp32 read of the forward pass. */
int rover_height_scan_obs_bf16(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                               int32_t n_rays, const float* pattern_box /* host */, const RoverScanGrid* grid,
                               const RoverPlaneCells* cells, float max_distance, float base_offset, const float* obs_head,
                               int32_t obs_stride, int32_t head_cols, uint16_t* obs_bf16, int32_t bf16_stride, void* stream);

/* The observation and host-buffer forms of rover_ray_cast (rays in any direction; B200-native additions like the two
 * entries above).  rover_ray_cast_obs / rover_ray_cast_obs_bf16 replace the same reference lines as rover_ray_cast
 * (rover_env_cfg.py:78-86 + observations.py:35-45) and take the arguments of rover_height_scan_obs /
 * rover_height_scan_obs_bf16 without pattern_box, plus ray_dirs_local and attach_yaw_only as in rover_ray_cast.  One
 * launch: the fp32 heights (not in the _bf16 form) are rover_ray_cast's bit for bit, obs_bf16 receives the bf16 (round
 * to nearest even) mirror of columns [0, head_cols + n_rays); any head_cols >= 0; n_rays == 0 mirrors the head only.
 * The head columns are read after the kernel in front of this one (the post-step that writes them) has completed.
 * cells is required, as for rover_ray_cast. */
int rover_ray_cast_obs(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                       const float* ray_dirs_local, int32_t n_rays, int32_t attach_yaw_only, const RoverScanGrid* grid /* host */,
                       const RoverPlaneCells* cells /* host */, float max_distance, float base_offset, float* obs,
                       int32_t obs_stride, int32_t head_cols, uint16_t* obs_bf16, int32_t bf16_stride, void* stream);
int rover_ray_cast_obs_bf16(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                            const float* ray_dirs_local, int32_t n_rays, int32_t attach_yaw_only,
                            const RoverScanGrid* grid /* host */, const RoverPlaneCells* cells /* host */, float max_distance,
                            float base_offset, const float* obs_head, int32_t obs_stride, int32_t head_cols,
                            uint16_t* obs_bf16, int32_t bf16_stride, void* stream);
/* rover_height_scan_host with rover_ray_cast as the scan: replaces the same reference lines as rover_ray_cast plus the
 * .cpu() / .to(device) round trip around them.  Arguments of rover_height_scan_host without pattern_box and variant, plus
 * ray_dirs_local and attach_yaw_only; the same work area (rover_height_scan_host_work_bytes) and n_slices semantics. */
int rover_ray_cast_host(const float* pos_host, const float* quat_host, int32_t n_envs, const float* ray_starts_local,
                        const float* ray_dirs_local, int32_t n_rays, int32_t attach_yaw_only, const RoverScanGrid* grid,
                        const RoverPlaneCells* cells, float max_distance, float base_offset, float* out_host,
                        int32_t out_stride, void* work, int64_t work_bytes, int32_t n_slices, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Fused MDP step.  Replaces, in one launch (SURVEY.md 8a rows a-1..a-23):
 *   AckermannAction2.process_actions/apply_actions/ackermann  rover_envs/mdp/actions/ackermann_actions.py:226-322
 *   ORBIT ActionManager.process_action (prev_action <- action <- new)
 *   episode_length_buf += 1                                    entrypoints/rover_env.py:79
 *   time_out / is_success / far_from_target / collision        mdp/terminations.py:14-64 (+ ORBIT mdp.time_out)
 *   the seven reward terms, weight * dt, episodic sums         mdp/rewards.py:14-137 (+ ORBIT RewardManager.compute)
 * It reads the PREVIOUS step's pos_cmd_b, as the reference's step ordering does (rover_env.py:82-86).
 * ------------------------------------------------------------------------------------------------- */
typedef struct RoverMdpParams {
    /* actions_cfg.py:20, robots/aau_rover/env_cfg.py:21-31 */
    float scale_lin, scale_ang, offset_lin, offset_ang;
    float wheelbase_length, middle_wheel_distance, rear_and_front_wheel_distance, wheel_radius;
    float min_radius;            /* (float)(middle_wheel_distance * 0.8) evaluated in double, ackermann_actions.py:264 */
    float wheel_diameter;        /* (float)(wheel_radius * 2) evaluated in double, ackermann_actions.py:503 (variant 3) */
    /* rover_env_cfg.py:128-163 */
    float weight[ROVER_NUM_REWARD_TERMS];
    float reached_threshold, far_threshold;
    float step_dt;               /* sim.dt * decimation (rover_env_cfg.py:269-270) */
    int32_t max_episode_length;  /* ceil(episode_length_s / step_dt) */
    /* rover_env_cfg.py:104-112 */
    float obs_distance_scale, obs_heading_scale;
    /* terrain_importer.py:132, rover_env_cfg.py:191-200, randomizations.py:12 */
    float target_distance, resampling_time, heading_lo, heading_hi, spawn_z_offset;
    int32_t num_bodies;          /* contact-sensor bodies B: force_matrix_w is [n_envs, B, 1, 3] */
    int32_t action_variant;      /* 2 = AckermannAction2 (default, actions_cfg.py:17), 1 = AckermannAction
                                    (ackermann_actions.py:19-158), 3 = ackermann() of AckermannAction3 (:423-505) */
    float episode_length_s;      /* max_episode_length_s (rover_env_cfg.py:269): divisor of the "Episode Reward/..." log */
} RoverMdpParams;

typedef struct RoverMdpState {     /* persistent manager state, mutated in place */
    float* action;                 /* [N,2] action_manager.action                        */
    float* prev_action;            /* [N,2] action_manager.prev_action                   */
    float* pos_cmd_w;              /* [N,3] TerrainBasedPositionCommand.pos_command_w    */
    float* heading_cmd_w;          /* [N]                                                */
    float* pos_cmd_b;              /* [N,3] .command                                     */
    float* heading_cmd_b;          /* [N]                                                */
    float* time_left;              /* [N]   CommandTerm.time_left                        */
    int64_t* command_counter;      /* [N]                                                */
    int64_t* episode_length_buf;   /* [N]   env.episode_length_buf (int64 like ORBIT)    */
    float* episode_sums;           /* [N,7] RewardManager._episode_sums                  */
    float* env_origins;            /* [N,3] terrain.env_origins                          */
    float* err_pos;                /* [N]   metrics["error_pos"]                         */
    float* err_heading;            /* [N]   metrics["error_heading"]                     */
} RoverMdpState;

typedef struct RoverMdpOut {
    float* processed_actions;      /* [N,2] */
    float* joint_pos;              /* [N,4] steering targets  [FL,RL,RR,FR] */
    float* joint_vel;              /* [N,6] drive targets     [ML,FL,RL,RR,MR,FR] */
    float* reward;                 /* [N]   */
    float* term_rewards;           /* [N,7] weight*value*dt per term */
    float* term_values;            /* [N,7] unweighted term values (what the reference's reward functions return) */
    uint8_t* terminated;           /* [N]   */
    uint8_t* truncated;            /* [N]   */
    uint8_t* term_flags;           /* [N,4] time_limit,is_success,far_from_target,collision */
    uint8_t* reset_flags;          /* [N]   terminated | truncated */
    int32_t* block_reset_counts;   /* [ceil(N/ROVER_MDP_BLOCK)] resets per thread block (rank scan input) */
} RoverMdpOut;

#define ROVER_MDP_BLOCK 64

/* new_actions [N,2]; force_matrix_w [N,B,1,3] (contact_sensor.data.force_matrix_w).
 * phases: ROVER_PRE_ACTIONS = action-manager shift + Ackermann (what runs BEFORE the physics step),
 *         ROVER_PRE_TERMS   = counters + terminations + rewards (what runs AFTER it); both = the fused launch. */
#define ROVER_PRE_ACTIONS 1
#define ROVER_PRE_TERMS 2
#define ROVER_PRE_ALL 3
int rover_mdp_pre_step(const float* new_actions, const float* force_matrix_w, int32_t n_envs,
                       const RoverMdpParams* params /* host */, const RoverMdpState* state /* host struct */,
                       const RoverMdpOut* out /* host struct */, int32_t phases, void* stream);

/* Stand-alone action kinematics (any of the three variants; joint orders as the reference returns them):
 *   variant 2: joint_pos [FL,RL,RR,FR], joint_vel [ML,FL,RL,RR,MR,FR]       ackermann_actions.py:316-317
 *   variant 1: joint_pos [FL,FR,RL,RR], joint_vel [FL,FR,ML,MR,RL,RR]       ackermann_actions.py:111, 158
 *   variant 3: joint_pos [FL,FR,RL,RR], joint_vel [FL,FR,ML,MR,RL,RR]       ackermann_actions.py:499-501 */
int rover_ackermann(const float* actions /* [N,2] raw */, int32_t n_envs, const RoverMdpParams* params /* host */,
                    float* processed /* [N,2] */, float* joint_pos /* [N,4] */, float* joint_vel /* [N,6] */,
                    void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Reset + command update + observation head.  Replaces, in one launch (rows a-4..a-6, a-22..a-28):
 *   reset_root_state_rover                        mdp/randomizations.py:12-39
 *   ORBIT manager .reset(ids) combine rules       (action/reward/command/termination), episode stats
 *   TerrainBasedPositionCommand._resample_command utils/terrains/terrain_importer.py:74-95
 *   RoverTerrainImporter.sample_new_targets       :134-175 (rejection loop, bounded to n_rounds)
 *   TerrainManager.check_if_target_is_valid       utils/terrains/terrain_utils.py:202-223
 *   HeightmapManager.get_height_at                :62-84
 *   CommandTerm.compute: _update_metrics, time_left, _update_command  terrain_importer.py:97-106
 *   last_action / distance / angle observations   mdp/observations.py:15-32, rover_env_cfg.py:103-112
 * Random variates are inputs so that oracle and kernel consume identical numbers:
 *   spawn_perm[j] (int64) = spawn row of the j-th reset env (ascending env id);
 *   yaw_u[N], heading_u[N], theta_u[N, n_rounds] = uniform [0,1) variates indexed by env id.
 * root_pos_w / root_quat_w are updated in place for reset envs (write_root_pose_to_sim).
 * stats [ROVER_STATS_LEN] f32 is ACCUMULATED (atomicAdd): 7 reward sums, 4 termination counts, err_pos sum,
 * err_heading sum, number of resets, rounds-exhausted count, time-resample count.  The reduction is
 * deterministic (per-block partials in `scratch`, summed in block order by the last block to finish).
 * obs [N, obs_stride]: columns 0..3 are written (actions(2), distance*0.11, angle/pi).
 * ------------------------------------------------------------------------------------------------- */
typedef struct RoverTerrainTables {
    const float* heightmap;       /* [H,W] */
    const uint8_t* safe_mask;     /* [H,W] 1 = rock/unsafe */
    int32_t height, width;        /* H, W */
    float offset_x, offset_y;     /* (min_x, min_y) added (sic) to xy/res, terrain_utils.py:75 */
    float resolution;             /* 0.05 */
    const float* spawn_table;     /* [n_spawns,3] */
    int32_t n_spawns;
    int32_t reserved;
} RoverTerrainTables;

/* `phases` selects which parts of the post-step run (all of them in the fused step); the single-purpose
 * combinations back the individual manager-term calls of the reference API:
 *   ROVER_PHASE_SPAWN     reset_root_state_rover for envs with reset_flags != 0
 *   ROVER_PHASE_MANAGERS  action / reward / command-metric / termination manager resets + statistics, ep_len = 0
 *   ROVER_PHASE_RESAMPLE  CommandTerm._resample for envs with reset_flags != 0
 *   ROVER_PHASE_METRICS   _update_metrics
 *   ROVER_PHASE_TIME      time_left -= dt and the time-based resample
 *   ROVER_PHASE_COMMAND   _update_command
 *   ROVER_PHASE_OBS       observation head */
#define ROVER_PHASE_SPAWN 1
#define ROVER_PHASE_MANAGERS 2
#define ROVER_PHASE_RESAMPLE 4
#define ROVER_PHASE_METRICS 8
#define ROVER_PHASE_TIME 16
#define ROVER_PHASE_COMMAND 32
#define ROVER_PHASE_OBS 64
#define ROVER_PHASE_ALL 127

int rover_mdp_post_step(float* root_pos_w, float* root_quat_w, int32_t n_envs, const RoverMdpParams* params,
                        const RoverMdpState* state, const RoverMdpOut* out, const RoverTerrainTables* tables,
                        const int64_t* spawn_perm, const float* yaw_u, const float* heading_u, const float* theta_u,
                        int32_t n_rounds, int64_t* out_spawn_index /* [N], -1 if not reset */, float* stats,
                        float* scratch /* [ceil(N/ROVER_MDP_BLOCK)*ROVER_STATS_LEN + 1] f32, zeroed once */,
                        float* obs, int32_t obs_stride, int32_t phases, void* stream);

/* Where the random variates of the reset path come from (randomizations.py:22, 30; terrain_importer.py:94-95, 169).
 *   rng_state == NULL: explicit arrays, as documented above (parity tests feed the oracle the same numbers);
 *   rng_state != NULL: DEVICE uint64[2] = {seed, step}.  The kernel evaluates the counter-based generator of
 *     csrc/rng.cuh in registers -- Philox4x32-10, key = seed, counter = (env, step, stream); the spawn row of env i is a
 *     keyed bijection of [0, n_spawns) at i (K reset envs draw K distinct, uniformly random rows: the distribution of
 *     randperm(len)[:K], without needing the reset rank) -- and its last block advances `step`, so the launch is
 *     CUDA-graph safe and needs no torch generator call on the step path.
 *     rover_rng_variates() evaluates the same functions on the host: spawn_by_env[i], yaw_u[i], heading_u[i],
 *     theta_u[i, r] for one (seed, step) -- what a kernel launched with that state consumes, bit for bit (to feed them
 *     through the explicit arrays: spawn_perm[j] = spawn_by_env[id of the j-th reset env]). */
typedef struct RoverResetVariates {
    const int64_t* spawn_perm;
    const float* yaw_u;
    const float* heading_u;
    const float* theta_u;
    int32_t n_rounds;          /* bound of the rejection loop (both modes) */
    int32_t reserved;
    uint64_t* rng_state;
} RoverResetVariates;

/* The post-step with every option (the entries above forward to it):
 *   variates: explicit arrays or the in-kernel generator (see RoverResetVariates);
 *   log_out (DEVICE f32[16], may be NULL): extras["log"] as the ORBIT managers' reset() build it (SURVEY.md A.2) --
 *     [0..6] Episode Reward/<term> = mean(episode_sums[ids]) / episode_length_s, [7..10] Episode Termination/<term>
 *     counts, [11], [12] Metrics/target_pose/error_pos|error_heading means, [13] number of resets, [14] rounds
 *     exhausted, [15] time-based resamples -- written ONLY by a launch (with ROVER_PHASE_MANAGERS) in which at least one
 *     env reset: the reference calls _reset_idx only then (rover_env.py:89-91), so the last values persist otherwise. */
int rover_mdp_post_step_v3(float* root_pos_w, float* root_quat_w, int32_t n_envs, const RoverMdpParams* params,
                           const RoverMdpState* state, const RoverMdpOut* out, const RoverTerrainTables* tables,
                           const RoverResetVariates* variates /* host */, int64_t* out_spawn_index, float* stats,
                           float* scratch, float* log_out, float* obs, int32_t obs_stride, int32_t phases,
                           const struct RoverStatsExchange* xchg /* host, may be NULL */, void* stream);
/* HOST function (no GPU work): the variates of one (seed, step) into host arrays; any output may be NULL.
 * spawn_by_env [min(n_envs, n_spawns)], yaw_u [n_envs], heading_u [n_envs], theta_u [n_envs, n_rounds]. */
int rover_rng_variates(uint64_t seed, uint64_t step, int32_t n_envs, int32_t n_rounds, int32_t n_spawns,
                       int64_t* spawn_by_env, float* yaw_u, float* heading_u, float* theta_u);
/* HOST: one Philox4x32-10 block (Random123 known-answer vectors pin it: tests/test_rng_cpu.py) */
int rover_philox4x32_10(const uint32_t counter[4], const uint32_t key[2], uint32_t out[4]);
/* The MDP step's functions that are not correctly rounded, evaluated elementwise by the same device code the step kernels
 * run (test support: an fp32 model of the step takes them from here, tests/mdp_exact.py).  DEVICE f32 arrays of n:
 * ROVER_MDP_MATH_ATAN2: out = atan2f(a, b); ROVER_MDP_MATH_SIN: out = sinf(a); ROVER_MDP_MATH_COS: out = cosf(a)
 * (b unused, may be NULL).  Asynchronous on `stream`. */
#define ROVER_MDP_MATH_ATAN2 0
#define ROVER_MDP_MATH_SIN 1
#define ROVER_MDP_MATH_COS 2
int rover_mdp_math(int32_t op, const float* a, const float* b, float* out, int32_t n, void* stream);

/* rover_mdp_pre_step + rover_mdp_post_step_x in ONE launch, for callers whose physics does not sit between the two (the
 * synthetic-physics loop of bench.py; a simulator that hands over root state and contacts before the step): the reset
 * rank that the post-step needs comes from a decoupled look-back over the blocks' reset counts instead of a second
 * launch, and every env's pre-step outputs are consumed by the thread that produced them.  Same outputs, bit for bit.
 * lookback: DEVICE uint64 [ceil(N / ROVER_MDP_BLOCK) + 2], zeroed once; the kernel maintains it (CUDA-graph safe).
 * (rover_mdp_step_v3 with the in-kernel generator needs neither a rank nor a look-back: lookback may be NULL there.)
 * Measured on a B200 at 16384 envs inside a CUDA graph: 34.4 us against 33.1 us for the two launches (the look-back
 * chain costs more than the launch boundary it removes), so the two-launch form stays the default in this package;
 * the entry is kept, parity-tested, for callers that launch kernel by kernel (that case is not measured). */
int rover_mdp_step(const float* new_actions, const float* force_matrix_w, float* root_pos_w, float* root_quat_w,
                   int32_t n_envs, const RoverMdpParams* params, const RoverMdpState* state, const RoverMdpOut* out,
                   const RoverTerrainTables* tables, const int64_t* spawn_perm, const float* yaw_u, const float* heading_u,
                   const float* theta_u, int32_t n_rounds, int64_t* out_spawn_index, float* stats, float* scratch,
                   uint64_t* lookback, float* obs, int32_t obs_stride, int32_t pre_phases, int32_t phases,
                   const struct RoverStatsExchange* xchg /* host, may be NULL; defined below */, void* stream);
/* the same with RoverResetVariates and log_out (see rover_mdp_post_step_v3) */
int rover_mdp_step_v3(const float* new_actions, const float* force_matrix_w, float* root_pos_w, float* root_quat_w,
                      int32_t n_envs, const RoverMdpParams* params, const RoverMdpState* state, const RoverMdpOut* out,
                      const RoverTerrainTables* tables, const RoverResetVariates* variates /* host */,
                      int64_t* out_spawn_index, float* stats, float* scratch, uint64_t* lookback, float* log_out, float* obs,
                      int32_t obs_stride, int32_t pre_phases, int32_t phases, const struct RoverStatsExchange* xchg,
                      void* stream);

/* The WHOLE non-physics step in one launch: rover_mdp_step_v3 (in-kernel variates) + rover_height_scan (variant 5) as one
 * persistent kernel.  One warp of every scan CTA runs the MDP step of the CTA's own environments, 32 at a time and one
 * batch ahead of the scan, and hands each final root pose to the scan's producer warp through shared memory as soon as
 * it is known; the MDP step's latency chain (three dependent cold misses, ~24 us as a launch of its own at 16384 envs)
 * hides behind the scan.  Possible because the in-kernel spawn draw needs no reset rank: an env's step depends on that
 * env only.  Replaces everything RoverEnv.step does outside PhysX (entrypoints/rover_env.py:61-102) when nothing has to
 * run between the action term and the reward terms.
 *   Same state / outputs / tables / rng_state as rover_mdp_step_v3; obs [N, obs_stride] receives the head (columns 0..3)
 *   AND the heights (columns 4 .. 4 + n_rays).  scratch: DEVICE float [scratch_floats >= min(N, #SMs) * 16 + 1], zeroed
 *   once, a buffer of its OWN (not the one passed to rover_mdp_post_step*).  Per-env results are bit-identical to
 *   rover_mdp_step_v3 followed by rover_height_scan; the statistics are summed per CTA instead of per 64-env block
 *   (same values up to fp32 summation order, still deterministic). */
int rover_step_fused(const float* new_actions, const float* force_matrix_w, float* root_pos_w, float* root_quat_w,
                     int32_t n_envs, const RoverMdpParams* params, const RoverMdpState* state, const RoverMdpOut* out,
                     const RoverTerrainTables* tables, uint64_t* rng_state, int32_t n_rounds, int64_t* out_spawn_index,
                     float* stats, float* scratch, int32_t scratch_floats, float* log_out, float* obs, int32_t obs_stride,
                     int32_t pre_phases, int32_t phases, const struct RoverStatsExchange* xchg /* host, may be NULL */,
                     const float* ray_starts_local, int32_t n_rays, const float* pattern_box /* host */,
                     const RoverScanGrid* grid /* host */, const RoverPlaneCells* cells /* host */, float max_distance,
                     float base_offset, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Multi-GPU episode statistics without a collective launch (SURVEY.md 8e: the only cross-rank quantity on the path).
 * Each rank owns a MAILBOX with one slot per rank; the last block of rover_mdp_post_step_x adds the launch's 16
 * statistics to the rank's running totals (fp64) and stores them into its slot of EVERY rank's mailbox -- plain
 * stores over NVLink peer mappings, sequence-numbered -- so the exchange rides on the kernel that produces the
 * numbers (one system-scope fence per step: values into the idle one of two buffers, then the sequence number).
 * rover_stats_read sums the slots in rank order (deterministic) whenever a log line is wanted.
 * Replaces the logging reductions of the ORBIT managers' reset() (consumed at rover_envs/utils/skrl_utils.py:139-142)
 * for env shards on several GPUs; torch.distributed (NCCL) only carries the 64-byte IPC handles once at start-up.
 * ------------------------------------------------------------------------------------------------- */
#define ROVER_MAILBOX_SLOT_BYTES 512 /* uint64 sequence + 2 x 16 doubles (double-buffered), padded */

typedef struct RoverStatsExchange {
    void* const* peer_mailbox; /* DEVICE array [world]: mailbox base of every rank as mapped into this process */
    double* cumulative;        /* DEVICE [16]: this rank's running totals */
    uint64_t* sequence;        /* DEVICE [1]: this rank's sequence counter (even = published) */
    int32_t rank, world;
} RoverStatsExchange;

/* cudaMalloc'ed, zeroed device memory that can be exported to other processes of the node (not from a pooled allocator) */
int rover_p2p_alloc(void** out_ptr, int64_t bytes);
int rover_p2p_free(void* ptr);
int rover_p2p_export(void* ptr, uint8_t handle_out[64]);          /* cudaIpcGetMemHandle */
int rover_p2p_open(const uint8_t handle[64], void** out_ptr);     /* cudaIpcOpenMemHandle (peer access enabled lazily) */
int rover_p2p_close(void* ptr);
/* rover_mdp_post_step plus the publication of the statistics (xchg may be NULL: identical to rover_mdp_post_step) */
int rover_mdp_post_step_x(float* root_pos_w, float* root_quat_w, int32_t n_envs, const RoverMdpParams* params,
                          const RoverMdpState* state, const RoverMdpOut* out, const RoverTerrainTables* tables,
                          const int64_t* spawn_perm, const float* yaw_u, const float* heading_u, const float* theta_u,
                          int32_t n_rounds, int64_t* out_spawn_index, float* stats, float* scratch, float* obs,
                          int32_t obs_stride, int32_t phases, const RoverStatsExchange* xchg /* host */, void* stream);
/* Publish this rank's running totals to every mailbox now (one small launch).  The single-launch step with in-kernel
 * variates (rover_mdp_step_v3 / rover_mdp_step with rng_state) publishes at the START of a launch, from warps that would
 * otherwise idle, the totals as of the PREVIOUS launch -- the two NVLink round trips of a publication then cost the step
 * nothing (they sat between the launch-wide reduction and the end of the kernel: 5 us per step at 2 GPUs) -- so the
 * mailboxes run one launch behind.  For exact totals: rover_stats_publish on every rank, synchronise, barrier, then
 * rover_stats_read.  (The other step entry points publish at the end of each launch, as before.) */
int rover_stats_publish(const struct RoverStatsExchange* xchg /* host */, void* stream);
/* out [16] f64 (device): sum over the world's slots of the local mailbox, in rank order; a slot that is being written is
 * re-read (sequence lock), so every addend is one rank's totals after some whole number of its steps */
int rover_stats_read(const void* mailbox_local, int32_t world, double* out, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Policy forward.  Replaces GaussianNeuralNetwork.compute + HeightmapEncoder
 * (rover_envs/envs/navigation/learning/skrl/models.py:24-36, 89-102) and skrl GaussianMixin.act.
 * Weights are packed once (host -> device) by rover_policy_pack; bf16 operands, fp32 accumulation
 * on the tcgen05 tensor cores.
 * ------------------------------------------------------------------------------------------------- */
typedef struct RoverPolicyWeights {
    const float* w[6];   /* nn.Linear weights [out,in] fp32, order: enc0, enc2, mlp0, mlp2, mlp4, mlp6 */
    const float* b[6];   /* biases */
    int32_t in_dim[6], out_dim[6];  /* out_dim[5] = 2 (policy mean) or 1 (value) */
} RoverPolicyWeights;

/* returns the number of bytes the packed blob needs (when packed == NULL) or packs into it */
int64_t rover_policy_pack(const RoverPolicyWeights* weights /* host struct, device pointers */, void* packed,
                          void* stream);
/* obs [N, obs_stride] fp32 (965 columns used), rows 16-byte aligned (obs_stride % 4 == 0); mean [N,2] fp32 */
int rover_policy_forward(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed, float* mean,
                         void* stream);
/* Value network forward.  Replaces DeterministicNeuralNetwork.compute (models.py:105-162; built by
 * gaussian_model_skrl, configure_models.py:54-64): the same encoder + MLP as the policy with its own weights, one
 * linear output, no tanh.  `packed` comes from rover_policy_pack with out_dim[5] == 1; value [N] fp32. */
int rover_value_forward(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed, float* value,
                        void* stream);
/* Policy AND value network in ONE pass over the observation -- what a PPO rollout evaluates every step (skrl PPO:
 * policy.act in the trainer loop, skrl_utils.py:139-142, value.act in record_transition; models.py:89-102 + :151-162).
 * The observation tile streams through the SM once and meets both heightmap encoders; mean [N,2] and value [N] are
 * bit-identical to rover_policy_forward / rover_value_forward on the same blobs. */
int rover_policy_value_forward(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed_policy,
                               const void* packed_value, float* mean, float* value, void* stream);
/* The same two networks on a bf16 copy of the observation, obs_bf16 [N, stride] (stride % 8 == 0, rows 16-byte
 * aligned; columns 0..963 are read), as rover_height_scan_obs writes it.  A TMA tile of that buffer is the MMA operand
 * as it lands (no conversion stage, half the bytes); results are bit-identical to the fp32 entry points fed with
 * observations that round to the same bf16 values. */
int rover_policy_forward_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed, float* mean,
                              void* stream);
int rover_value_forward_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed, float* value,
                             void* stream);
/* Policy AND value network in ONE pass over the bf16 observation (models.py:89-102 + :151-162, as
 * rover_policy_value_forward): each 64-column tile of obs_bf16 (layout of rover_policy_forward_bf16) meets both
 * heightmap encoders.  mean [N,2] and value [N] are bit-identical to rover_policy_forward_bf16 /
 * rover_value_forward_bf16 on the same blobs, and to rover_policy_value_forward on an fp32 observation that rounds to
 * the same bf16 values. */
int rover_policy_value_forward_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed_policy,
                                    const void* packed_value, float* mean, float* value, void* stream);
/* Height scan FUSED with the heightmap encoder of the policy (or value) network -- BASELINE.json configs[3], "policy
 * forward fused with the observation kernel".  rover_scan_encoder_fused replaces height_scan_rover
 * (mdp/observations.py:35-45, over ORBIT RayCaster / warp raycast) and HeightmapEncoder (learning/skrl/models.py:24-36,
 * called at :95-97) in ONE launch: the 961 heights of an environment go as bf16 from the scan's consumer warps straight
 * into the shared-memory operand of the layer-0 tcgen05.mma -- whose other operand, W0 (80 x 961), stays in tensor
 * memory for the whole launch -- and never make the round trip through L2 / HBM (3844 B/env written + 3860 B/env read
 * back in the unfused pair).  rover_policy_mlp_forward then runs the MLP (64 -> 256 -> 160 -> 128 -> 2 | 1,
 * models.py:97-102 / :151-162) on the encoder output.
 *   obs [N, obs_stride] fp32: columns 0..3 (written by rover_mdp_post_step) are READ; the heights are written to columns
 *     4..964 only when write_obs != 0 (a rollout that records its states needs them; pure inference does not) -- and,
 *     whatever write_obs says, for environments whose table window cannot be staged (they resolve through that row).
 *   packed_fused: image from rover_policy_pack_fused (size query: packed == NULL; layers 0 and 1 of `weights`), 16-byte
 *     aligned.  enc_bf16 [N, 64] bf16, 128-byte aligned: [LeakyReLU encoder output (60), obs[:, 0:4]] per environment.
 *   rover_policy_mlp_forward: `packed` = the blob of rover_policy_pack (its layers 2..5 are read); out [N,2] means
 *     (value_head == 0; tanh applied) or [N] values (value_head != 0, weights packed with out_dim[5] == 1).
 * Needs n_rays == 961, a flat-z pattern and the planar plane-cell table.  Heights (when written) are exactly those of
 * rover_height_scan; the pair's output equals rover_policy_forward's bit for bit (same bf16 operands, same K order;
 * tests/test_gpu_fused_policy.py). */
int64_t rover_policy_pack_fused(const RoverPolicyWeights* weights /* host struct, device pointers */, void* packed,
                                void* stream);
int rover_scan_encoder_fused(const float* pos_w, const float* quat_w, int32_t n_envs, const float* ray_starts_local,
                             int32_t n_rays, const float* pattern_box /* host */, const RoverScanGrid* grid /* host */,
                             const RoverPlaneCells* cells /* host */, float max_distance, float base_offset, float* obs,
                             int32_t obs_stride, int32_t write_obs, const void* packed_fused, uint16_t* enc_bf16,
                             void* stream);
int rover_policy_mlp_forward(const uint16_t* enc_bf16, int32_t n_envs, const void* packed, float* out, int32_t value_head,
                             void* stream);
/* actions = clamp(mean + exp(clamp(log_std,-20,2)) * eps, -1, 1); log_prob [N] = sum_j log N(a_j) */
int rover_gaussian_act(const float* mean, const float* log_std, const float* eps, int32_t n_envs, float* actions,
                       float* log_prob, void* stream);
/* The forward pass with skrl 1.1.0 GaussianMixin.act in its last epilogue (models.py:39-102; SURVEY.md A.4): ONE launch
 * writes mean [N,2] (outputs["mean_actions"]), actions [N,2] and log_prob [N] (NULL: not written), where
 *   eps[i] = normal2({seed, step}, env_offset + i)   (Philox4x32-10 + Box-Muller, csrc/rng.cuh; two N(0,1) per env)
 * and actions / log_prob are what rover_gaussian_act gives for (mean, log_std, eps) -- the same device function, the
 * same bits.  The noise of env i depends on (seed, step, env_offset + i) only: not on n_envs, not on torch's generator.
 *   rng_state: device int64[2] {seed, step}, 8-byte aligned.  The launch reads it after the kernel in front of it has
 *     finished and leaves step + 1 (graph-capturable; step must stay below 2^40 - 1: while the launch runs, bits 40..63
 *     of the step word count its blocks).  Same distribution as torch.randn, not the same numbers (by design).
 *   env_offset >= 0, env_offset + n_envs <= 2^32: the first env's index in the noise stream (a shard of a larger batch).
 *   log_std [2] fp32 (the raw parameter; clamped to [-20, 2] as rover_gaussian_act does).  mean, actions 8-byte aligned.
 * rover_policy_value_act also writes value [N] of the value network, as rover_policy_value_forward does. */
int rover_policy_act(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed, const float* log_std,
                     int64_t* rng_state, int32_t env_offset, float* mean, float* actions, float* log_prob, void* stream);
int rover_policy_act_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed,
                          const float* log_std, int64_t* rng_state, int32_t env_offset, float* mean, float* actions,
                          float* log_prob, void* stream);
int rover_policy_value_act(const float* obs, int32_t obs_stride, int32_t n_envs, const void* packed_policy,
                           const void* packed_value, const float* log_std, int64_t* rng_state, int32_t env_offset,
                           float* mean, float* value, float* actions, float* log_prob, void* stream);
/* rover_policy_value_act on the bf16 observation of rover_policy_value_forward_bf16 (skrl GaussianMixin.act,
 * models.py:39-102, + DeterministicNeuralNetwork.compute, :151-162): one launch, the same noise stream and step
 * advance; mean, value, actions and log_prob equal rover_policy_value_forward_bf16 + rover_gaussian_act fed the eps of
 * rover_action_noise bit for bit. */
int rover_policy_value_act_bf16(const uint16_t* obs_bf16, int32_t stride, int32_t n_envs, const void* packed_policy,
                                const void* packed_value, const float* log_std, int64_t* rng_state, int32_t env_offset,
                                float* mean, float* value, float* actions, float* log_prob, void* stream);
/* The eps [N,2] (8-byte aligned) that the next rover_policy_*act launch with rng_state and env_offset draws, computed on
 * the device with the same code (host libm's log / sin / cos round differently).  advance != 0: the step advances by one
 * as an act launch would; advance == 0 leaves rng_state unchanged.  Feed it to rover_gaussian_act to reproduce an act
 * launch (GaussianMixin.act with explicit noise). */
int rover_action_noise(int64_t* rng_state, int32_t env_offset, int32_t n_envs, float* eps_out, int32_t advance,
                       void* stream);
/* The sampling's functions that are not correctly rounded, evaluated elementwise by the same device code the policy
 * kernels run (test support: an fp32 model of the sampling takes them from here, tests/act_exact.py).  DEVICE f32 arrays
 * of n: ROVER_POLICY_MATH_LOG: out0 = logf(a); ROVER_POLICY_MATH_EXP: out0 = expf(a) (out1 unused, may be NULL);
 * ROVER_POLICY_MATH_SINCOSPI: sincospif(a, out0, out1), out0 = sin(pi a), out1 = cos(pi a).  Asynchronous on `stream`. */
#define ROVER_POLICY_MATH_LOG 0
#define ROVER_POLICY_MATH_EXP 1
#define ROVER_POLICY_MATH_SINCOSPI 2
int rover_policy_math(int32_t op, const float* a, float* out0, float* out1, int32_t n, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * PPO returns and advantages.  Replaces skrl 1.1.0 PPO._update's compute_gae (agents/torch/ppo/ppo.py; third-party,
 * restated in DESIGN.md section 2): the backward loop over the memory_size rows of the rollout memory, returns =
 * advantages + values, then advantages normalised over all T * N entries.
 *   rewards, values [T, n_envs] fp32 and dones [T, n_envs] uint8 (0 = not done), row-major (the memory's [T, N, 1]
 *   tensors); last_values [n_envs]: the value network on the last next_states.  Per environment, i = T-1 .. 0:
 *     adv = (rewards[i] - values[i]) + ((discount_factor * not_done[i]) * (nv + lambda_coefficient * adv)),
 *   nv = values[i+1] (last_values for i = T-1), adv = 0 before the first step, every operation one fp32 rounding (no
 *   contraction; a done step multiplies by 0, it does not branch).  returns = adv + values.  advantages receives
 *   fl32(fl32(adv - mean_f) / fl32(std_f + 1e-8f)) with mean_f = fl32(sum / n), std_f = fl32(sqrt(M2 / (n - 1))) (NaN
 *   for n = 1), sum and M2 = sum (adv - sum / n)^2 accumulated in fp64 in a fixed order: deterministic, graph-capturable.
 *   `work`: device scratch of rover_ppo_gae_work_bytes(T, n_envs) bytes, 8-byte aligned.  Outputs must not overlap the
 *   inputs or each other. */
int64_t rover_ppo_gae_work_bytes(int32_t T, int32_t n_envs);
int rover_ppo_gae(const float* rewards, const uint8_t* dones, const float* values, const float* last_values, int32_t T,
                  int32_t n_envs, float discount_factor, float lambda_coefficient, float* returns, float* advantages,
                  void* work, int64_t work_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Init-time terrain tables (SURVEY.md 8 f-3).  Not on the step path; built once per terrain.
 * rover_mesh_to_heightmap replaces mesh_to_heightmap (rover_envs/utils/terrains/terrain_utils.py:23-57): per face, the
 * cells covered by its XY bounding box take max(cell, max z of the face).  heightmap [rows, cols] fp32 must be
 * pre-filled with -99 (the reference's "no data" value); (min_x, min_y) = mesh bounds shrunk by the 1 m border,
 * (cell_x, cell_y) = (max - min) / grid_size as the reference computes them in fp32.  Indices truncate toward zero,
 * only the upper index is clamped and negative indices wrap once (Python indexing) -- the reference's quirks, kept
 * because the per-step lookups read the table they define.  *out_of_range (device, zeroed by the caller) counts faces
 * whose indices fall beyond the wrap range (the reference raises IndexError there).  Bit-identical: max() does not
 * depend on the visiting order.
 * rover_steep_mask replaces the first stage of find_rocks_in_heightmap (terrain_utils.py:265-279): Sobel gradients
 * with wrap-around borders in float64, steep = |grad| > threshold (uint8 0/1).  The morphological clean-up that follows
 * (:281-311, OpenCV / scipy) stays on the host.
 * ------------------------------------------------------------------------------------------------- */
int rover_mesh_to_heightmap(const float* vertices /* [V,3] */, const int32_t* faces /* [F,3] */, int32_t n_faces,
                            float min_x, float min_y, float cell_x, float cell_y, int32_t rows, int32_t cols,
                            float* heightmap, int32_t* out_of_range, void* stream);
int rover_steep_mask(const float* heightmap, int32_t rows, int32_t cols, double threshold, uint8_t* steep /* [rows, cols] */,
                     void* stream);
/* The morphological clean-up that follows (terrain_utils.py:281-311; OpenCV + scipy in the reference):
 * rover_morph_box = cv2.dilate / cv2.erode with a k x k box of ones on a 0/1 image (anchor k / 2, outside pixels neutral;
 *   MORPH_CLOSE = dilate then erode, MORPH_OPEN = erode then dilate); src, tmp, dst [rows, cols] uint8, all distinct.
 * rover_fill_holes = scipy.ndimage.binary_fill_holes (4-connected background flood from the border); `reach` [rows, cols]
 *   uint8 and `changed` (1 int32) are device scratch.  This call synchronises the stream (it polls for convergence) -- it
 *   is init-time code, not on the step path.  Both reproduce the library results bit for bit
 *   (tests/test_gpu_terrain_build.py). */
int rover_morph_box(const uint8_t* src, int32_t rows, int32_t cols, int32_t k, int32_t erode, uint8_t* tmp, uint8_t* dst,
                    void* stream);
int rover_fill_holes(const uint8_t* mask, int32_t rows, int32_t cols, uint8_t* reach, int32_t* changed, uint8_t* out,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ROVER_B200_H */
