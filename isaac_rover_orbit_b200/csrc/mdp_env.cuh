// Per-environment device functions of the fused MDP step (shared by mdp_step.cu, whose kernels run one thread per env in
// 64-thread blocks, and height_scan_step.cu, where a warp of the persistent scan kernel runs them for the CTA's envs).
// Reference lines restated: see mdp_step.cu.
#pragma once
#include <cstring>

#include "common.cuh"
#include "rng.cuh"

namespace rover {

__device__ __forceinline__ float sgnf(float x) { return (x > 0.f) ? 1.f : ((x < 0.f) ? -1.f : 0.f); }

// torch.remainder(a, 2pi) followed by the (a > pi) fold  (ORBIT wrap_to_pi, A.1)
__device__ __forceinline__ float wrap_to_pi(float a) {
    const float two_pi = 6.2831855f, pi = 3.1415927f;
    float m = fmodf(a, two_pi);
    if (m != 0.f && m < 0.f) m = __fadd_rn(m, two_pi);
    if (m > pi) m = __fsub_rn(m, two_pi);
    return m;
}

struct YawQuat {
    float cw, sz;
};

// ORBIT yaw_quat (A.1)
__device__ __forceinline__ YawQuat yaw_quat(float w, float x, float y, float z) {
    const float siny = __fmul_rn(2.f, __fadd_rn(__fmul_rn(w, z), __fmul_rn(x, y)));
    const float cosy = __fsub_rn(1.f, __fmul_rn(2.f, __fadd_rn(__fmul_rn(y, y), __fmul_rn(z, z))));
    const float half = __fdiv_rn(atan2f(siny, cosy), 2.f);
    const float s = sinf(half), c = cosf(half);
    const float n = fmaxf(sqrtf(__fadd_rn(__fmul_rn(c, c), __fmul_rn(s, s))), 1e-9f);
    return {__fdiv_rn(c, n), __fdiv_rn(s, n)};
}

// ORBIT ArticulationData.heading_w (A.1): atan2 of the rotated x axis
__device__ __forceinline__ float heading_w(float w, float x, float y, float z) {
    const float ty = __fmul_rn(z, 2.f), tz = __fmul_rn(-y, 2.f);  // t = 2 * (xyz x (1,0,0)) = (0, 2z, -2y)
    const float cx = __fsub_rn(__fmul_rn(y, tz), __fmul_rn(z, ty));
    const float cy = __fsub_rn(0.f, __fmul_rn(x, tz));  // z*t.x - x*t.z with t.x = 0
    const float fx = __fadd_rn(1.f, cx);
    const float fy = __fadd_rn(__fmul_rn(w, ty), cy);
    return atan2f(fy, fx);
}

__device__ __forceinline__ float norm2(float x, float y) {
    return sqrtf(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));
}

// contact_sensor force_matrix_w [B,1,3] of one env: L2 norm over bodies per axis, summed over axes, > 1
template <int kBodies>
__device__ __forceinline__ bool collision_active_fixed(const float* __restrict__ f) {
    // all loads are issued before the first use (one memory round trip); accumulation order = body order
    float v[3 * kBodies];
#pragma unroll
    for (int k = 0; k < 3 * kBodies; ++k) v[k] = __ldg(f + k);
    float sx = 0.f, sy = 0.f, sz = 0.f;
#pragma unroll
    for (int b = 0; b < kBodies; ++b) {
        sx = __fadd_rn(sx, __fmul_rn(v[3 * b], v[3 * b]));
        sy = __fadd_rn(sy, __fmul_rn(v[3 * b + 1], v[3 * b + 1]));
        sz = __fadd_rn(sz, __fmul_rn(v[3 * b + 2], v[3 * b + 2]));
    }
    return __fadd_rn(__fadd_rn(sqrtf(sx), sqrtf(sy)), sqrtf(sz)) > 1.f;
}

__device__ __forceinline__ bool collision_active(const float* __restrict__ f, int num_bodies) {
    if (num_bodies == 14) return collision_active_fixed<14>(f);  // AAU rover: 6 Drive + 4 Steer + 3 Boogie + Body
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (int b = 0; b < num_bodies; ++b) {
        const float x = __ldg(f + 3 * b), y = __ldg(f + 3 * b + 1), z = __ldg(f + 3 * b + 2);
        sx = __fadd_rn(sx, __fmul_rn(x, x));
        sy = __fadd_rn(sy, __fmul_rn(y, y));
        sz = __fadd_rn(sz, __fmul_rn(z, z));
    }
    return __fadd_rn(__fadd_rn(sqrtf(sx), sqrtf(sy)), sqrtf(sz)) > 1.f;
}

// ---- AckermannAction2.ackermann (ackermann_actions.py:238-322): jp [FL,RL,RR,FR], jv [ML,FL,RL,RR,MR,FR]
__device__ __forceinline__ void ackermann_v2(const RoverMdpParams& P, float lin_p, float ang_p, float* jp, float* jv) {
    float dir = sgnf(lin_p);
    const float turn = sgnf(ang_p);
    if (dir == 0.f) dir = 1.f;                                                  // :255
    const float v = fabsf(lin_p), w = fabsf(ang_p);
    const bool moving = (w != 0.f) || (v != 0.f);                               // :262
    float R = moving ? __fdiv_rn(v, w) : INFINITY;                              // :265-266 (x/0 = inf)
    const float r_min = P.min_radius;                                           // :264
    if (R < r_min) R = r_min;                                                   // :267
    const float half_mw = P.middle_wheel_distance / 2.f, half_fr = P.rear_and_front_wheel_distance / 2.f;
    const float r_ml = __fsub_rn(R, half_mw), r_mr = __fadd_rn(R, half_mw);     // :271-272
    const float r_l = __fsub_rn(R, half_fr), r_r = __fadd_rn(R, half_fr);       // :273-276
    const bool point = R < P.middle_wheel_distance;                             // :278
    const float spin = __fmul_rn(__fadd_rn(v, 1.f), turn);
    const float v_l = point ? -spin : __fmul_rn((w == 0.f) ? v : __fmul_rn(r_l, w), dir);
    const float v_r = point ? spin : __fmul_rn((w == 0.f) ? v : __fmul_rn(r_r, w), dir);
    const float v_ml = point ? -spin : __fmul_rn((w == 0.f) ? v : __fmul_rn(r_ml, w), dir);
    const float v_mr = point ? spin : __fmul_rn((w == 0.f) ? v : __fmul_rn(r_mr, w), dir);
    const float ack = __fmul_rn(atan2f(P.wheelbase_length, r_l), turn);         // :305 (FL radius for all four)
    const float q = 0.78539816339744830962f;
    jv[0] = __fdiv_rn(v_ml, P.wheel_radius);                                    // [ML,FL,RL,RR,MR,FR] :316
    jv[1] = __fdiv_rn(v_l, P.wheel_radius);
    jv[2] = __fdiv_rn(v_l, P.wheel_radius);
    jv[3] = __fdiv_rn(v_r, P.wheel_radius);
    jv[4] = __fdiv_rn(v_mr, P.wheel_radius);
    jv[5] = __fdiv_rn(v_r, P.wheel_radius);
    jp[0] = point ? -q : ack;                                                   // [FL,RL,RR,FR] :317
    jp[1] = point ? q : ack;
    jp[2] = point ? -q : ack;
    jp[3] = point ? q : ack;
}

// ---- AckermannAction.ackermann (ackermann_actions.py:91-158): jp [FL,FR,RL,RR], jv [FL,FR,ML,MR,RL,RR]
__device__ __forceinline__ void ackermann_v1(float lin, float ang, float* jp, float* jv) {
    const float wx[6] = {-0.385f, 0.385f, -0.447f, 0.447f, -0.385f, 0.385f};    // :97-108 (x right, y forward)
    const float wy[6] = {0.438f, 0.438f, 0.f, 0.f, -0.411f, -0.411f};
    float p = copysignf(__fdiv_rn(lin, ang), -ang);                             // :117-118
    p = (fabsf(p) > 0.45f) ? p : 0.f;                                           // :122
    const float lin2 = (p != 0.f) ? lin : 0.f;                                  // :123
    const float w_lin = copysignf(ang, lin2);                                   // :134
    float steer[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const float dx = __fsub_rn(p, wx[k]), dy = __fsub_rn(0.f, wy[k]);
        const float dist = sqrtf(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));   // :127
        const float side = (k & 1) ? 1.f : -1.f;                                // :130-131
        const float av = (lin2 != 0.f) ? w_lin : __fmul_rn(ang, side);          // :136-137
        float vel = __fmul_rn(dist, av);                                        // :141
        vel = (dist > 1000.f) ? lin2 : vel;                                     // :144
        jv[k] = __fdiv_rn(vel, 0.2f);                                           // :147
        float s = atan2f(wy[k], __fsub_rn(wx[k], p));                           // :149-154
        if (s < -1.57f) s = __fadd_rn(s, 3.1415927f);                           // :155
        if (s > 1.57f) s = __fsub_rn(s, 3.1415927f);                            // :156
        steer[k] = s;
    }
    jp[0] = steer[0];                                                           // :158
    jp[1] = steer[1];
    jp[2] = steer[4];
    jp[3] = steer[5];
}

// ---- ackermann() used by AckermannAction3 (ackermann_actions.py:423-505): jp [FL,FR,RL,RR], jv [FL,FR,ML,MR,RL,RR]
__device__ __forceinline__ void ackermann_v3(const RoverMdpParams& P, float lin_p, float ang_p, float* jp, float* jv) {
    float dir = sgnf(lin_p);
    const float turn = sgnf(ang_p);
    if (dir == 0.f) dir = 1.f;
    const float v = fabsf(lin_p), w = fabsf(ang_p);
    const bool moving = (w != 0.f) || (v != 0.f);
    const float R = moving ? __fdiv_rn(v, w) : INFINITY;                        // :443-444 (no clamp, :445)
    const float hm = __fmul_rn(P.middle_wheel_distance / 2.f, turn), hf = __fmul_rn(P.rear_and_front_wheel_distance / 2.f, turn);
    const float r_ml = __fsub_rn(R, hm), r_mr = __fadd_rn(R, hm);               // :449-450
    const float r_l = __fsub_rn(R, hf), r_r = __fadd_rn(R, hf);                 // :451-454
    const bool point = R < P.min_radius;                                        // :461
    const float spin = __fmul_rn(__fadd_rn(v, 1.f), turn);
    const float v_l = point ? -spin : __fmul_rn((w == 0.f) ? v : __fmul_rn(r_l, w), dir);
    const float v_r = point ? spin : __fmul_rn((w == 0.f) ? v : __fmul_rn(r_r, w), dir);
    const float v_ml = point ? -spin : __fmul_rn((w == 0.f) ? v : __fmul_rn(r_ml, w), dir);
    const float v_mr = point ? spin : __fmul_rn((w == 0.f) ? v : __fmul_rn(r_mr, w), dir);
    const float half_wl = P.wheelbase_length / 2.f;
    const float y_front = __fsub_rn(half_wl, P.offset_lin), y_rear = __fadd_rn(half_wl, P.offset_lin);  // :488-497
    const float q = 0.78539816339744830962f;
    jp[0] = point ? -q : __fmul_rn(atan2f(y_front, r_l), turn);                 // FL
    jp[1] = point ? q : __fmul_rn(atan2f(y_front, r_r), turn);                  // FR
    jp[2] = point ? q : __fmul_rn(atan2f(y_rear, r_l), -turn);                  // RL
    jp[3] = point ? -q : __fmul_rn(atan2f(y_rear, r_r), -turn);                 // RR
    const float diam = P.wheel_diameter;                                        // :503 (float)(wheel_radius * 2)
    jv[0] = __fdiv_rn(v_l, diam);
    jv[1] = __fdiv_rn(v_r, diam);
    jv[2] = __fdiv_rn(v_ml, diam);
    jv[3] = __fdiv_rn(v_mr, diam);
    jv[4] = __fdiv_rn(v_l, diam);
    jv[5] = __fdiv_rn(v_r, diam);
}

__device__ __forceinline__ void ackermann_dispatch(const RoverMdpParams& P, float lin_p, float ang_p, float* jp, float* jv) {
    if (P.action_variant == 1) ackermann_v1(lin_p, ang_p, jp, jv);
    else if (P.action_variant == 3) ackermann_v3(P, lin_p, ang_p, jp, jv);
    else ackermann_v2(P, lin_p, ang_p, jp, jv);
}

// collision_active on values already in registers (the AAU rover's 14 bodies); accumulation order = body order
template <int kBodies>
__device__ __forceinline__ bool collision_active_regs(const float (&v)[3 * kBodies]) {
    float sx = 0.f, sy = 0.f, sz = 0.f;
#pragma unroll
    for (int b = 0; b < kBodies; ++b) {
        sx = __fadd_rn(sx, __fmul_rn(v[3 * b], v[3 * b]));
        sy = __fadd_rn(sy, __fmul_rn(v[3 * b + 1], v[3 * b + 1]));
        sz = __fadd_rn(sz, __fmul_rn(v[3 * b + 2], v[3 * b + 2]));
    }
    return __fadd_rn(__fadd_rn(sqrtf(sx), sqrtf(sy)), sqrtf(sz)) > 1.f;
}

struct NoMidHook {
    __device__ __forceinline__ void operator()() const {}
};

// The per-env work of the pre-step (one thread per env); returns the env's reset flag.
// The step is bound by the latency of ONE warp's dependent chain, so the function is laid out for that: every global
// load of the env is issued first (the compiler cannot hoist loads over the stores in between -- each late load was
// another L2 round trip in the chain), then the action term's kinematics, then `mid()` -- a hook in which the caller
// may start loads of its own that the rest of the pre-step hides (the fused step: variate state -> spawn row) -- then
// terminations and rewards.
// kParts: kPreState = action-manager shift + terminations + rewards, kPreKinematics = the action term's kinematics (a
// pure function of the new action: the single-launch step gives it to a second warp, off the env's critical path).
constexpr int kPreState = 1, kPreKinematics = 2, kPreAll = 3;
struct NoResetHook {
    __device__ __forceinline__ void operator()(bool) const {}
};

// on_reset(reset) is called by every thread (also those without an env) as soon as the env's reset decision exists --
// after the terminations, before the rewards.
template <int kParts = kPreAll, class Mid = NoMidHook, class OnReset = NoResetHook>
__device__ __forceinline__ bool pre_step_env(int i, const float* __restrict__ new_actions, const float* __restrict__ force,
                                             int n, const RoverMdpParams& P, const RoverMdpState& S, const RoverMdpOut& O,
                                             int phases, Mid mid = Mid(), OnReset on_reset = OnReset()) {
    constexpr int kFixedBodies = 14;  // AAU rover: 6 Drive + 4 Steer + 3 Boogie + Body
    const bool valid = i < n;
    const bool terms = valid && (phases & ROVER_PRE_TERMS) && (kParts & kPreState);
    const bool fixed_bodies = P.num_bodies == kFixedBodies;
    bool reset = false;
    // ---- loads
    float2 a_old = make_float2(0.f, 0.f), a = a_old;
    long long ep = 0;
    float bx = 0.f, by = 0.f;
    float fv[3 * kFixedBodies];
    float sums_in[ROVER_NUM_REWARD_TERMS];
    if (valid) {
        if (phases & ROVER_PRE_ACTIONS) {
            if (kParts & kPreState) a_old = reinterpret_cast<const float2*>(S.action)[i];
            a = reinterpret_cast<const float2*>(new_actions)[i];
        } else if (kParts & kPreState) {
            a = reinterpret_cast<const float2*>(S.action)[i];
            a_old = reinterpret_cast<const float2*>(S.prev_action)[i];
        }
    }
    if (terms) {
        ep = S.episode_length_buf[i] + 1;
        bx = S.pos_cmd_b[3 * (size_t)i], by = S.pos_cmd_b[3 * (size_t)i + 1];
        if (fixed_bodies) {
            const float* f = force + (size_t)i * kFixedBodies * 3;
#pragma unroll
            for (int k = 0; k < 3 * kFixedBodies; ++k) fv[k] = __ldg(f + k);
        }
        const float* sums = S.episode_sums + ROVER_NUM_REWARD_TERMS * (size_t)i;
#pragma unroll
        for (int k = 0; k < ROVER_NUM_REWARD_TERMS; ++k) sums_in[k] = sums[k];
    }
    if (valid && (phases & ROVER_PRE_ACTIONS)) {
        // ---- ActionManager.process_action: prev <- action <- new; term.process_actions (ackermann_actions.py:226-229)
        if (kParts & kPreState) {
            reinterpret_cast<float2*>(S.prev_action)[i] = a_old;
            reinterpret_cast<float2*>(S.action)[i] = a;
        }
        if (kParts & kPreKinematics) {
            const float lin_p = __fadd_rn(__fmul_rn(a.x, P.scale_lin), P.offset_lin);
            const float ang_p = __fadd_rn(__fmul_rn(a.y, P.scale_ang), P.offset_ang);
            reinterpret_cast<float2*>(O.processed_actions)[i] = make_float2(lin_p, ang_p);

            ackermann_dispatch(P, lin_p, ang_p, O.joint_pos + 4 * (size_t)i, O.joint_vel + 6 * (size_t)i);
        }
    }
    mid();
    float d = 0.f, ang = 0.f;
    bool coll = false, t_succ = false, t_far = false;
    const float max_len = (float)P.max_episode_length;
    if (terms) {
        // ---- counters (rover_env.py:79)
        S.episode_length_buf[i] = ep;

        // ---- shared quantities of the PREVIOUS command (rover_env.py:82-86 run before the command update)
        d = norm2(bx, by);
        coll = fixed_bodies ? collision_active_regs<kFixedBodies>(fv)
                            : collision_active(force + (size_t)i * P.num_bodies * 3, P.num_bodies);

        // ---- terminations (terminations.py:14-64, ORBIT mdp.time_out)
        const bool t_out = ep >= (long long)P.max_episode_length;
        t_succ = d < P.reached_threshold;
        t_far = d > P.far_threshold;
        const bool terminated = t_succ || t_far || coll;
        reset = t_out || terminated;
        O.terminated[i] = terminated;
        O.truncated[i] = t_out;
        reinterpret_cast<uchar4*>(O.term_flags)[i] = make_uchar4(t_out, t_succ, t_far, coll);
        O.reset_flags[i] = reset;
    }
    on_reset(reset);
    if (terms) {
        ang = atan2f(by, bx);
        // ---- rewards (rewards.py:14-137), RewardManager: value * weight * dt, summed in declaration order
        float val[ROVER_NUM_REWARD_TERMS];
        val[0] = __fdiv_rn(__fdiv_rn(1.f, __fadd_rn(1.f, __fmul_rn(__fmul_rn(0.11f, d), d))), max_len);
        val[1] = t_succ ? __fdiv_rn((float)((long long)P.max_episode_length - ep), max_len) : 0.f;
        {
            const float d_lin = __fmul_rn(__fsub_rn(a.y, a_old.y), 3.f);
            const float d_ang = __fmul_rn(__fsub_rn(a.x, a_old.x), 3.f);
            float p_ang = (d_ang > 0.05f) ? __fmul_rn(d_ang, d_ang) : 0.f;
            float p_lin = (d_lin > 0.05f) ? __fmul_rn(d_lin, d_lin) : 0.f;
            p_ang = __fmul_rn(p_ang, p_ang);
            p_lin = __fmul_rn(p_lin, p_lin);
            val[2] = __fdiv_rn(__fadd_rn(p_ang, p_lin), max_len);
        }
        val[3] = (fabsf(ang) > 2.f) ? __fdiv_rn(fabsf(ang), max_len) : 0.f;
        val[4] = (a.x < 0.f) ? (float)(1.0 / (double)P.max_episode_length) : 0.f;
        val[5] = coll ? 1.f : 0.f;
        val[6] = t_far ? 1.f : 0.f;
        float total = 0.f;
        float* sums = S.episode_sums + ROVER_NUM_REWARD_TERMS * (size_t)i;
        float* tr = O.term_rewards + ROVER_NUM_REWARD_TERMS * (size_t)i;
        float* tv = O.term_values + ROVER_NUM_REWARD_TERMS * (size_t)i;
#pragma unroll
        for (int k = 0; k < ROVER_NUM_REWARD_TERMS; ++k) {
            const float c = __fmul_rn(__fmul_rn(val[k], P.weight[k]), P.step_dt);
            total = __fadd_rn(total, c);
            sums[k] = __fadd_rn(sums_in[k], c);
            tr[k] = c;
            tv[k] = val[k];
        }
        O.reward[i] = total;
    }
    return reset;
}

// --------------------------------------------------------------------------------------------------------------

struct Tables {
    const float* __restrict__ heightmap;
    const uint8_t* __restrict__ safe_mask;
    int H, W;
    float offx, offy, res;
    const float* __restrict__ spawn;
    int n_spawns;
};

// terrain_utils.py:75-81 / :211-218: cell = trunc(xy / res + (min_x, min_y)), clamped (offset ADDED, sic)
__device__ __forceinline__ void terrain_cell(const Tables& T, float x, float y, int& col, int& row) {
    const float sx = __fadd_rn(__fdiv_rn(x, T.res), T.offx);
    const float sy = __fadd_rn(__fdiv_rn(y, T.res), T.offy);
    // .long() truncates toward zero, then clamp(0, W - 1): truncation is monotone and the bounds are integers, so
    // clamping the float first gives the same cell (NaN -> 0 either way) without 64-bit integer min / max
    col = (int)fminf(fmaxf(sx, 0.f), (float)(T.W - 1));
    row = (int)fminf(fmaxf(sy, 0.f), (float)(T.H - 1));
}

// CommandTerm._resample + _resample_command + sample_new_targets (terrain_importer.py:74-95, 134-175).
// The reference's rejection loop is sequential (one host sync per round).  Here it is WARP-COOPERATIVE: the few envs of
// a warp that resample this step (~5 %: 1.6 per warp) are served four at a time, eight lanes per env, lane k of a group
// evaluating round r0 + k -- its variate, sin / cos, the terrain cell, the mask byte and (speculatively) the height
// under the candidate -- so a warp pays ONE candidate's instruction chain and one memory round trip per pass instead of
// eight unrolled candidates in every lane's instruction stream (that was 40 % of the step kernel's instructions).  The
// first valid round wins, else the last one tried: the same candidate the sequential loop accepts.
// The random variates of the reset path: explicit arrays (parity tests: oracle and kernel read the same numbers) or the
// counter-based generator of rng.cuh evaluated in registers (rng != nullptr: {seed, step} in device memory, the step
// counter advanced by the launch itself, so the launch can sit in a CUDA graph).
struct VariatesDev {
    const long long* __restrict__ spawn_perm;
    const float* __restrict__ yaw_u;
    const float* __restrict__ heading_u;
    const float* __restrict__ theta_u;
    unsigned long long* rng;
    int n_rounds;
};

// Must be called by all 32 lanes of a converged warp.  need: this lane's env resamples around (ox, oy).  Lanes with
// `need` get the accepted candidate in (cx, cy, cz) and return true if every round was rejected.
// A pass serves the four lowest pending envs, eight lanes per env, lane k of a group evaluating round r0 + k; an env whose
// eight candidates were all rejected goes on to rounds r0 + 8 .. in the next batch.  (kPer = 4 -- eight envs per pass, four
// rounds each -- was measured slower, 71.4 against 70.6 us for the cfg-3 step: an env that needs a fifth round then pays
// a second cold miss, and on the bench terrain some block of every launch holds one.)
template <bool kRng>
__device__ __forceinline__ bool resample_warp(int i, bool need, const RoverMdpParams& P, const Tables& T, float ox, float oy,
                                              const float* __restrict__ theta_u, const RngKey& key, int n_rounds,
                                              float& cx, float& cy, float& cz) {
    constexpr unsigned kFull = 0xffffffffu;
    constexpr int kPer = 8, kGroups = 32 / kPer;  // rounds (= lanes) per env and envs per pass
    const float pi_f = 3.1415927f;  // torch.pi as fp32; the reference computes rand * 2 * pi left to right
    const unsigned lane = threadIdx.x & 31u;
    const unsigned grp = lane / kPer, k = lane % kPer;
    bool bad = need;
    for (int r0 = 0; r0 < n_rounds; r0 += kPer) {
        unsigned pending = __ballot_sync(kFull, bad);
        while (pending) {
            // owners of this pass: the lowest lanes still pending; group g serves the g-th of them
            unsigned rest = pending;
            int owner = -1;
#pragma unroll
            for (unsigned g = 0; g < (unsigned)kGroups; ++g) {
                const int b = rest ? __ffs(rest) - 1 : -1;
                if (g == grp) owner = b;
                rest &= rest - 1u;
            }
            const bool active = owner >= 0 && r0 + (int)k < n_rounds;
            const int src = owner >= 0 ? owner : (int)lane;
            const int si = __shfl_sync(kFull, i, src);
            const float sox = __shfl_sync(kFull, ox, src), soy = __shfl_sync(kFull, oy, src);
            float xk = 0.f, yk = 0.f, zk = 0.f;
            bool good = false;
            if (active) {
                float u;
                if (kRng) {  // rounds 4q .. 4q+3 = Philox stream 1 + q of the env
                    uint32_t w[4];
                    rng_env_stream(key, (uint32_t)si, 1u + (uint32_t)(r0 + (int)k) / 4u, w);
                    const uint32_t lo = (k & 1u) ? w[1] : w[0], hi = (k & 1u) ? w[3] : w[2];
                    u = u01((k & 2u) ? hi : lo);
                } else {
                    u = __ldg(theta_u + (size_t)si * n_rounds + r0 + (int)k);
                }
                const float th = __fmul_rn(__fmul_rn(u, 2.f), pi_f);                  // :169
                xk = __fadd_rn(__fmul_rn(cosf(th), P.target_distance), sox);          // :172
                yk = __fadd_rn(__fmul_rn(sinf(th), P.target_distance), soy);          // :173
                int col, row;
                terrain_cell(T, xk, yk, col, row);
                const uint8_t m = __ldg(T.safe_mask + (size_t)row * T.W + col);       // :220
                zk = __ldg(T.heightmap + (size_t)row * T.W + col);                    // :154, used if this round wins
                good = m != 1;
            }
            const unsigned good_b = __ballot_sync(kFull, good), act_b = __ballot_sync(kFull, active);
            // an owner finds its group: the number of pending lanes below it
            const unsigned my_g = (unsigned)__popc(pending & ((1u << lane) - 1u));
            const bool served = ((pending >> lane) & 1u) != 0u && my_g < (unsigned)kGroups;  // (a lane served earlier may still be `bad`)
            const unsigned sh = served ? (unsigned)kPer * my_g : 0u;
            const unsigned g_good = (good_b >> sh) & ((1u << kPer) - 1u), g_act = (act_b >> sh) & ((1u << kPer) - 1u);
            const int pick = g_good ? __ffs(g_good) - 1 : 31 - __clz(g_act | 1u);  // first valid round, else the last tried
            const int from = served ? (int)sh + pick : (int)lane;
            const float nx = __shfl_sync(kFull, xk, from), ny = __shfl_sync(kFull, yk, from), nz = __shfl_sync(kFull, zk, from);
            if (served) {
                cx = nx, cy = ny, cz = nz;                                            // :154 (+ default_root_state z = 0)
                bad = g_good == 0u;
            }
            pending = rest;
        }
    }
    return bad;
}

constexpr int kStats = ROVER_STATS_LEN;

struct StatsExchangeDev {
    void* const* peer_mailbox;
    double* cumulative;
    unsigned long long* sequence;
    int rank, world;  // world == 0: no exchange
};

// Sum of each of the 16 statistics over the 32 lanes of a warp, written to out[0..15].  Transposing reduction: every
// butterfly stage halves the number of values a lane still carries (8 + 4 + 2 + 1 + 1 = 16 shuffles instead of 16 x 5),
// a fixed summation tree (deterministic).  Only envs that reset or re-drew their target contribute, so most lanes hold
// zeros and a warp without such an env skips the shuffles.
__device__ __forceinline__ void warp_stats_reduce(float (&st)[kStats], int lane, float* __restrict__ out) {
    static_assert(kStats == 16, "reduction layout");
    constexpr unsigned kFull = 0xffffffffu;
    bool any = false;
#pragma unroll
    for (int k = 0; k < kStats; ++k) any |= st[k] != 0.f;
    if (__ballot_sync(kFull, any) == 0u) {
        if (lane < kStats) out[lane] = 0.f;
        return;
    }
#pragma unroll
    for (int width = 8; width >= 1; width >>= 1) {  // lanes' bit (4, 3, 2, 1) picks the half it keeps
        const bool up = (lane & (2 * width)) != 0;
#pragma unroll
        for (int j = 0; j < width; ++j) {
            const float send = up ? st[j] : st[j + width], keep = up ? st[j + width] : st[j];
            st[j] = keep + __shfl_xor_sync(kFull, send, 2 * width);
        }
    }
    st[0] += __shfl_xor_sync(kFull, st[0], 1);
    if ((lane & 1) == 0) out[lane >> 1] = st[0];  // statistic index = lane bits 4..1
}

// look-back descriptor of the fused step: [epoch : 30 | status : 2 | value : 32]
constexpr unsigned long long kDescAggregate = 1ull, kDescPrefix = 2ull;
__device__ __forceinline__ unsigned long long make_lookback(unsigned epoch, unsigned long long status, unsigned value) {
    return ((unsigned long long)(epoch & 0x3fffffffu) << 34) | (status << 32) | value;
}

// The block-level work of the post-step.  kFused = false: the reset flags and the per-block reset counts come from the
// pre-step launch.  kFused = true (rover_mdp_step): `reset_in` comes from pre_step_env of the same thread and the rank of
// the block's first reset env from a decoupled look-back over the blocks' reset counts (no second launch).
// Per-env registers of the post-step: everything that does not depend on the reset decision is loaded up front, so that a
// launch pays one memory round trip for them instead of one per dependent stage (the step is latency-bound).
struct EnvRegs {
    float px, py, pz, cwx, cwy, cwz, chead, time_left, yaw_var, heading_var;
    float4 q;
    float2 act;
};

template <bool kRng>
__device__ __forceinline__ void post_env_load(int i, bool valid, const float* __restrict__ root_pos_w,
                                              const float* __restrict__ root_quat_w, const RoverMdpState& S,
                                              const VariatesDev& V, EnvRegs& r) {
    r.px = r.py = r.pz = r.cwx = r.cwy = r.cwz = r.chead = r.time_left = r.yaw_var = r.heading_var = 0.f;
    r.q = make_float4(1.f, 0.f, 0.f, 0.f);
    r.act = make_float2(0.f, 0.f);
    if (valid) {
        r.px = root_pos_w[3 * (size_t)i], r.py = root_pos_w[3 * (size_t)i + 1], r.pz = root_pos_w[3 * (size_t)i + 2];
        r.q = reinterpret_cast<const float4*>(root_quat_w)[i];  // (w,x,y,z)
        r.cwx = S.pos_cmd_w[3 * (size_t)i], r.cwy = S.pos_cmd_w[3 * (size_t)i + 1], r.cwz = S.pos_cmd_w[3 * (size_t)i + 2];
        r.chead = S.heading_cmd_w[i];
        r.act = reinterpret_cast<const float2*>(S.action)[i];
        r.time_left = S.time_left[i];
        if (!kRng) {
            r.yaw_var = __ldg(V.yaw_u + i);
            r.heading_var = __ldg(V.heading_u + i);
        }
    }
}

// The per-env work of the post-step (one thread per env): spawn / manager resets / resample / command update /
// observation head; `st` receives the env's contribution to the 16 episode statistics.  On return r.px .. r.q hold the
// env's FINAL root pose (the spawn pose if it reset).
// The spawn row an env WOULD get if it reset this step, fetched before the reset decision exists (fused step, in-kernel
// variates: the row is a function of {seed, step, env} alone).  The chain  rng state -> Philox -> spawn row  -- two cold
// misses -- then runs beside the pre-step instead of behind it; the 95 % of the lanes that do not reset ignore the row.
struct SpawnEarly {
    bool have = false;
    long long idx = -1;
    float x = 0.f, y = 0.f, z = 0.f;
    bool have_variates = false;  // yaw_u / heading_u of the env's variate stream 0 computed by someone else as well
    float yaw_u = 0.f, heading_u = 0.f;
};

// get_target(x, y, z, exhausted) -> true if the env's new target was drawn elsewhere (the split CTA's kinematics warps run
// the rejection sampling beside the env warps); false: post_env_work draws it itself.  Warp-uniform.
struct NoTargetHook {
    __device__ __forceinline__ bool operator()(float&, float&, float&, bool&) const { return false; }
};

struct NoStatsHook {
    __device__ __forceinline__ void operator()(float (&)[kStats]) const {}
};

struct NoPoseHook {
    __device__ __forceinline__ void operator()(float, float, float, const float4&) const {}
};

// on_pose(px, py, pz, q) is called (valid envs only) as soon as the env's FINAL root pose is known -- right after the
// spawn -- so that a consumer of the pose (the height scan fused behind this step, height_scan_step.cu) can start while
// the rest of the env's work (target rejection sampling, command update, stores) is still running.
// on_stats(st) is called by ALL lanes (warp-converged, valid or not) once the env's 16 statistics are final -- after the
// target draw, before metrics / command update / observation head.
template <bool kRng, class OnPose = NoPoseHook, class OnStats = NoStatsHook, class GetTarget = NoTargetHook>
__device__ __forceinline__ void post_env_work(int i, bool valid, bool reset, int rank, EnvRegs& r,
                                              float* __restrict__ root_pos_w, float* __restrict__ root_quat_w,
                                              const RoverMdpParams& P, const RoverMdpState& S, const RoverMdpOut& O,
                                              const Tables& T, const VariatesDev& V, const RngKey& key,
                                              long long* __restrict__ out_spawn_index, float* __restrict__ obs,
                                              int obs_stride, int phases, float (&st)[kStats], OnPose on_pose = OnPose(),
                                              const SpawnEarly early = SpawnEarly(), OnStats on_stats = OnStats(),
                                              GetTarget get_target = GetTarget()) {
    const long long* __restrict__ spawn_perm = V.spawn_perm;
    const float* __restrict__ theta_u = V.theta_u;
    const int n_rounds = V.n_rounds;
    float &px = r.px, &py = r.py, &pz = r.pz, &cwx = r.cwx, &cwy = r.cwy, &cwz = r.cwz, &chead = r.chead;
    float &time_left = r.time_left, &yaw_var = r.yaw_var, &heading_var = r.heading_var;
    float4& q = r.q;
    float2& act = r.act;
#pragma unroll
    for (int k = 0; k < kStats; ++k) st[k] = 0.f;
    long long spawn_idx = -1;
    bool cmd_dirty = false;
    // Which envs draw a new target this step is known up front: a reset env (CommandTerm.reset -> _resample), or one whose
    // timer runs out in CommandManager.compute below.  The two never meet in one env: the reset sets time_left =
    // resampling_time, which the launcher requires to exceed step_dt -- so one cooperative draw serves both, and sharing
    // the env's variates between them is safe.
    const bool rs_reset = valid && reset && (phases & ROVER_PHASE_RESAMPLE);
    const bool rs_timer = valid && !rs_reset && (phases & ROVER_PHASE_TIME) && __fsub_rn(time_left, P.step_dt) <= 0.f;
    float org_x = 0.f, org_y = 0.f;  // env origin of a freshly spawned env stays in registers (no store -> load round trip)
    if (valid) {
        if (kRng && early.have_variates) {
            yaw_var = early.yaw_u, heading_var = early.heading_u;
        } else if (kRng && (reset || rs_timer)) {  // the only envs that consume variates this step
            uint32_t w[4];
            rng_env_stream(key, (uint32_t)i, 0u, w);
            yaw_var = u01(w[0]);
            heading_var = u01(w[1]);
        }
        bool origin_known = false;
        if (reset && (phases & ROVER_PHASE_SPAWN)) {
            // -- reset_root_state_rover (randomizations.py:12-39)
            if (kRng && early.have) {
                spawn_idx = early.idx;
                px = early.x, py = early.y;
                pz = __fadd_rn(early.z, P.spawn_z_offset);
            } else {
                if (kRng) spawn_idx = (long long)spawn_perm_at(make_spawn_perm_key(key, (uint32_t)T.n_spawns), (uint32_t)i);
                else spawn_idx = __ldg(spawn_perm + rank);
                const float* sp = T.spawn + 3 * (size_t)spawn_idx;
                px = __ldg(sp);
                py = __ldg(sp + 1);
                pz = __fadd_rn(__ldg(sp + 2), P.spawn_z_offset);
            }
            const float angle = __fmul_rn(__fmul_rn(yaw_var, 2.f), 3.1415927f);
            const float half = __fdiv_rn(angle, 2.f);
            q = make_float4(cosf(half), 0.f, 0.f, sinf(half));
            org_x = px, org_y = py, origin_known = true;
            S.env_origins[3 * (size_t)i] = px;
            S.env_origins[3 * (size_t)i + 1] = py;
            S.env_origins[3 * (size_t)i + 2] = pz;
            root_pos_w[3 * (size_t)i] = px;
            root_pos_w[3 * (size_t)i + 1] = py;
            root_pos_w[3 * (size_t)i + 2] = pz;
            reinterpret_cast<float4*>(root_quat_w)[i] = q;
        }
        on_pose(px, py, pz, q);
        if ((rs_reset || rs_timer) && !origin_known) {
            org_x = S.env_origins[3 * (size_t)i];
            org_y = S.env_origins[3 * (size_t)i + 1];
        }
    }
    // -- _resample_command around the (new) env origin, all lanes of the warp together
    float nwx = 0.f, nwy = 0.f, nwz = 0.f;
    bool exhausted = false;
    if (!get_target(nwx, nwy, nwz, exhausted))
        exhausted = resample_warp<kRng>(i, rs_reset || rs_timer, P, T, org_x, org_y, theta_u, key, n_rounds, nwx, nwy, nwz);
    if (valid) {
        if (reset && (phases & ROVER_PHASE_MANAGERS)) {
            // -- ActionManager.reset
            act = make_float2(0.f, 0.f);
            reinterpret_cast<float2*>(S.action)[i] = act;
            reinterpret_cast<float2*>(S.prev_action)[i] = act;
            // -- RewardManager.reset: episodic sums of reset envs -> stats, then zero
            float* sums = S.episode_sums + ROVER_NUM_REWARD_TERMS * (size_t)i;
#pragma unroll
            for (int k = 0; k < ROVER_NUM_REWARD_TERMS; ++k) {
                st[k] = sums[k];
                sums[k] = 0.f;
            }
            // -- TerminationManager.reset: per-term counts
            const uchar4 tf = reinterpret_cast<const uchar4*>(O.term_flags)[i];
            st[7] = tf.x;
            st[8] = tf.y;
            st[9] = tf.z;
            st[10] = tf.w;
            // -- CommandTerm.reset: metrics -> stats, zero, counter = 0, then _resample (counter += 1)
            st[11] = S.err_pos[i];
            st[12] = S.err_heading[i];
            st[13] = 1.f;
            S.err_pos[i] = 0.f;
            S.err_heading[i] = 0.f;
            S.command_counter[i] = 0;
            S.episode_length_buf[i] = 0;
        }
        if (rs_reset) {
            // -- CommandTerm._resample: time_left, counter += 1, the new command
            cwx = nwx, cwy = nwy, cwz = nwz;
            chead = __fadd_rn(__fmul_rn(heading_var, __fsub_rn(P.heading_hi, P.heading_lo)), P.heading_lo);  // uniform_(lo, hi)
            st[14] = exhausted ? 1.f : 0.f;
            S.command_counter[i] += 1;
            time_left = P.resampling_time;
            cmd_dirty = true;
        }
        if (rs_timer) {  // (applied below, after the metrics; its statistics are known now)
            st[14] += exhausted ? 1.f : 0.f;
            st[15] = 1.f;
        }
    }
    on_stats(st);
    if (valid) {
        if (out_spawn_index) out_spawn_index[i] = spawn_idx;

        // -- CommandManager.compute(dt): metrics, time_left, time-based resample, _update_command
        const float hw = heading_w(q.x, q.y, q.z, q.w);
        if (phases & ROVER_PHASE_METRICS) {
            const float ex = __fsub_rn(cwx, px), ey = __fsub_rn(cwy, py), ez = __fsub_rn(cwz, pz);
            S.err_pos[i] = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(ez, ez)));
            S.err_heading[i] = fabsf(wrap_to_pi(__fsub_rn(chead, hw)));
        }
        if (phases & ROVER_PHASE_TIME) time_left = __fsub_rn(time_left, P.step_dt);
        if (rs_timer) {  // (time_left <= 0 after the decrement, decided above)
            cwx = nwx, cwy = nwy, cwz = nwz;
            chead = __fadd_rn(__fmul_rn(heading_var, __fsub_rn(P.heading_hi, P.heading_lo)), P.heading_lo);
            S.command_counter[i] += 1;
            time_left = P.resampling_time;
            cmd_dirty = true;
        }
        if (phases & (ROVER_PHASE_TIME | ROVER_PHASE_RESAMPLE)) S.time_left[i] = time_left;
        if (cmd_dirty) {
            S.pos_cmd_w[3 * (size_t)i] = cwx;
            S.pos_cmd_w[3 * (size_t)i + 1] = cwy;
            S.pos_cmd_w[3 * (size_t)i + 2] = cwz;
            S.heading_cmd_w[i] = chead;
        }
        float pbx = S.pos_cmd_b[3 * (size_t)i], pby = S.pos_cmd_b[3 * (size_t)i + 1];
        if (phases & ROVER_PHASE_COMMAND) {
        // _update_command (terrain_importer.py:97-101): quat_rotate_inverse(yaw_quat(q), target - root)
        const float vx = __fsub_rn(cwx, px), vy = __fsub_rn(cwy, py), vz = __fsub_rn(cwz, pz);
        // a - b + c with q_vec = (0, 0, sz): the products with the yaw quaternion's zero x / y components are kept -- they
        // decide the sign of a zero result (pos_cmd_b.z of a level target with |yaw| > pi / 2 is -0 in ORBIT's formula)
        const YawQuat yq = yaw_quat(q.x, q.y, q.z, q.w);
        const float k = __fsub_rn(__fmul_rn(2.f, __fmul_rn(yq.cw, yq.cw)), 1.f);
        const float zx = __fmul_rn(0.f, vx), zy = __fmul_rn(0.f, vy), zz = __fmul_rn(0.f, vz);
        const float b_x = __fmul_rn(__fmul_rn(__fsub_rn(zz, __fmul_rn(yq.sz, vy)), yq.cw), 2.f);
        const float b_y = __fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(yq.sz, vx), zz), yq.cw), 2.f);
        const float b_z = __fmul_rn(__fmul_rn(__fsub_rn(zy, zx), yq.cw), 2.f);
        const float dot = __fadd_rn(__fadd_rn(zx, zy), __fmul_rn(yq.sz, vz));
        const float c_xy = __fmul_rn(__fmul_rn(0.f, dot), 2.f);
        const float c_z = __fmul_rn(__fmul_rn(yq.sz, dot), 2.f);
        pbx = __fadd_rn(__fsub_rn(__fmul_rn(vx, k), b_x), c_xy);
        pby = __fadd_rn(__fsub_rn(__fmul_rn(vy, k), b_y), c_xy);
        const float pbz = __fadd_rn(__fsub_rn(__fmul_rn(vz, k), b_z), c_z);
        S.pos_cmd_b[3 * (size_t)i] = pbx;
        S.pos_cmd_b[3 * (size_t)i + 1] = pby;
        S.pos_cmd_b[3 * (size_t)i + 2] = pbz;
        S.heading_cmd_b[i] = wrap_to_pi(__fsub_rn(chead, hw));
        }

        // -- observation head (rover_env_cfg.py:103-112): last_action, distance * 0.11, angle / pi
        if (obs && (phases & ROVER_PHASE_OBS)) {
            float* o = obs + (size_t)i * obs_stride;
            o[0] = act.x;
            o[1] = act.y;
            o[2] = __fmul_rn(norm2(pbx, pby), P.obs_distance_scale);
            o[3] = __fmul_rn(atan2f(pby, pbx), P.obs_heading_scale);
        }
    }

}

}  // namespace rover
