// quadsim_kernels.cuh -- sm_100a device code of the batched quadrotor-swarm simulator.
//
// One thread owns one drone; the K drones of an environment occupy KG = pow2(K) adjacent lanes of a warp, so every
// cross-drone quantity (pair distances, collision rows, neighbour ranking, downwash, impulses) moves through
// __shfl_sync on the group's lane mask.  State is structure-of-arrays in HBM as float4 planes (one 16-byte vector
// load/store per thread per plane, 512 B per warp, fully coalesced); observations are staged per warp in shared
// memory and leave as 16-byte coalesced stores.  There are no tensor-core instructions: nothing here is a contraction.
//
// The arithmetic restates, in fp32, the reference's per-control-step path; each device function cites the reference
// file:line it follows (paths relative to gym_art/quadrotor_multi/ in priban42/quad-swarm-rl-stable-baselines3).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/quadsim.h"

#define QS_FULL 0xffffffffu
#define QS_PRAGMA_(x) _Pragma(#x)
#define QS_UNROLL(n) QS_PRAGMA_(unroll n)
#ifndef QS_SDF_UNROLL
#define QS_SDF_UNROLL 2         // obstacle-loop iterations in flight (SDF patch + hit test)
#endif
#ifndef QS_DW_UNROLL
#define QS_DW_UNROLL 1          // downwash source-loop iterations in flight
#endif
#ifndef QS_PAIR_UNROLL
#define QS_PAIR_UNROLL 4        // pair-pass iterations in flight
#endif
#ifndef QS_NB_PRED
#define QS_NB_PRED 2            // neighbour row-write iterations in flight (0: the branchy one-at-a-time form)
#endif
#ifndef QS_STEP_MINBLOCKS
#define QS_STEP_MINBLOCKS 4      // resident blocks per SM the step kernel is compiled for (register cap 65536/(threads*n))
#endif
#ifndef QS_STEP_MAXTHREADS
#define QS_STEP_MAXTHREADS 128
#endif
#define QS_PI_F 3.14159265358979323846f

namespace qs {

// ----------------------------------------------------------------------------------------------------------------
// constants and pointers handed to the kernels (by value, __grid_constant__ -> constant bank)
// ----------------------------------------------------------------------------------------------------------------
struct DevConst {
    int N, K, scenario, obs_repr, nbr_type, V, use_obstacles, use_downwash, apply_force, sense_noise;
    int ep_len, sim_steps, svd_period, obst_L, obst_W, M, D, S;   // D obs dim, S self-obs dim
    int small_angle;                                              // sqrt(3) * omega_max * dt / 2 <= 0.25 rad
    int lin_one, no_omega_damp;                                   // motor_linearity == 1 / damp_omega_quadratic == 0: the terms drop out (warp-uniform)
    uint32_t key0, key1;
    uint32_t rng_step;                                            // Philox counter word 1: launches (steps + resets) of the handle so far
    long long env_id_offset;
    float dt, hx, hy, hz, room_l, room_w, room_h, gravity, mass, inv_mass;
    float inertia[3], inv_inertia[3], thrust_max[4], torque_max[4], pcx[4], pcy[4], pcz[4], ccw[4];
    float arm, tau_up, tau_down, lin, vel_damp, damp_wq, omega_max, mu, ou_theta, ou_sigma;
    float s_pos, s_vel, s_gyro;
    float rew_pos, rew_effort, rew_crash, rew_orient, rew_spin, rew_col, rew_col_smooth, rew_col_obst;
    float thr_col, thr_fall, thr_obst, obst_rad, sdf_res;
    float spawn_box, spawn_min_z, approach_metric, grace_steps, final_grace_steps, control_dt;
    float control_freq;                                           // sim_freq / sim_steps (quadrotor_single.py:160)
    int cube_dim[3];                                              // qs_config.cube_dim
};

enum { PL_POS_VX = 0, PL_V_W, PL_W_R0, PL_R1, PL_R2_FLAGS, PL_ROT_DAMP, PL_CMDS_DAMP, PL_OU, PL_GOAL, PL_DIST_RING,
       PL_DIST_SUMS, PL_COUNT };

// per-env counters (int32 each)
enum { EC_COL = 0, EC_COL_SETTLE, EC_COL_FINAL, EC_ROOM, EC_FLOOR, EC_WALL, EC_CEIL, EC_OBST, EC_OBST_SETTLE,
       EC_SCENARIO, EC_COUNT };

struct DevPtrs {
    float4 *plane[PL_COUNT];   // each [N*K]
    int *tick;                 // [N]
    int *svd_ctr;              // [N]
    int *ecnt;                 // [N, EC_COUNT]
    float2 *obst_xy;           // [N, QS_MAX_OBSTACLES]
    float4 *scen;              // [N, QS_SC_COUNT / 4] formation-scenario rows (formation scenarios only, else null)
    int *ep_rec;               // [N, QS_ER_COUNT] record of the last finished episode per env (QS_ER_*)
    float4 *ep_agent;          // [N*K] per-drone part of that record
    // reset-first scheduling (step kernel): warp-tiles whose envs finish their episode in THIS step were listed by the
    // previous step and are processed by the first `hot_blocks` blocks of the grid, so that the long auto-reset path overlaps the
    // rest of the grid instead of extending its tail.  Three buffers rotate: consumed now / produced now / count cleared now.
    int *hot_list_cur, *hot_cnt_cur, *hot_flag_cur;   // flags: one int per warp-tile (set = a hot block owns this tile in this step)
    int *hot_list_next, *hot_cnt_next, *hot_flag_next;
    int *hot_cnt_clear;
    int hot_cap, hot_blocks;
    float4 *rew_info;          // [N*K, 2] optional (null = off): the raw reward terms of the step, infos[i]["rewards"] (QS_RI_*)
    qs_stats *stats;           // device aggregate
};

// flag bits kept in PL_R2_FLAGS.z
enum { F_ON_FLOOR = 1, F_CR_FLOOR = 2, F_CR_WALL = 4, F_CR_CEIL = 8, F_PREV_WALL = 16, F_PREV_CEIL = 32,
       F_PREV_ROOM = 64, F_PREV_OBST = 128, F_REACHED = 256, F_COL_AGENT = 512, F_COL_OBST = 1024,
       // transient (last sub-step): the drone sits exactly on a wall plane (collisions/room.py:14-15 `pos == room_box`)
       F_AT_XLO = 2048, F_AT_XHI = 4096, F_AT_YLO = 8192, F_AT_YHI = 16384,
       // obstacle `mix`: this episode runs o_static_same_goal (else o_random).  Kept per drone in the flag word, which the step kernel
       // loads anyway: as a separate per-env load it was spilled right after the load, which stalled the warp for a whole HBM round
       // trip before the state loads were even issued (ncu, profiles/README.md)
       F_SCEN_OSTATIC = 32768 };

// RNG sites: DESIGN.md "RNG contract" (identical table in oracle/quadsim_oracle.c)
enum { SITE_OU = 0, SITE_SENSOR = 1, SITE_SENSOR_IMPULSE = 2, SITE_SENSOR_RESET = 3, SITE_FLOOR_YAW = 4,
       SITE_PAIR = 5, SITE_OBST = 6, SITE_WALL = 7, SITE_CEILING = 8, SITE_DOWNWASH = 9, SITE_SPAWN = 10,
       SITE_SCENARIO = 11, SITE_CAMERA = 12 };


// ----------------------------------------------------------------------------------------------------------------
// Philox4x32-10, keyed (seed), counter (env gid, step counter, site|drone<<8|aux<<16, block)
// ----------------------------------------------------------------------------------------------------------------
struct Rng {
    uint32_t gid, step, k0, k1;
};

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

__device__ __forceinline__ uint4 rng_block(const Rng &g, int site, int drone, int aux, int block)
{
    uint32_t c2 = (uint32_t)site | ((uint32_t)drone << 8) | ((uint32_t)aux << 16);
    return philox4x32_10(g.gid, g.step, c2, (uint32_t)block, g.k0, g.k1);
}

// ((x >> 9) + 0.5) * 2^-23 : exactly representable in fp32, in (0,1)
__device__ __forceinline__ float u23(uint32_t x) { return fmaf((float)(x >> 9), 1.1920928955078125e-07f, 5.9604644775390625e-08f); }

// Box-Muller on the SFU: lg2.approx / sin.approx / cos.approx (abs error ~2^-21 on the unit draws, i.e. <= 1e-8 after
// scaling by the noise sigmas).  u in (0,1) so the log is finite; the angle is mapped to (-pi, pi) where the
// approximations are tightest: cos(2 pi u) = -cos(pi (2u-1)), sin(2 pi u) = -sin(pi (2u-1)).
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float &n0, float &n1)
{
    float rad = sqrtf(fmaxf(-1.3862943611198906f * __log2f(u23(a)), 0.0f));     // -2 ln u = -2 ln2 log2 u
    float ang = QS_PI_F * fmaf(2.0f, u23(b), -1.0f);
    n0 = -rad * __cosf(ang); n1 = -rad * __sinf(ang);
}

// idx-th uniform of stream (site, drone, aux)
__device__ __forceinline__ float rng_u(const Rng &g, int site, int drone, int aux, int idx)
{
    uint4 r = rng_block(g, site, drone, aux, idx >> 2);
    uint32_t x = (idx & 2) ? ((idx & 1) ? r.w : r.z) : ((idx & 1) ? r.y : r.x);
    return u23(x);
}
__device__ __forceinline__ void rng_u4(const Rng &g, int site, int drone, int aux, int block, float *u)
{
    uint4 r = rng_block(g, site, drone, aux, block);
    u[0] = u23(r.x); u[1] = u23(r.y); u[2] = u23(r.z); u[3] = u23(r.w);
}
__device__ __forceinline__ void rng_n4(const Rng &g, int site, int drone, int aux, int block, float *n)
{
    uint4 r = rng_block(g, site, drone, aux, block);
    box_muller(r.x, r.y, n[0], n[1]);
    box_muller(r.z, r.w, n[2], n[3]);
}

// One Philox block -> 4 standard normals, out of line: the hot path draws 4 blocks per drone-step and four inlined
// copies (~115 instructions each) do not fit the instruction-cache budget of the step kernel.
static __device__ __noinline__ float4 rng_normal4(uint32_t gid, uint32_t step, uint32_t c2, uint32_t block, uint32_t k0, uint32_t k1)
{
    uint4 r = philox4x32_10(gid, step, c2, block, k0, k1);
    float4 n;
    box_muller(r.x, r.y, n.x, n.y);
    box_muller(r.z, r.w, n.z, n.w);
    return n;
}
__device__ __forceinline__ float4 rng_n4v(const Rng &g, int site, int drone, int aux, int block)
{
    return rng_normal4(g.gid, g.step, (uint32_t)site | ((uint32_t)drone << 8) | ((uint32_t)aux << 16), (uint32_t)block, g.k0, g.k1);
}

// ----------------------------------------------------------------------------------------------------------------
// per-drone register state
// ----------------------------------------------------------------------------------------------------------------
struct Drone {
    float p[3], v[3], w[3], R[9], rd[4], cd[4], ou[4], goal[3];
    int flags;
    uint32_t colmask;
};

__device__ __forceinline__ void load_drone(const DevPtrs &P, int gi, Drone &q)
{
    // streamed once per step: keep them out of L1, which then holds the few spilled registers of the kernel
    float4 a = __ldcs(P.plane[PL_POS_VX] + gi), b = __ldcs(P.plane[PL_V_W] + gi), c = __ldcs(P.plane[PL_W_R0] + gi), d = __ldcs(P.plane[PL_R1] + gi),
           e = __ldcs(P.plane[PL_R2_FLAGS] + gi), f = __ldcs(P.plane[PL_ROT_DAMP] + gi), g = __ldcs(P.plane[PL_CMDS_DAMP] + gi),
           h = __ldcs(P.plane[PL_OU] + gi), k = __ldcs(P.plane[PL_GOAL] + gi);
    q.p[0] = a.x; q.p[1] = a.y; q.p[2] = a.z; q.v[0] = a.w; q.v[1] = b.x; q.v[2] = b.y;
    q.w[0] = b.z; q.w[1] = b.w; q.w[2] = c.x;
    q.R[0] = c.y; q.R[1] = c.z; q.R[2] = c.w; q.R[3] = d.x; q.R[4] = d.y; q.R[5] = d.z; q.R[6] = d.w; q.R[7] = e.x; q.R[8] = e.y;
    q.flags = __float_as_int(e.z); q.colmask = __float_as_uint(e.w);
    q.rd[0] = f.x; q.rd[1] = f.y; q.rd[2] = f.z; q.rd[3] = f.w;
    q.cd[0] = g.x; q.cd[1] = g.y; q.cd[2] = g.z; q.cd[3] = g.w;
    q.ou[0] = h.x; q.ou[1] = h.y; q.ou[2] = h.z; q.ou[3] = h.w;
    q.goal[0] = k.x; q.goal[1] = k.y; q.goal[2] = k.z;
}

// the motor-lag (rot_damp, cmds_damp) and thrust-noise planes: final as soon as the dynamics have run
__device__ __forceinline__ void store_motor_planes(const DevPtrs &P, int gi, const Drone &q)
{
    P.plane[PL_ROT_DAMP][gi] = make_float4(q.rd[0], q.rd[1], q.rd[2], q.rd[3]);
    P.plane[PL_CMDS_DAMP][gi] = make_float4(q.cd[0], q.cd[1], q.cd[2], q.cd[3]);
    P.plane[PL_OU][gi] = make_float4(q.ou[0], q.ou[1], q.ou[2], q.ou[3]);
}

template <bool WITH_MOTOR = true>
__device__ __forceinline__ void store_drone(const DevPtrs &P, int gi, const Drone &q, bool store_goal)
{
    P.plane[PL_POS_VX][gi] = make_float4(q.p[0], q.p[1], q.p[2], q.v[0]);
    P.plane[PL_V_W][gi] = make_float4(q.v[1], q.v[2], q.w[0], q.w[1]);
    P.plane[PL_W_R0][gi] = make_float4(q.w[2], q.R[0], q.R[1], q.R[2]);
    P.plane[PL_R1][gi] = make_float4(q.R[3], q.R[4], q.R[5], q.R[6]);
    P.plane[PL_R2_FLAGS][gi] = make_float4(q.R[7], q.R[8], __int_as_float(q.flags), __uint_as_float(q.colmask));
    if (WITH_MOTOR) store_motor_planes(P, gi, q);
    if (store_goal) P.plane[PL_GOAL][gi] = make_float4(q.goal[0], q.goal[1], q.goal[2], 0.0f);
}

__device__ __forceinline__ float clampf(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }
__device__ __forceinline__ float norm3f(float a, float b, float c) { return sqrtf(a * a + b * b + c * c); }

// unit vector (c, s) with angle atan2(y, x); atan2(0,0) = 0 -> (1, 0)
__device__ __forceinline__ void unit_dir(float x, float y, float &c, float &s)
{
    // one reciprocal square root instead of a square root and two divisions: in steady state most drones of a random-action rollout sit on
    // the floor and take this path twice per sub-step (3 % of the step's instructions with the divisions, profiles/README.md round 2)
    const float hh = x * x + y * y;
    if (hh > 0.0f) { const float inv = rsqrtf(hh); c = x * inv; s = y * inv; } else { c = 1.0f; s = 0.0f; }
}
__device__ __forceinline__ void set_yaw(float *R, float c, float s)
{
    R[0] = c; R[1] = -s; R[2] = 0.f; R[3] = s; R[4] = c; R[5] = 0.f; R[6] = 0.f; R[7] = 0.f; R[8] = 1.f;
}

// U V^T of svd(R) == orthogonal polar factor (quadrotor_dynamics.py:556-557): Newton X <- (X + X^-T)/2.
// R is within ~1e-5 of orthonormal after 100 Rodrigues steps, so 3 iterations reach fp32 round-off.
__device__ __forceinline__ void polar_orthonormalise(float *X)
{
#pragma unroll
    for (int it = 0; it < 3; ++it) {
        float c00 = X[4] * X[8] - X[5] * X[7], c01 = X[5] * X[6] - X[3] * X[8], c02 = X[3] * X[7] - X[4] * X[6];
        float c10 = X[2] * X[7] - X[1] * X[8], c11 = X[0] * X[8] - X[2] * X[6], c12 = X[1] * X[6] - X[0] * X[7];
        float c20 = X[1] * X[5] - X[2] * X[4], c21 = X[2] * X[3] - X[0] * X[5], c22 = X[0] * X[4] - X[1] * X[3];
        float id = 1.0f / (X[0] * c00 + X[1] * c01 + X[2] * c02);
        X[0] = 0.5f * (X[0] + c00 * id); X[1] = 0.5f * (X[1] + c01 * id); X[2] = 0.5f * (X[2] + c02 * id);
        X[3] = 0.5f * (X[3] + c10 * id); X[4] = 0.5f * (X[4] + c11 * id); X[5] = 0.5f * (X[5] + c12 * id);
        X[6] = 0.5f * (X[6] + c20 * id); X[7] = 0.5f * (X[7] + c21 * id); X[8] = 0.5f * (X[8] + c22 * id);
    }
}

// ----------------------------------------------------------------------------------------------------------------
// a1-a4  QuadrotorDynamics.step: one physics sub-step (quadrotor_dynamics.py:355-390, 504-656)
// ----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void dynamics_substep(const DevConst &c, const Rng &g, int drone, Drone &q, const float *cmd,
                                                 int substep, bool do_svd)
{
    const float dt = c.dt;
    // motor lag in sqrt-thrust space + OU noise, thrust / torque (:511-540)
    float tq0 = 0.f, tq1 = 0.f, tq2 = 0.f, thrust = 0.f;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        float cm = cmd[m];
        float tau = fminf((cm < q.cd[m]) ? c.tau_down : c.tau_up, 1.0f);
        q.rd[m] = tau * (sqrtf(cm) - q.rd[m]) + q.rd[m];
        float cdm = clampf(q.rd[m] * q.rd[m] + cm * q.ou[m], 0.0f, 1.0f);
        q.cd[m] = cdm;
        float th = c.lin_one ? c.thrust_max[m] * cdm : c.thrust_max[m] * ((1.0f - c.lin) * cdm * cdm + c.lin * cdm);
        tq0 += c.pcx[m] * th; tq1 += c.pcy[m] * th; tq2 += c.pcz[m] * th + c.torque_max[m] * c.ccw[m] * cdm;
        thrust += th;
    }
    // Rodrigues rotation about the world-frame angular velocity (:544-551): R <- exp([R w]x dt) R.  Since exp([R w]x) = R exp([w]x) R^T
    // this is R exp([w]x dt) -- the same matrix, built from the body-frame rate directly (no R w product, |R w| = |w|)
    float wx = q.w[0], wy = q.w[1], wz = q.w[2];
    float wn = norm3f(wx, wy, wz);
    if (wn != 0.0f) {
        float inv = 1.0f / wn, kx = wx * inv, ky = wy * inv, kz = wz * inv;
        float ang = wn * dt, s, ch;
        if (c.small_angle) {
            // |omega| <= sqrt(3) omega_max, so x = ang/2 <= 0.25 rad: degree-9/8 Taylor, truncation < 3e-12
            float x = 0.5f * ang, x2 = x * x;
            s = x * (1.0f + x2 * (-1.0f / 6.0f + x2 * (1.0f / 120.0f + x2 * (-1.0f / 5040.0f + x2 * (1.0f / 362880.0f)))));
            ch = 1.0f + x2 * (-0.5f + x2 * (1.0f / 24.0f + x2 * (-1.0f / 720.0f + x2 * (1.0f / 40320.0f))));
        } else sincosf(0.5f * ang, &s, &ch);
        float sn = 2.0f * s * ch, oc = 2.0f * s * s;               // sin(ang), 1 - cos(ang) without cancellation
        // dR = I + sn*K + oc*K^2,  K^2 = k k^T - I
        float d00 = 1.f + oc * (kx * kx - 1.f), d01 = -sn * kz + oc * kx * ky, d02 = sn * ky + oc * kx * kz;
        float d10 = sn * kz + oc * kx * ky, d11 = 1.f + oc * (ky * ky - 1.f), d12 = -sn * kx + oc * ky * kz;
        float d20 = -sn * ky + oc * kx * kz, d21 = sn * kx + oc * ky * kz, d22 = 1.f + oc * (kz * kz - 1.f);
        float n[9];
#pragma unroll
        for (int i = 0; i < 3; ++i) {                                  // R dR
            n[3 * i] = q.R[3 * i] * d00 + q.R[3 * i + 1] * d10 + q.R[3 * i + 2] * d20;
            n[3 * i + 1] = q.R[3 * i] * d01 + q.R[3 * i + 1] * d11 + q.R[3 * i + 2] * d21;
            n[3 * i + 2] = q.R[3 * i] * d02 + q.R[3 * i + 1] * d12 + q.R[3 * i + 2] * d22;
        }
#pragma unroll
        for (int j = 0; j < 9; ++j) q.R[j] = n[j];
    }
    if (__builtin_expect(do_svd, 0)) polar_orthonormalise(q.R);                           // :554-558
    // omega (:562-567)
    {
        float i0 = c.inertia[0] * q.w[0], i1 = c.inertia[1] * q.w[1], i2 = c.inertia[2] * q.w[2];
        float cr0 = -q.w[1] * i2 + q.w[2] * i1, cr1 = -q.w[2] * i0 + q.w[0] * i2, cr2 = -q.w[0] * i1 + q.w[1] * i0;
        float wd0 = c.inv_inertia[0] * (cr0 + tq0), wd1 = c.inv_inertia[1] * (cr1 + tq1), wd2 = c.inv_inertia[2] * (cr2 + tq2);
        float q0 = 0.f, q1 = 0.f, q2 = 0.f;
        if (!c.no_omega_damp) {
            q0 = clampf(c.damp_wq * q.w[0] * q.w[0], 0.f, 1.f); q1 = clampf(c.damp_wq * q.w[1] * q.w[1], 0.f, 1.f);
            q2 = clampf(c.damp_wq * q.w[2] * q.w[2], 0.f, 1.f);
        }
        q.w[0] = clampf(q.w[0] + (1.f - q0) * dt * wd0, -c.omega_max, c.omega_max);
        q.w[1] = clampf(q.w[1] + (1.f - q1) * dt * wd1, -c.omega_max, c.omega_max);
        q.w[2] = clampf(q.w[2] + (1.f - q2) * dt * wd2, -c.omega_max, c.omega_max);
    }
    // position, room clip and wall / ceiling flags (:570, :367-374).
    // Threshold predicates are evaluated as  dt*v  vs  (bound - p): the difference is exact in fp32 near the bound
    // (Sterbenz), so the decision equals the exact-arithmetic one on the same inputs even when |dt*v| is below the
    // fp32 resolution of p (a drone resting against a wall, or lifting off the floor by 1e-10 m).
    float dx = dt * q.v[0], dy = dt * q.v[1], dz = dt * q.v[2];
    const float gx_hi = c.hx - q.p[0], gx_lo = -c.hx - q.p[0], gy_hi = c.hy - q.p[1], gy_lo = -c.hy - q.p[1], gz_hi = c.hz - q.p[2];
    const bool floor_hit = dz <= (c.arm - q.p[2]);
    int fl = q.flags & ~(F_CR_FLOOR | F_CR_WALL | F_CR_CEIL | F_AT_XLO | F_AT_XHI | F_AT_YLO | F_AT_YHI);
    if (dx > gx_hi || dx < gx_lo || dy > gy_hi || dy < gy_lo) fl |= F_CR_WALL;
    if (dz > gz_hi) fl |= F_CR_CEIL;
    fl |= (dx <= gx_lo ? F_AT_XLO : 0) | (dx >= gx_hi ? F_AT_XHI : 0) | (dy <= gy_lo ? F_AT_YLO : 0) | (dy >= gy_hi ? F_AT_YHI : 0);
    q.p[0] = clampf(q.p[0] + dx, -c.hx, c.hx); q.p[1] = clampf(q.p[1] + dy, -c.hy, c.hy); q.p[2] = clampf(q.p[2] + dz, 0.0f, c.hz);
    // floor_interaction_numba (:576-646), floor threshold = arm (:385)
    float fx = q.R[2] * thrust, fy = q.R[5] * thrust, fz = q.R[8] * thrust;   // R @ [0,0,T], old R
    float ax, ay, az;
    if (floor_hit) {
        q.p[2] = c.arm;
        if (fl & F_ON_FLOOR) {
            float cy, sy;
            unit_dir(q.R[0] + 1e-6f, q.R[3], cy, sy);
            set_yaw(q.R, cy, sy);
            float fr = c.mu * (c.mass * 9.81f - fz);
            if (q.v[0] * q.v[0] + q.v[1] * q.v[1] + q.v[2] * q.v[2] < 1e-12f) {      // |v| < 1e-6 (:601)
                float fm = sqrtf(fx * fx + fy * fy);
                float fn = fmaxf(fm - fr, 0.0f);
                if (fn == 0.0f) { fx = 0.f; fy = 0.f; }
                else { float cf, sf; unit_dir(fx, fy, cf, sf); fx = fn * cf; fy = fn * sf; }
            } else {
                float cf, sf;
                unit_dir(q.v[0], q.v[1], cf, sf);                    // :608 numba path: friction opposes velocity
                fx -= cf * fr; fy -= sf * fr;
            }
        } else {
            fl |= F_ON_FLOOR | F_CR_FLOOR;
            q.v[0] = q.v[1] = q.v[2] = 0.f; q.w[0] = q.w[1] = q.w[2] = 0.f;
            float cy, sy;
            if (q.R[8] < 0.f) {                                      // :623-626 upside down -> random yaw
                float th = -1.0f + 2.0f * rng_u(g, SITE_FLOOR_YAW, drone, substep, 0);
                sincospif(th, &sy, &cy);
            } else {
                unit_dir(q.R[0] + 1e-6f, q.R[3], cy, sy);
            }
            set_yaw(q.R, cy, sy);
#pragma unroll
            for (int m = 0; m < 4; ++m) { q.cd[m] = 0.f; q.rd[m] = 0.f; }
        }
        ax = fx * c.inv_mass; ay = fy * c.inv_mass; az = fmaxf(0.0f, -9.81f + fz * c.inv_mass);
    } else {
        fl &= ~F_ON_FLOOR;
        ax = fx * c.inv_mass; ay = fy * c.inv_mass; az = -9.81f + fz * c.inv_mass;
    }
    q.flags = fl;
    // compute_velocity_and_acceleration (:649-656); the accelerometer output never reaches an observation
    float kd = 1.0f - c.vel_damp;
    q.v[0] = kd * q.v[0] + dt * ax; q.v[1] = kd * q.v[1] + dt * ay; q.v[2] = kd * q.v[2] + dt * az;
}

// ----------------------------------------------------------------------------------------------------------------
// a9  self observation: SensorNoise.add_noise_numba + state_xyz_vxyz_R_omega* (sensor_noise.py:172-261, get_state.py:226-292)
// ----------------------------------------------------------------------------------------------------------------
// the three noise blocks of one self observation (9 of the 12 normals are used)
struct SensorNoise { float4 n, m, l; };
__device__ __forceinline__ SensorNoise sensor_noise(const Rng &g, int site, int drone)
{
    SensorNoise s;
    s.n = rng_n4v(g, site, drone, 0, 0); s.m = rng_n4v(g, site, drone, 0, 1); s.l = rng_n4v(g, site, drone, 0, 2);
    return s;
}

__device__ __forceinline__ void self_obs(const DevConst &c, const SensorNoise &sn, const Drone &q, float *o)
{
    float p0 = q.p[0], p1 = q.p[1], p2 = q.p[2], v0 = q.v[0], v1 = q.v[1], v2 = q.v[2], w0 = q.w[0], w1 = q.w[1], w2 = q.w[2];
    if (c.sense_noise) {
        const float4 n = sn.n, m = sn.m, l = sn.l;
        p0 += c.s_pos * n.x; p1 += c.s_pos * n.y; p2 += c.s_pos * n.z;
        v0 += c.s_vel * n.w; v1 += c.s_vel * m.x; v2 += c.s_vel * m.y;
        w0 += c.s_gyro * m.z; w1 += c.s_gyro * m.w; w2 += c.s_gyro * l.x;
        // R -> quaternion -> R round trip with zero rotation noise (sensor_noise.py:34-63, 205-210; quad_utils.py:162-168): the identity
        // on rotation matrices.  In the float64 reference it returns R to 1e-16; evaluated literally in fp32 it only adds round-off
        // (~3e-7) on top of R, so the observation carries R itself (closer to the reference than the literal form, and ~50
        // instructions + 2 SFU operations less per drone-step)
#pragma unroll
        for (int a = 0; a < 9; ++a) o[6 + a] = q.R[a];
    } else {
#pragma unroll
        for (int a = 0; a < 9; ++a) o[6 + a] = q.R[a];
    }
    o[0] = p0 - q.goal[0]; o[1] = p1 - q.goal[1]; o[2] = p2 - q.goal[2];
    o[3] = v0; o[4] = v1; o[5] = v2; o[15] = w0; o[16] = w1; o[17] = w2;
    if (c.obs_repr == QS_OBS_XYZ_VXYZ_R_OMEGA_FLOOR) o[18] = p2;
    if (c.obs_repr == QS_OBS_XYZ_VXYZ_R_OMEGA_WALL) {
        o[18] = clampf(p0 + c.hx, 0.f, 5.f); o[19] = clampf(p1 + c.hy, 0.f, 5.f); o[20] = clampf(p2, 0.f, 5.f);
        o[21] = clampf(c.hx - p0, 0.f, 5.f); o[22] = clampf(c.hy - p1, 0.f, 5.f); o[23] = clampf(c.hz - p2, 0.f, 5.f);
    }
}

// ----------------------------------------------------------------------------------------------------------------
// impulses (all lanes of a group compute the same event redundantly; the lanes involved keep the result)
// ----------------------------------------------------------------------------------------------------------------
// compute_new_vel, collisions/utils.py:8-19
__device__ __forceinline__ void compute_new_vel(float max_mag, float *v, const float *shift, float decay)
{
    float n0 = v[0] + shift[0], n1 = v[1] + shift[1], n2 = v[2] + shift[2];
    float mag = norm3f(n0, n1, n2), den = (mag == 0.0f) ? mag + 1e-5f : mag;
    float d0 = n0 / den, d1 = n1 / den, d2 = n2 / den;
    mag = fminf(mag * decay, max_mag);
    v[0] += d0 * mag - v[0]; v[1] += d1 * mag - v[1]; v[2] += d2 * mag - v[2];
}
// compute_new_omega, collisions/utils.py:22-33
__device__ __forceinline__ void compute_new_omega(const float *u4, float magn_scale, float *out)
{
    float omax = magn_scale * QS_PI_F;
    float a = -1.f + 2.f * u4[0], b = -1.f + 2.f * u4[1], cc = -1.f + 2.f * u4[2];
    float mag = norm3f(a, b, cc), den = (mag == 0.0f) ? mag + 1e-5f : mag;
    float m2 = 0.5f * omax + 0.5f * omax * u4[3];
    out[0] = a / den * m2; out[1] = b / den * m2; out[2] = cc / den * m2;
}

// perform_collision_between_drones, collisions/quadrotors.py:9-59.  Inputs are drone i ("1") and drone j ("2").
static __device__ __noinline__ void pair_impulse(const Rng g, int i, int j, const float *p1, const float *p2, float *v1, float *v2,
                                          float *w1, float *w2)
{
    float n0 = p1[0] - p2[0], n1 = p1[1] - p2[1], n2 = p1[2] - p2[2];
    float nm = norm3f(n0, n1, n2), den = (nm == 0.0f) ? nm + 1e-5f : nm;
    n0 /= den; n1 /= den; n2 /= den;
    float a1 = v1[0] * n0 + v1[1] * n1 + v1[2] * n2, a2 = v2[0] * n0 + v2[1] * n1 + v2[2] * n2;
    float vc[3] = { (a2 - a1) * n0, (a2 - a1) * n1, (a2 - a1) * n2 };
    float s1[3] = { vc[0], vc[1], vc[2] }, s2[3] = { -vc[0], -vc[1], -vc[2] };
    for (int att = 0; att < 3; ++att) {
        float x[4], y[4], z[4];
        rng_n4(g, SITE_PAIR, i, j, att * 3 + 0, x);
        rng_n4(g, SITE_PAIR, i, j, att * 3 + 1, y);
        rng_n4(g, SITE_PAIR, i, j, att * 3 + 2, z);
        float cons[3] = { 0.8f * x[0], 0.8f * x[1], 0.8f * x[2] };
        float e1[3] = { cons[0] + 0.15f * x[3], cons[1] + 0.15f * y[0], cons[2] + 0.15f * y[1] };
        float e2[3] = { -cons[0] + 0.15f * y[2], -cons[1] + 0.15f * y[3], -cons[2] + 0.15f * z[0] };
#pragma unroll
        for (int a = 0; a < 3; ++a) { s1[a] = vc[a] + e1[a]; s2[a] = -vc[a] + e2[a]; }
        float t1 = (v1[0] + s1[0]) * n0 + (v1[1] + s1[1]) * n1 + (v1[2] + s1[2]) * n2;
        float t2 = (v2[0] + s2[0]) * n0 + (v2[1] + s2[1]) * n1 + (v2[2] + s2[2]) * n2;
        if (t1 > 0.f && 0.f > t2) break;
    }
    float maxv = fmaxf(norm3f(v1[0], v1[1], v1[2]), norm3f(v2[0], v2[1], v2[2]));
    float u[4], t[4];
    rng_u4(g, SITE_PAIR, i, j, 9, u);                                 // idx 36..39
    rng_u4(g, SITE_PAIR, i, j, 10, t);                                // idx 40..43
    compute_new_vel(maxv, v1, s1, 0.2f + 0.6f * u[0]);
    compute_new_vel(maxv, v2, s2, 0.2f + 0.6f * u[1]);
    float u4[4] = { u[2], u[3], t[0], t[1] }, w[3];
    compute_new_omega(u4, 20.0f, w);
    w1[0] += w[0]; w1[1] += w[1]; w1[2] += w[2];
    w2[0] -= w[0]; w2[1] -= w[1]; w2[2] -= w[2];
}

// perform_collision_with_obstacle, collisions/obstacles.py:9-50
static __device__ __noinline__ void obstacle_impulse(const DevConst &c, const Rng g, int drone, const float *p, float *v, float *w,
                                              float ox, float oy)
{
    float n0 = p[0] - ox, n1 = p[1] - oy;
    float nm = sqrtf(n0 * n0 + n1 * n1), den = (nm == 0.0f) ? nm + 1e-5f : nm;
    n0 /= den; n1 /= den;
    float vm = norm3f(v[0], v[1], v[2]);
    float nv[3] = { vm * n0, vm * n1, 0.f }, noise[3] = { 0.f, 0.f, 0.f };
    for (int att = 0; att < 3; ++att) {
        float x[4], y[4];
        rng_n4(g, SITE_OBST, drone, 0, att * 2, x);
        rng_n4(g, SITE_OBST, drone, 0, att * 2 + 1, y);
        float t[3] = { 0.1f * x[0] + 0.05f * x[3], 0.1f * x[1] + 0.05f * y[0], 0.1f * x[2] + 0.05f * y[1] };
        if ((nv[0] + t[0]) * n0 + (nv[1] + t[1]) * n1 > 0.f) { noise[0] = t[0]; noise[1] = t[1]; noise[2] = t[2]; break; }
    }
    float dz = p[2] - 0.5f * c.room_h;
    float d3 = norm3f(p[0] - ox, p[1] - oy, dz);
    float shift[3] = { nv[0] - v[0] + noise[0], nv[1] - v[1] + noise[1], nv[2] - v[2] + noise[2] };
    float u[4], t[4];
    rng_u4(g, SITE_OBST, drone, 0, 6, u);                             // idx 24..27
    rng_u4(g, SITE_OBST, drone, 0, 7, t);                             // idx 28..31
    float decay = (d3 < c.obst_rad) ? 1.0f : 0.2f + 0.6f * u[0];
    compute_new_vel(vm, v, shift, decay);
    float u4[4] = { u[1], u[2], u[3], t[0] }, dw[3];
    compute_new_omega(u4, 1.0f, dw);
    w[0] += dw[0]; w[1] += dw[1]; w[2] += dw[2];
}

// perform_collision_with_wall / _ceiling, collisions/room.py:6-45, 91-113
static __device__ __noinline__ void room_impulse(const DevConst &c, const Rng g, int drone, int flags, float *v, float *w, bool is_wall)
{
    int site = is_wall ? SITE_WALL : SITE_CEILING;
    float u[12];
    rng_u4(g, site, drone, 0, 0, u); rng_u4(g, site, drone, 0, 1, u + 4); rng_u4(g, site, drone, 0, 2, u + 8);
    float sp = norm3f(v[0], v[1], v[2]);
    float lo = 0.2f * sp, hi = 0.8f * sp;
    float real = clampf(lo + (hi - lo) * u[0], 0.1f, 6.0f);
    float d0 = -1.f + 2.f * u[1], d1 = -1.f + 2.f * u[2], d2;
    int k;
    if (is_wall) {
        if (flags & F_AT_XLO) d0 = 0.1f + 0.9f * u[4]; else if (flags & F_AT_XHI) d0 = -1.0f + 0.9f * u[4];
        if (flags & F_AT_YLO) d1 = 0.1f + 0.9f * u[5]; else if (flags & F_AT_YHI) d1 = -1.0f + 0.9f * u[5];
        k = 6;
    } else k = 4;
    d2 = -1.0f + 0.5f * u[k];
    float dm = norm3f(d0, d1, d2) + 1e-5f;
    v[0] = real * (d0 / dm); v[1] = real * (d1 / dm); v[2] = real * (d2 / dm);
    float w0 = -1.f + 2.f * u[k + 1], w1 = -1.f + 2.f * u[k + 2], w2 = -1.f + 2.f * u[k + 3];
    float wm = norm3f(w0, w1, w2) + 1e-5f;
    float omax = 20.f * QS_PI_F, mag = 0.5f * omax + 0.5f * omax * u[k + 4];
    w[0] += w0 / wm * mag; w[1] += w1 / wm * mag; w[2] += w2 / wm * mag;
}

// ----------------------------------------------------------------------------------------------------------------
// reset
// ----------------------------------------------------------------------------------------------------------------
// get_cell_centers, obstacles/utils.py:47-58
__device__ __forceinline__ void cell_center(const DevConst &c, int index, float &x, float &y)
{
    int i = index / c.obst_W, jj = index - i * c.obst_W, j = c.obst_W - 1 - jj;
    x = (float)i + 0.5f - (float)(c.obst_L / 2);
    y = (float)j + 0.5f - (float)(c.obst_W / 2);
}

// k distinct ids of n via partial Fisher-Yates (oracle rnd_choice).  Returns through `a` (first k entries).
__device__ __forceinline__ void choice_fy(const Rng &g, int aux, int n, int k, unsigned char *a)
{
    for (int i = 0; i < n; ++i) a[i] = (unsigned char)i;
    for (int t = 0; t < k; ++t) {
        float u = rng_u(g, SITE_SCENARIO, 0xFF, aux, t);
        int r = t + (int)floorf(u * (float)(n - t));
        r = min(r, n - 1);
        unsigned char tmp = a[t]; a[t] = a[r]; a[r] = tmp;
    }
}

// obst_generation_given_density (quadrotor_multi.py:405-426) + Scenario_o_random / o_static_same_goal .reset
// (scenarios/obstacles/o_random.py:26-52, o_static_same_goal.py:27-48, o_base.py:69-81,124-153).
//
// Called by ALL lanes of the env's lane group (`gmask`), converged.  An auto-reset inside the step kernel keeps its whole warp --
// and, in the last wave of the grid, the whole kernel -- waiting, so the latency of this function is what a steady-state step pays
// for resets (profiles/README.md, round 2).  Hence:
//   * every uniform the scenario needs (7 streams, <= 2 + (M + 4 K) / 4 Philox blocks) is drawn ONCE, one block per lane of the
//     group in parallel, into `scratch` (the group's rows of the observation tile, which the reset observation overwrites anyway);
//     the sequential form evaluated a whole Philox block per uniform, every lane redundantly;
//   * the sequential part (two or three partial Fisher-Yates shuffles, the free-cell list, the largest-empty-square scan) runs on
//     the group's first lane only, on byte arrays in shared memory (they were thread-local memory), and publishes one spawn cell
//     and one goal cell per drone;
//   * the new obstacle centres also go to `obst_sm` (the warp's staged copy) so that the SDF of the reset observation does not
//     chain M dependent global loads.
// Same counters, same arithmetic, same results as the sequential form (which remains as the fallback when `scratch` is too small).
__device__ __forceinline__ int obst_rng_blocks(int M, int K) { return ((M + 3) >> 2) + 4 * ((K + 3) >> 2) + 2; }
__device__ __forceinline__ int obst_scratch_floats(int M, int K) { return 4 * obst_rng_blocks(M, K) + 16 + 16 + 16; }   // table + cells[64] + free[64] + result[64]

static __device__ __noinline__ void obstacle_scenario_reset(const DevConst &c, const Rng g, int d, int KG, uint32_t gmask, bool store, float2 *obst_xy,
                                                     float2 *obst_sm, float *scratch, int cap, float *spawn, float *goal, int &scenario_now)
{
    const int L = c.obst_L, W = c.obst_W, M = c.M, K = c.K, cells = L * W;
    const int nb0 = (M + 3) >> 2, nbK = (K + 3) >> 2, nblk = nb0 + 4 * nbK + 2;
    const bool fast = scratch != nullptr && cap >= obst_scratch_floats(M, K);
    float *utab = scratch;
    unsigned char *arr = reinterpret_cast<unsigned char *>(scratch + 4 * nblk), *freec = arr + 64, *res = arr + 128;
    // block e of the table: streams in the order aux 0 (obstacle cells), 2 (spawn cells), 5 (goal cells), 3 (spawn z), 6 (goal z), 1 (mix), 4 (goal z, shared)
    const int off2 = nb0, off5 = nb0 + nbK, off3 = nb0 + 2 * nbK, off6 = nb0 + 3 * nbK, off1 = nb0 + 4 * nbK, off4 = off1 + 1;
    if (fast) {
        __syncwarp(gmask);                                              // the tile rows are free: terminal observations were copied out
        for (int e = d; e < nblk; e += KG) {
            int aux, blk;
            if (e < off2) { aux = 0; blk = e; }
            else if (e < off5) { aux = 2; blk = e - off2; }
            else if (e < off3) { aux = 5; blk = e - off5; }
            else if (e < off6) { aux = 3; blk = e - off3; }
            else if (e < off1) { aux = 6; blk = e - off6; }
            else if (e < off4) { aux = 1; blk = 0; }
            else { aux = 4; blk = 0; }
            float u[4];
            rng_u4(g, SITE_SCENARIO, 0xFF, aux, blk, u);
            *reinterpret_cast<float4 *>(utab + 4 * e) = make_float4(u[0], u[1], u[2], u[3]);
        }
        __syncwarp(gmask);
    }
#define QS_OBST_U(aux, off, idx) (fast ? utab[4 * (off) + (idx)] : rng_u(g, SITE_SCENARIO, 0xFF, (aux), (idx)))
    int scen = c.scenario;
    if (scen == QS_SCENARIO_O_MIX) {
        int mode_index = (int)floorf(QS_OBST_U(1, off1, 0) * 100.0f);
        // a single drone draws from QUADS_MODE_LIST_OBSTACLES_SINGLE = ['o_random'] (mix.py:49-51, utils.py:23)
        scen = (K == 1 || mode_index % 2 == 0) ? QS_SCENARIO_O_RANDOM : QS_SCENARIO_O_STATIC_SAME_GOAL;
    }
    scenario_now = scen;
    if (fast) {
        if (d == 0) {
            // k distinct ids of n: partial Fisher-Yates (oracle rnd_choice), in place on arr[0..n)
            for (int i = 0; i < cells; i += 4) *reinterpret_cast<uint32_t *>(arr + i) = 0x03020100u + 0x01010101u * (uint32_t)i;
            for (int t = 0; t < M; ++t) {
                int r = min(t + (int)floorf(utab[t] * (float)(cells - t)), cells - 1);
                unsigned char tmp = arr[t]; arr[t] = arr[r]; arr[r] = tmp;
            }
            unsigned long long map = 0ull;                              // bit rid*W + cid
            for (int m = 0; m < M; ++m) {
                int rid = arr[m] / W, cid = arr[m] - rid * W;
                map |= 1ull << (rid * W + cid);
                float x, y;
                cell_center(c, rid + L * cid, x, y);
                if (store) obst_xy[m] = make_float2(x, y);
                if (obst_sm != nullptr) obst_sm[m] = make_float2(x, y);
            }
            int nf = 0;
            for (int cell = 0; cell < cells; ++cell) if (!((map >> cell) & 1ull)) freec[nf++] = (unsigned char)cell;   // row-major (rid, cid)
            for (int i = 0; i < nf; i += 4) *reinterpret_cast<uint32_t *>(arr + i) = 0x03020100u + 0x01010101u * (uint32_t)i;
            for (int t = 0; t < K; ++t) {
                int r = min(t + (int)floorf(utab[4 * off2 + t] * (float)(nf - t)), nf - 1);
                unsigned char tmp = arr[t]; arr[t] = arr[r]; arr[r] = tmp;
            }
            for (int t = 0; t < K; ++t) res[t] = freec[arr[t]];
            if (scen == QS_SCENARIO_O_STATIC_SAME_GOAL) {
                // largest empty square; dp row/col 0 copy the obstacle map itself (o_base.py:134-136).  Two rolling rows of the table.
                unsigned char *prev = arr, *cur = freec;               // the free-cell list is no longer needed
                int max_size = 0, cx = 0, cy = 0;
                for (int j = 0; j < W; ++j) prev[j] = (unsigned char)((map >> j) & 1ull);
                for (int r = 1; r < L; ++r) {
                    cur[0] = (unsigned char)((map >> (r * W)) & 1ull);
                    for (int j = 1; j < W; ++j) {
                        int v = 0;
                        if (!((map >> (r * W + j)) & 1ull)) {
                            v = min(min((int)prev[j], (int)cur[j - 1]), (int)prev[j - 1]) + 1;
                            if (v > max_size) { max_size = v; cx = r - (max_size - 1) / 2; cy = j - (max_size - 1) / 2; }
                        }
                        cur[j] = (unsigned char)v;
                    }
                    unsigned char *t = prev; prev = cur; cur = t;
                }
                res[K] = (unsigned char)cx; res[K + 1] = (unsigned char)cy;
            } else {
                for (int i = 0; i < nf; i += 4) *reinterpret_cast<uint32_t *>(arr + i) = 0x03020100u + 0x01010101u * (uint32_t)i;
                for (int t = 0; t < K; ++t) {
                    int r = min(t + (int)floorf(utab[4 * off5 + t] * (float)(nf - t)), nf - 1);
                    unsigned char tmp = arr[t]; arr[t] = arr[r]; arr[r] = tmp;
                }
                for (int t = 0; t < K; ++t) res[K + t] = freec[arr[t]];
            }
        }
        __syncwarp(gmask);
        const int dk = d < K ? d : 0;
        {
            const int cell = res[dk], rid = cell / W, cid = cell - rid * W;
            cell_center(c, rid + L * cid, spawn[0], spawn[1]);
            spawn[2] = 1.0f + 2.0f * utab[4 * off3 + dk];
        }
        if (scen == QS_SCENARIO_O_STATIC_SAME_GOAL) {
            cell_center(c, (int)res[K] + W * (int)res[K + 1], goal[0], goal[1]);
            goal[2] = 1.5f + 1.5f * utab[4 * off4];
        } else {
            const int cell = res[K + dk], rid = cell / W, cid = cell - rid * W;
            cell_center(c, rid + L * cid, goal[0], goal[1]);
            goal[2] = 1.0f + 2.0f * utab[4 * off6 + dk];
        }
        __syncwarp(gmask);                                              // the scratch rows are rewritten by the reset observation next
        return;
    }
#undef QS_OBST_U
    // ---- sequential form: every lane evaluates everything (same keys -> same values)
    const int drone = d;
    const bool leader = store && d == 0;
    unsigned char a[64];
    choice_fy(g, 0, L * W, M, a);
    unsigned long long map = 0ull;                                      // bit rid*W + cid
    for (int m = 0; m < M; ++m) {
        int rid = a[m] / W, cid = a[m] - rid * W;
        map |= 1ull << (rid * W + cid);
        float x, y;
        cell_center(c, rid + L * cid, x, y);
        if (leader) obst_xy[m] = make_float2(x, y);
        if (d == 0 && obst_sm != nullptr) obst_sm[m] = make_float2(x, y);
    }
    unsigned char freel[64];
    int nf = 0;
    for (int cell = 0; cell < L * W; ++cell) if (!((map >> cell) & 1ull)) freel[nf++] = (unsigned char)cell;   // row-major (rid, cid)
    {
        choice_fy(g, 2, nf, K, a);
        int cell = freel[a[drone < K ? drone : 0]], rid = cell / W, cid = cell - rid * W;
        cell_center(c, rid + L * cid, spawn[0], spawn[1]);
        spawn[2] = 1.0f + 2.0f * rng_u(g, SITE_SCENARIO, 0xFF, 3, drone);
    }
    if (scen == QS_SCENARIO_O_STATIC_SAME_GOAL) {
        // largest empty square; dp row/col 0 copy the obstacle map itself (o_base.py:134-136)
        int dp[64], max_size = 0, cx = 0, cy = 0;
        for (int j = 0; j < W; ++j) dp[j] = (int)((map >> j) & 1ull);
        for (int r = 1; r < L; ++r) {
            dp[r * W] = (int)((map >> (r * W)) & 1ull);
            for (int j = 1; j < W; ++j) {
                int v = 0;
                if (!((map >> (r * W + j)) & 1ull)) {
                    v = min(min(dp[(r - 1) * W + j], dp[r * W + j - 1]), dp[(r - 1) * W + j - 1]) + 1;
                    if (v > max_size) { max_size = v; cx = r - (max_size - 1) / 2; cy = j - (max_size - 1) / 2; }
                }
                dp[r * W + j] = v;
            }
        }
        cell_center(c, cx + W * cy, goal[0], goal[1]);
        goal[2] = 1.5f + 1.5f * rng_u(g, SITE_SCENARIO, 0xFF, 4, 0);
    } else {
        choice_fy(g, 5, nf, K, a);
        int cell = freel[a[drone < K ? drone : 0]], rid = cell / W, cid = cell - rid * W;
        cell_center(c, rid + L * cid, goal[0], goal[1]);
        goal[2] = 1.0f + 2.0f * rng_u(g, SITE_SCENARIO, 0xFF, 6, drone);
    }
}

// QuadrotorSingle._reset, quadrotor_single.py:401-469
// out = { x, y, z, cos(yaw), sin(yaw) }
static __device__ __noinline__ void drone_reset(const DevConst &c, const Rng g, int drone, const float *spawn, float *out)
{
    float u[4];
    rng_u4(g, SITE_SPAWN, drone, 0, 0, u);
    float px = (-c.spawn_box + 2.0f * c.spawn_box * u[0]) + spawn[0];
    float py = (-c.spawn_box + 2.0f * c.spawn_box * u[1]) + spawn[1];
    float pz = fmaxf((-c.spawn_box + 2.0f * c.spawn_box * u[2]) + spawn[2], c.spawn_min_z);
    float hx = -px, hy = -py, hn = sqrtf(hx * hx + hy * hy);
    if (!(hn < 0.00001f)) { hx /= hn; hy /= hn; }
    float cy, sy;
    unit_dir(hx, hy, cy, sy);                                           // fallback: face the origin
    bool found = false;
    for (int blk = 0; blk < 16 && !found; ++blk) {                      // randyaw() rejection loop (:454-456)
        rng_u4(g, SITE_SPAWN, drone, 1, blk, u);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            if (!found) {
                float s, cc;
                sincospif(-1.0f + 2.0f * u[t], &s, &cc);
                if (!(cc * hx + s * hy < 0.5f)) { cy = cc; sy = s; found = true; }
            }
        }
    }
    out[0] = px; out[1] = py; out[2] = pz; out[3] = cy; out[4] = sy;
}

// ----------------------------------------------------------------------------------------------------------------
// group helpers
// ----------------------------------------------------------------------------------------------------------------
template <int KG>
__device__ __forceinline__ uint32_t group_mask(int lane) { return (KG == 32) ? QS_FULL : (((1u << KG) - 1u) << (lane & ~(KG - 1))); }

// neighbour + obstacle part of the observation, written into the warp's shared-memory tile row `o`.
// vs: the velocity snapshot the reference's `self.vel` holds (stale at reset, quadrotor_multi.py:477).
// `stage` is this warp's 32 x 2 float4 exchange buffer: every lane publishes (pos, vs), the group syncs, and each lane
// reads its K-1 neighbours as broadcast 16-byte shared-memory loads.
// `ob`: the env's obstacle centres (the warp's shared-memory copy in the step path, global memory right after a reset)
// a14 in one pass over the env's obstacles: the 3x3 SDF patch (get_surround_sdfs, obstacles/utils.py:5-27; the min over
// obstacles commutes with the sqrt) and the first obstacle the drone touches (collision_detection, obstacles/utils.py:31-43:
// 2-D distance <= arm + size/2, lowest index wins) -- the centre cell of the patch IS that distance.
// Brute-force form, every obstacle against every patch point: a candidate-list form (patch only for the centres near the drone) ran
// fewer instructions with less ILP and was slower (cfg3 102.4 -> 110.5 us).
__device__ __forceinline__ void obstacle_sdf_and_hit(const DevConst &c, const float2 *ob, float px, float py, float *r, int &hit)
{
    const float gx[3] = { px - c.sdf_res, px, px + c.sdf_res }, gy[3] = { py - c.sdf_res, py, py + c.sdf_res };
    const float obst2 = c.thr_obst * c.thr_obst * 1.0001f;
    float md[9];
#pragma unroll
    for (int a = 0; a < 9; ++a) md[a] = 10000.0f;                       // (100)^2
    hit = -1;
    QS_UNROLL(QS_SDF_UNROLL)
    for (int m = 0; m < c.M; ++m) {
        const float2 xy = ob[m];
        float dx2[3], dy2[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) { float dx = gx[a] - xy.x, dy = gy[a] - xy.y; dx2[a] = dx * dx; dy2[a] = dy * dy; }
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) md[a * 3 + b] = fminf(md[a * 3 + b], dx2[a] + dy2[b]);
        const float d2 = dx2[1] + dy2[1];
        if (d2 <= obst2 && hit < 0 && __fsqrt_rn(d2) <= c.thr_obst) hit = m;
    }
#pragma unroll
    for (int a = 0; a < 9; ++a) r[a] = sqrtf(md[a]) - c.obst_rad;
}

// SDF = false: the caller already wrote the SDF patch of these positions (step path: together with the hit test)
// COMPACT: the rolled, branchy form of the row writes for kernel variants whose hot code is already at the instruction-cache limit
// Relative position of a neighbour, clipped to the observation Box (quadrotor_multi.py:337-339).  In the step path both positions
// come out of the dynamics' room clip (|x|,|y| <= room/2, 0 <= z <= room_h), so the difference cannot leave the Box and the clip is
// the identity; only the reset path (drones may spawn outside a small room) evaluates it.
template <bool CLIP>
__device__ __forceinline__ float rel_pos(float x, float lim) { return CLIP ? clampf(x, -lim, lim) : x; }

template <int KG, bool OBST, bool SDF, bool COMPACT = false>
__device__ __forceinline__ void group_obs_tail(const DevConst &c, const float2 *ob, int d, int lane, uint32_t gmask, bool valid,
                                               const Drone &q, const float *vs, float *o, float4 *stage)
{
    const int base = lane & ~(KG - 1);
    if (c.nbr_type == QS_NEIGHBOR_POS_VEL && KG > 1) {
        // a15: neighborhood_indices + get_rel_pos_vel_item + clip (quadrotor_multi.py:275-380)
        __syncwarp(gmask);
        stage[2 * lane] = make_float4(q.p[0], q.p[1], q.p[2], 0.f);
        stage[2 * lane + 1] = make_float4(vs[0], vs[1], vs[2], 0.f);
        __syncwarp(gmask);
        const float INF = __int_as_float(0x7f800000);
        if (c.V < c.K - 1) {
            // rank by ||[dp, dv]|| (6-vector, :357-359), max(., 0.01).  The ranking is done on the squared metric
            // (monotone, so the order is the same away from ties) and as a stable rank count -- candidate a precedes b
            // iff met[a] <= met[b] for a < b -- which equals argsort(kind='stable')[:V] (first-minimum selection).
            float met[KG];
#pragma unroll
            for (int j = 0; j < KG; ++j) {
                float4 a = stage[2 * (base + j)], b = stage[2 * (base + j) + 1];
                float r0 = a.x - q.p[0], r1 = a.y - q.p[1], r2 = a.z - q.p[2], r3 = b.x - vs[0], r4 = b.y - vs[1], r5 = b.z - vs[2];
                float ss = r0 * r0 + r1 * r1 + r2 * r2 + r3 * r3 + r4 * r4 + r5 * r5;
                met[j] = (j < c.K && j != d) ? fmaxf(ss, 1.0e-4f) : INF;
            }
            if ((KG >= 16 || (OBST && KG >= 4)) && c.V * 3 < 2 * (KG - 1)) {
                // few rows out of many candidates (6 of 31; 2 of 7 in the obstacle recipe): V rounds of first-minimum selection cost
                // ~3 KG instructions each, the all-pairs rank count below ~2 KG (KG - 1) plus a row pass over every candidate.
                // Compiled into the wide-group kernels and the obstacle variants only: the plain 8-lane kernel keeps a single
                // selection path (its hot code has to stay inside the instruction cache).
#pragma unroll 1
                for (int sidx = 0; sidx < c.V; ++sidx) {
                    float best = INF; int jb = 0;
#pragma unroll
                    for (int j = 0; j < KG; ++j) if (met[j] < best) { best = met[j]; jb = j; }
#pragma unroll
                    for (int j = 0; j < KG; ++j) met[j] = (j == jb) ? INF : met[j];
                    if (valid) {
                        float4 a = stage[2 * (base + jb)], b = stage[2 * (base + jb) + 1];
                        float *r = o + c.S + 6 * sidx;
                        r[0] = rel_pos<SDF>(a.x - q.p[0], c.room_l); r[1] = rel_pos<SDF>(a.y - q.p[1], c.room_w); r[2] = rel_pos<SDF>(a.z - q.p[2], c.room_h);
                        r[3] = clampf(b.x - vs[0], -6.f, 6.f); r[4] = clampf(b.y - vs[1], -6.f, 6.f); r[5] = clampf(b.z - vs[2], -6.f, 6.f);
                    }
                }
            } else if (KG <= 8) {
                // stable rank count with the ranks packed 4 bits per candidate: one compare + one select + one add per pair.
                // Lanes that are not candidates (self, j >= K) carry +inf and therefore rank behind every real candidate, so a
                // rank below V (< K - 1) always belongs to a real one.  The packed form also lets the row writes be a rolled
                // loop (unrolled they are 8 x 30 instructions executed once each; the hot path must stay inside the 32 KB
                // L1.5 instruction cache).
                uint32_t acc[4] = { 0u, 0u, 0u, 0u };                   // four independent chains instead of one of 28 dependent adds
#pragma unroll
                for (int a = 0, n = 0; a < KG; ++a)
#pragma unroll
                    for (int b = a + 1; b < KG; ++b, ++n) acc[n & 3] += (met[b] < met[a]) ? (1u << (4 * a)) : (1u << (4 * b));
                const uint32_t pk = (acc[0] + acc[1]) + (acc[2] + acc[3]);
                if (valid) {
                    if (QS_NB_PRED > 0 && !COMPACT) {
                    // loads and arithmetic for every candidate, only the six stores under the predicate: no divergent branch
                    // (and its reconvergence) per iteration, and two iterations in flight hide the shared-memory latency
                    QS_UNROLL((QS_NB_PRED > 0 ? QS_NB_PRED : 1))
                    for (int j = 0; j < KG; ++j) {
                        const int rk = (int)((pk >> (4 * j)) & 15u);
                        const float4 a = stage[2 * (base + j)], b = stage[2 * (base + j) + 1];
                        const float r0 = rel_pos<SDF>(a.x - q.p[0], c.room_l), r1 = rel_pos<SDF>(a.y - q.p[1], c.room_w), r2 = rel_pos<SDF>(a.z - q.p[2], c.room_h);
                        const float r3 = clampf(b.x - vs[0], -6.f, 6.f), r4 = clampf(b.y - vs[1], -6.f, 6.f), r5 = clampf(b.z - vs[2], -6.f, 6.f);
                        float *r = o + c.S + 6 * rk;
                        if (rk < c.V) { r[0] = r0; r[1] = r1; r[2] = r2; r[3] = r3; r[4] = r4; r[5] = r5; }
                    }
                    } else {
#pragma unroll 1
                    for (int j = 0; j < KG; ++j) {
                        const int rk = (int)((pk >> (4 * j)) & 15u);
                        if (rk < c.V) {
                            float4 a = stage[2 * (base + j)], b = stage[2 * (base + j) + 1];
                            float *r = o + c.S + 6 * rk;
                            r[0] = rel_pos<SDF>(a.x - q.p[0], c.room_l); r[1] = rel_pos<SDF>(a.y - q.p[1], c.room_w); r[2] = rel_pos<SDF>(a.z - q.p[2], c.room_h);
                            r[3] = clampf(b.x - vs[0], -6.f, 6.f); r[4] = clampf(b.y - vs[1], -6.f, 6.f); r[5] = clampf(b.z - vs[2], -6.f, 6.f);
                        }
                    }
                    }
                }
            } else {
                int rank[KG];
#pragma unroll
                for (int j = 0; j < KG; ++j) rank[j] = 0;
#pragma unroll
                for (int a = 0; a < KG; ++a)
#pragma unroll
                    for (int b = a + 1; b < KG; ++b) {
                        bool b_first = met[b] < met[a];
                        rank[a] += b_first ? 1 : 0;
                        rank[b] += b_first ? 0 : 1;
                    }
                if (valid) {
#pragma unroll
                    for (int j = 0; j < KG; ++j) {
                        if (rank[j] < c.V && met[j] < INF) {
                            float4 a = stage[2 * (base + j)], b = stage[2 * (base + j) + 1];
                            float *r = o + c.S + 6 * rank[j];
                            r[0] = rel_pos<SDF>(a.x - q.p[0], c.room_l); r[1] = rel_pos<SDF>(a.y - q.p[1], c.room_w); r[2] = rel_pos<SDF>(a.z - q.p[2], c.room_h);
                            r[3] = clampf(b.x - vs[0], -6.f, 6.f); r[4] = clampf(b.y - vs[1], -6.f, 6.f); r[5] = clampf(b.z - vs[2], -6.f, 6.f);
                        }
                    }
                }
            }
        } else if (valid) {
            for (int j = 0; j < c.K; ++j) {                                // all others, index order (:350-351)
                if (j == d) continue;
                int sidx = j - (j > d ? 1 : 0);
                float4 a = stage[2 * (base + j)], b = stage[2 * (base + j) + 1];
                float *r = o + c.S + 6 * sidx;
                r[0] = rel_pos<SDF>(a.x - q.p[0], c.room_l); r[1] = rel_pos<SDF>(a.y - q.p[1], c.room_w); r[2] = rel_pos<SDF>(a.z - q.p[2], c.room_h);
                r[3] = clampf(b.x - vs[0], -6.f, 6.f); r[4] = clampf(b.y - vs[1], -6.f, 6.f); r[5] = clampf(b.z - vs[2], -6.f, 6.f);
            }
        }
    }
    if (OBST && SDF && valid) {
        int hit;
        obstacle_sdf_and_hit(c, ob, q.p[0], q.p[1], o + c.S + ((c.nbr_type == QS_NEIGHBOR_POS_VEL) ? 6 * c.V : 0), hit);
    }
}

}  // namespace qs
#include "scenario_kernels.cuh"
namespace qs {

// Reset of one environment (QuadrotorEnvMulti.reset, quadrotor_multi.py:440-519), executed by the env's lane group.
// SCEN: one of the formation scenarios (scenario_kernels.cuh) instead of the fixed static_same_goal.
// Must be called by every lane of the env's lane group (`gmask`), converged.  `scratch`: `cap` floats of shared memory owned by the
// group whose contents are dead (its rows of the observation tile); `obst_sm`: the env's slot of the warp's staged obstacle centres
// (null where there is none).
template <int KG, bool OBST, bool SCEN>
__device__ __forceinline__ void group_reset(const DevConst &c, const DevPtrs &P, const Rng &g, int env, int d, bool valid, uint32_t gmask, float *scratch,
                                            int cap, float2 *obst_sm, Drone &q, int &scenario_now)
{
    float spawn[3], goal[3], out[5];
    if (OBST) {
        int scen = 0;
        float *sc16 = reinterpret_cast<float *>((reinterpret_cast<size_t>(scratch) + 15) & ~(size_t)15);     // 16-byte aligned table
        obstacle_scenario_reset(c, g, d, KG, gmask, env < c.N, P.obst_xy + (size_t)env * QS_MAX_OBSTACLES, obst_sm, sc16,
                                cap - (int)(sc16 - scratch), spawn, goal, scen);
        scenario_now = scen;
    } else if (SCEN) {
        goal[0] = goal[1] = 0.f; goal[2] = 2.0f;
        if (env < c.N) formation_reset(c, g, d, valid && d == 0, reinterpret_cast<float *>(P.scen + (size_t)env * (QS_SC_COUNT / 4)), goal);
        spawn[0] = goal[0]; spawn[1] = goal[1]; spawn[2] = goal[2];     // e.spawn_point = scenario.goals[i], quadrotor_multi.py:469-470
        scenario_now = c.scenario;
    } else {
        goal[0] = 0.f; goal[1] = 0.f; goal[2] = 2.0f;                     // static_same_goal: formation size 0 (scenarios/utils.py:30)
        spawn[0] = 0.f; spawn[1] = 0.f; spawn[2] = 2.0f;
        scenario_now = QS_SCENARIO_STATIC_SAME_GOAL;
    }
    drone_reset(c, g, d, spawn, out);
    q.goal[0] = goal[0]; q.goal[1] = goal[1]; q.goal[2] = goal[2];
    q.p[0] = out[0]; q.p[1] = out[1]; q.p[2] = out[2];
    set_yaw(q.R, out[3], out[4]);
    q.v[0] = q.v[1] = q.v[2] = 0.f; q.w[0] = q.w[1] = q.w[2] = 0.f;
#pragma unroll
    for (int m = 0; m < 4; ++m) { q.rd[m] = 0.f; q.cd[m] = 0.f; }
    q.flags = (OBST && scenario_now == QS_SCENARIO_O_STATIC_SAME_GOAL) ? F_SCEN_OSTATIC : 0; q.colmask = 0u;
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// coalesced copy of the warp's observation tile (rows contiguous in global memory) out of shared memory
__device__ __forceinline__ void warp_store_tile(const float *tile, float *dst, int count, int lane)
{
    if (((((size_t)dst) & 15) == 0) && ((count & 3) == 0)) {
        const float4 *s = reinterpret_cast<const float4 *>(tile);
        float4 *o = reinterpret_cast<float4 *>(dst);
        for (int i = lane; i < (count >> 2); i += 32) __stcs(o + i, s[i]);
    } else {
        for (int i = lane; i < count; i += 32) __stcs(dst + i, tile[i]);
    }
}

// ----------------------------------------------------------------------------------------------------------------
// The step kernel: QuadrotorEnvMulti.step (quadrotor_multi.py:521-842) for every env, one launch.
// ----------------------------------------------------------------------------------------------------------------
// One warp-tile (32 lanes = 32/KG envs) per warp, state read straight from HBM.  A persistent form (resident grid, TMA bulk
// prefetch of the next warp-tile) was measured slower and removed: profiles/README.md.

// 4-byte asynchronous global -> shared copy (LDGSTS): the per-env scalars travel without a register
__device__ __forceinline__ void cp_async4(void *dst_smem, const void *src_gmem)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem) : "memory");
}
__device__ __forceinline__ void prefetch_row(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// FEAT: compile-time feature set (bit 0 obstacles, bit 1 downwash).  The big optional passes are specialised away instead of
// being skipped at run time: a cfg2 launch then carries none of their code or registers (an "uber-kernel" with run-time
// flags cost the plain 8-quad swarm 9 % when the obstacle / downwash code was reshaped).
template <int KG, int FEAT>
__global__ void __launch_bounds__(QS_STEP_MAXTHREADS, QS_STEP_MINBLOCKS) step_kernel(const __grid_constant__ DevConst c, const __grid_constant__ DevPtrs P,
                                                   const float4 *__restrict__ actions, float *__restrict__ obs,
                                                   float *__restrict__ rew, uint8_t *__restrict__ done, float *__restrict__ term_obs,
                                                   uint8_t *__restrict__ reset_success)
{
    extern __shared__ __align__(16) float smem[];
    constexpr bool OBST = (FEAT & 1) != 0, DOWNWASH = (FEAT & 2) != 0, SCEN = (FEAT & 4) != 0;
    const int lane = threadIdx.x & 31, warp_in_block = threadIdx.x >> 5, warps_per_block = blockDim.x >> 5;
    const int d = lane % KG;
    const uint32_t gmask = group_mask<KG>(lane);
    const int base = lane & ~(KG - 1);
    constexpr int GPW = 32 / KG;                                        // env groups per warp
    const int rows_per_warp = GPW * c.K;
    float4 *stage = reinterpret_cast<float4 *>(smem) + (size_t)warp_in_block * 64;          // 32 lanes x 2 float4
    float *tile = smem + (size_t)warps_per_block * 256 + (size_t)warp_in_block * rows_per_warp * c.D;   // this warp's obs rows
    const int row = (lane / KG) * c.K + d;
    float *orow = tile + (size_t)row * c.D;
    const int n_wt = (c.N + GPW - 1) / GPW;                             // warp-tiles
    // obstacle centres of this warp-tile's envs (GPW x M float2), staged once per tile: the hit test and the SDF read each of
    // them K times, and the serial `first hit wins` loop would otherwise chain M dependent global loads
    const size_t ob_off = ((size_t)warps_per_block * 256 + (size_t)warps_per_block * rows_per_warp * c.D + 3) & ~(size_t)3;
    const int ob_per_warp = OBST ? GPW * c.M : 0;
    float2 *ob_sm = reinterpret_cast<float2 *>(smem + ob_off) + (size_t)warp_in_block * ob_per_warp;
    const float2 *ob_env = ob_sm + (lane / KG) * c.M;
    // formation scenarios (never with obstacles): the scenario rows of this warp-tile's envs live where the obstacle centres would
    float4 *sc_sm = reinterpret_cast<float4 *>(smem + ob_off) + (size_t)warp_in_block * (GPW * (QS_SC_COUNT / 4));
    const float4 *sc_env = sc_sm + (lane / KG) * (QS_SC_COUNT / 4);
    // per-thread scratch slots behind the staged obstacle centres or scenario rows: 4 x blockDim float4 (the step's pre-generated
    // normals), then 3 ints per thread (tick, svd counter, reset-first flag)
    const size_t park_off = (ob_off + (OBST ? (size_t)warps_per_block * ob_per_warp * 2 : (SCEN ? (size_t)warps_per_block * GPW * QS_SC_COUNT : 0)) + 3) & ~(size_t)3;
    int wt = (int)blockIdx.x * warps_per_block + warp_in_block;
    constexpr bool HOT_OK = (FEAT & 5) != 0 && KG < 32;                // same rule as qs_create's e->hot
    const bool HOT = HOT_OK && P.hot_flag_cur != nullptr;   // warp-uniform (the flag travels with the early-draw scalars)
    bool hot_role = false;
    if (HOT) {
        if (blockIdx.x == 0 && threadIdx.x == 0) *P.hot_cnt_clear = 0;  // the buffer the previous step consumed: the next step produces into it
        if ((int)blockIdx.x < P.hot_blocks) {
            // (volatile loads: the hot blocks' own dependent look-up, marked so that prologue_check.py can tell it from the state loads)
            if (wt >= min(*(volatile int *)P.hot_cnt_cur, P.hot_cap)) return;   // no listed tile for this warp
            wt = ((volatile int *)P.hot_list_cur)[wt];
            hot_role = true;
        } else wt -= P.hot_blocks * warps_per_block;
    }
    // at most one trip: the loop shape is kept because an early `return` for wt >= n_wt compiles to different (longer) code
    for (; wt < n_wt; wt += n_wt) {
    const int warp_env0 = wt * GPW;                                     // first env of this warp-tile
    const int env = warp_env0 + lane / KG;
    const bool valid = env < c.N && d < c.K;
    const int gi = env * c.K + d;
    const int warp_rows = max(0, min(GPW, c.N - warp_env0)) * c.K;      // valid rows of this warp-tile

    Drone q;
    float4 act = make_float4(0.f, 0.f, 0.f, 0.f);
    int tick = 0, svd = 0;
    // The RNG counter is (global env id, launch counter, site | drone | aux, block): nothing in it is loaded from memory, so the
    // step's regular draws can be generated while the state loads are in flight (below)
    Rng g; g.k0 = c.key0; g.k1 = c.key1; g.gid = 0; g.step = c.rng_step;
    int scen_now = 0;
    float4 ring = make_float4(0.f, 0.f, 0.f, 0.f), sums = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 sc_row[(QS_SC_COUNT / 4 + KG - 1) / KG];
    float2 ob_v[4];                                                     // obstacle centres: issued first, they depend on nothing
    if (OBST) {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int k = lane + 32 * t, e = k / c.M, m = k - e * c.M;
            ob_v[t] = (k < ob_per_warp && warp_env0 + e < c.N) ? __ldcs(P.obst_xy + (size_t)(warp_env0 + e) * QS_MAX_OBSTACLES + m) : make_float2(0.f, 0.f);
        }
    }
    // ---- the step's regular draws -- OU thrust noise (numba_utils.py:103) and the sensor noise of the self observation
    // (sensor_noise.py:240-259) -- depend on (global env id, launch counter, drone) only, none of which is loaded: four Philox blocks +
    // Box-Muller (~15 % of the step's instructions) run in the shadow of the state's trip from HBM instead of after it.  The
    // generator is inlined in a rolled 4-trip loop (a call would make the compiler move in-flight load destinations out of the
    // callee's registers first, i.e. wait for the loads) and parks its 16 normals in the thread's shared-memory slots, so they
    // hold no registers while the dynamics run.
    // PFM: prefetch the state rows into L2 before the draws -- measured per variant (profiles/README.md round 2)
    constexpr int PFM = (SCEN || KG >= 32) ? 1 : 0;
    float4 *nz = reinterpret_cast<float4 *>(smem + park_off) + threadIdx.x;      // [4][blockDim.x]
    const int nz_stride = blockDim.x;
    int *sl = reinterpret_cast<int *>(smem + park_off + 16 * blockDim.x) + 3 * threadIdx.x;
    auto early_draws = [&]() {
        const int nblk = c.sense_noise ? 4 : 1;
#pragma unroll 1
        for (int i = 0; i < nblk; ++i) {
            const uint32_t c2 = (i == 0 ? (uint32_t)SITE_OU : (uint32_t)SITE_SENSOR) | ((uint32_t)d << 8);
            const uint4 r = philox4x32_10(g.gid, g.step, c2, i == 0 ? 0u : (uint32_t)(i - 1), g.k0, g.k1);
            float4 n;
            box_muller(r.x, r.y, n.x, n.y);
            box_muller(r.z, r.w, n.z, n.w);
            nz[i * nz_stride] = n;
        }
    };
    // Every prologue load is UNCONDITIONAL on a clamped, always-valid row (lanes past the batch / past K re-read a valid row and are
    // overwritten below): one straight-line block, so that all loads are issued before the first consumer.  Under `if (valid)` the
    // compiler closed the divergent region with register moves of the loaded values in front of the per-env scalar loads -- a
    // second serialised HBM round trip at the top of every warp (profiles/tools/prologue_check.py guards this in the SASS).
    const int env_c = min(env, c.N - 1), gi_c = env_c * c.K + min(d, c.K - 1);
    g.gid = (uint32_t)(c.env_id_offset + env_c);
    if (PFM) {
        // Pending register loads in front of the generator loop make the compiler copy some of their destinations out of the loop's
        // registers first -- i.e. wait for the first load.  So the rows are PREFETCHED (no destination registers), the draws run
        // while they travel from HBM, and the loads proper follow as cache hits.
#pragma unroll
        for (int pl = 0; pl < PL_COUNT; ++pl) prefetch_row(P.plane[pl] + gi_c);
        prefetch_row(actions + gi_c);
        if (d == 0) { prefetch_row(P.tick + env_c); prefetch_row(P.svd_ctr + env_c); }
        if (HOT) { cp_async4(sl + 2, P.hot_flag_cur + min(wt, n_wt - 1)); cp_async_commit(); }
        early_draws();
        if (HOT) {
            cp_async_wait_all();
            if (!hot_role && sl[2] != 0) {
                if (lane == 0 && wt < n_wt) P.hot_flag_cur[wt] = 0;
                return;
            }
        }
        tick = P.tick[env_c]; svd = P.svd_ctr[env_c];
    } else {
        // The two per-env scalars travel global -> shared (LDGSTS) and are read after the draws below: as pending register loads
        // the compiler copied them out of the generator loop's registers first, i.e. waited for them before the loop.
        cp_async4(sl, P.tick + env_c); cp_async4(sl + 1, P.svd_ctr + env_c);
        if (HOT) cp_async4(sl + 2, P.hot_flag_cur + min(wt, n_wt - 1));
        cp_async_commit();
    }
    if (SCEN) {                                                         // scenario row: loaded with the state, parked in shared memory
#pragma unroll
        for (int k = 0; k < (QS_SC_COUNT / 4 + KG - 1) / KG; ++k)
            sc_row[k] = P.scen[(size_t)env_c * (QS_SC_COUNT / 4) + min(d + k * KG, QS_SC_COUNT / 4 - 1)];
    }
    load_drone(P, gi_c, q);
    act = __ldcs(actions + gi_c);
    // The last-5-s window sums (:762-767) are only needed in the last 500 steps of an episode, but the load is unconditional: a
    // predicate on `tick` made the compiler wait for the tick load BEFORE issuing the state loads (79.0 -> 76.6 us for 16 extra
    // bytes read per drone-step).
    ring = __ldcs(P.plane[PL_DIST_RING] + gi_c);
    sums = __ldcs(P.plane[PL_DIST_SUMS] + gi_c);
    if (!PFM) {
        early_draws();
        cp_async_wait_all();
        tick = sl[0]; svd = sl[1];
        if (HOT && !hot_role && sl[2] != 0) {                           // a hot block processes this tile in this step
            if (lane == 0 && wt < n_wt) P.hot_flag_cur[wt] = 0;         // leave the buffer clean for its next use
            return;
        }
    }
    if (env >= c.N) { tick = 0; svd = 0; }                              // first consumer of a loaded value: after the draws
    if (SCEN) {
        if (env < c.N) {
#pragma unroll
            for (int k = 0; k < (QS_SC_COUNT / 4 + KG - 1) / KG; ++k)
                if (d + k * KG < QS_SC_COUNT / 4) sc_sm[(lane / KG) * (QS_SC_COUNT / 4) + d + k * KG] = sc_row[k];
        }
        __syncwarp();
    }
    if (!valid) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { q.p[a] = 1.0e6f * (float)(lane + 1); q.v[a] = 0.f; q.w[a] = 0.f; q.goal[a] = 0.f; }
#pragma unroll
        for (int a = 0; a < 9; ++a) q.R[a] = (a % 4 == 0) ? 1.f : 0.f;
#pragma unroll
        for (int a = 0; a < 4; ++a) { q.rd[a] = q.cd[a] = q.ou[a] = 0.f; }
        q.flags = 0; q.colmask = 0;
    }
    if (OBST) {
        // obstacle centres of this warp-tile's envs -> shared memory.  The first 128 were loaded before the state (above); every
        // load is issued before the first shared-memory store (a load -> store loop serialises one HBM round trip per trip)
#pragma unroll
        for (int t = 0; t < 4; ++t) if (lane + 32 * t < ob_per_warp) ob_sm[lane + 32 * t] = ob_v[t];
        for (int k0 = lane + 128; k0 < ob_per_warp; k0 += 128) {        // more than 32 obstacles per env: further trips
            float2 v[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int k = k0 + 32 * t, e = k / c.M, m = k - e * c.M;
                v[t] = (k < ob_per_warp && warp_env0 + e < c.N) ? __ldcs(P.obst_xy + (size_t)(warp_env0 + e) * QS_MAX_OBSTACLES + m) : make_float2(0.f, 0.f);
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) if (k0 + 32 * t < ob_per_warp) ob_sm[k0 + 32 * t] = v[t];
        }
        __syncwarp();
    }

    // ---- per-drone: RawControl.step -> QuadrotorDynamics.step (quadrotor_control.py:53-57, quadrotor_dynamics.py:215-221)
    const int time_remain = c.ep_len - tick;                           // quadrotor_single.py:361
    float a4[4] = { act.x, act.y, act.z, act.w }, cmd[4];
#pragma unroll
    for (int m = 0; m < 4; ++m) cmd[m] = 0.5f * (clampf(a4[m], -1.0f, 1.0f) + 1.0f);
    if (valid) {
        const float4 nv = nz[0];                                       // OUNoiseNumba.noise, numba_utils.py:101-105
        const float n[4] = { nv.x, nv.y, nv.z, nv.w };
#pragma unroll
        for (int m = 0; m < 4; ++m) q.ou[m] = q.ou[m] + (c.ou_theta * (0.0f - q.ou[m]) + c.ou_sigma * n[m]);
        for (int s = 0; s < c.sim_steps; ++s) {
            svd += 1;
            bool fire = svd >= c.svd_period;
            if (fire) svd = 0;
            dynamics_substep(c, g, d, q, cmd, s, fire);
        }
        store_motor_planes(P, gi, q);                                  // final (a reset below rewrites them): 12 registers less from here on
    }
    // ---- compute_reward_weighted (quadrotor_single.py:34-92), dt = physics dt
    const bool on_floor = (q.flags & F_ON_FLOOR) != 0;
    const float dist = norm3f(q.goal[0] - q.p[0], q.goal[1] - q.p[1], q.goal[2] - q.p[2]);
    float reward;
    {
        float effort = sqrtf(a4[0] * a4[0] + a4[1] * a4[1] + a4[2] * a4[2] + a4[3] * a4[3]);
        float orient = on_floor ? 1.0f : -q.R[8];
        float spin = norm3f(q.w[0], q.w[1], q.w[2]);
        float crash = on_floor ? 1.0f : 0.0f;
        reward = -c.dt * (c.rew_pos * dist + c.rew_effort * effort + c.rew_crash * crash + c.rew_orient * orient + c.rew_spin * spin);
        // infos[i]["rewards"] raw terms, each scaled by dt like the reference's rew_info (quadrotor_single.py:69-84)
        if (__builtin_expect(P.rew_info != nullptr, 0) && valid) P.rew_info[2 * gi] = make_float4(-c.dt * dist, -c.dt * effort, -c.dt * crash, -c.dt * orient);
    }
    tick += 1;
    // a non-finite state cannot be stepped further: force-reset the env and count it (reference raises, quadrotor_single.py:87-90)
    float chk = q.p[0] + q.p[1] + q.p[2] + q.v[0] + q.v[1] + q.v[2] + q.w[0] + q.w[1] + q.w[2] + q.R[0] + q.R[4] + q.R[8] + reward;
    const bool bad = valid && !isfinite(chk);
    const uint32_t bad_ballot = __ballot_sync(QS_FULL, bad) & gmask;
    const bool all_done = (tick > c.ep_len) || (bad_ballot != 0u);     // quadrotor_single.py:366-367

    // ---- 1.1 drone-drone collisions (collisions/quadrotors.py:63-103, quadrotor_multi.py:537-568)
    uint32_t rowmask = 0u;
    float prox = 0.f;
    if (KG > 1) {
        const float pen_ratio = -c.rew_col_smooth / c.thr_fall;
        stage[2 * lane] = make_float4(q.p[0], q.p[1], q.p[2], 0.f);
        __syncwarp(gmask);
        // pre-filter on the squared distance (slightly widened), exact `<=` tests on the rounded distance only for near pairs
        const float thr_far = fmaxf(c.thr_col, c.thr_fall), fall2 = thr_far * thr_far * 1.0001f;
        // four iterations in flight: rolled (one at a time) every iteration waited out its own shared-memory load (80.6 vs 84.6 us);
        // fully unrolled the hot code outgrows the instruction cache again (QS_PAIR_UNROLL is a tuning knob).  The formation-scenario
        // variant, whose hot code is larger, stays rolled (100.8 vs 103.8 us)
        QS_UNROLL((SCEN ? 1 : QS_PAIR_UNROLL))
        for (int j = 0; j < KG; ++j) {
            float4 o4 = stage[2 * (base + j)];
            float dx = q.p[0] - o4.x, dy = q.p[1] - o4.y, dz = q.p[2] - o4.z;
            float d2 = dx * dx + dy * dy + dz * dz;
            bool other = (j != d) && (j < c.K) && valid;
            if (other && d2 <= fall2) {
                float dd = __fsqrt_rn(d2);
                if (dd <= c.thr_col) rowmask |= 1u << j;
                if (dd <= c.thr_fall) prox += pen_ratio * dd + c.rew_col_smooth;
            }
        }
    }
    const uint32_t new_pairs = rowmask & ~q.colmask;                   // :545-546
    const bool is_unique = (rowmask != 0u) && (q.colmask == 0u);       // setdiff1d over flattened ids, :548
    const uint32_t uniq_ballot = __ballot_sync(QS_FULL, is_unique) & gmask;
    const int n_unique = __popc(uniq_ballot);
    const bool unique_any_nonzero = (uniq_ballot & ~(1u << base)) != 0u;   // `.any()` drops a lone agent 0, :611
    const int col_tick = n_unique >> 1;                                // :557
    const bool settled = (float)tick >= c.grace_steps;
    if (col_tick > 0 && settled && is_unique) q.flags |= F_COL_AGENT;  // agent_col_agent, :560-563

    // ---- 1.2 obstacles (obstacles/utils.py:31-43, quadrotor_multi.py:571-597)
    int obst_hit = -1;
    bool obst_new = false;
    if (OBST) {
        // positions are final for this step (impulses only touch vel / omega), so the SDF patch of the observation is
        // produced here in the same pass as the hit test and goes straight into the warp's observation tile
        if (valid) obstacle_sdf_and_hit(c, ob_env, q.p[0], q.p[1], orow + c.S + ((c.nbr_type == QS_NEIGHBOR_POS_VEL) ? 6 * c.V : 0), obst_hit);
        obst_new = (obst_hit >= 0) && !(q.flags & F_PREV_OBST);
        q.flags = (obst_hit >= 0) ? (q.flags | F_PREV_OBST) : (q.flags & ~F_PREV_OBST);
    }
    const uint32_t obst_ballot = __ballot_sync(QS_FULL, obst_new) & gmask;
    const int n_obst_new = __popc(obst_ballot);
    if (n_obst_new > 0 && settled && obst_new) q.flags |= F_COL_OBST;

    // ---- 1.3 room (quadrotor_multi.py:390-403, 600-606): prev lists hold last step's NEW crashes
    const bool new_wall = (q.flags & F_CR_WALL) && !(q.flags & F_PREV_WALL);
    const bool new_ceil = (q.flags & F_CR_CEIL) && !(q.flags & F_PREV_CEIL);
    const bool cr_floor = (q.flags & F_CR_FLOOR) != 0;
    const bool new_room = (cr_floor || new_wall || new_ceil) && !(q.flags & F_PREV_ROOM);
    q.flags = (q.flags & ~(F_PREV_WALL | F_PREV_CEIL | F_PREV_ROOM)) | (new_wall ? F_PREV_WALL : 0) | (new_ceil ? F_PREV_CEIL : 0) |
              (new_room ? F_PREV_ROOM : 0);
    const uint32_t wall_ballot = __ballot_sync(QS_FULL, new_wall) & gmask;
    const uint32_t ceil_ballot = __ballot_sync(QS_FULL, new_ceil) & gmask;
    const uint32_t floor_ballot = __ballot_sync(QS_FULL, cr_floor && valid) & gmask;
    const uint32_t room_ballot = __ballot_sync(QS_FULL, new_room) & gmask;
    const uint32_t pair_ballot = __ballot_sync(QS_FULL, new_pairs != 0u) & gmask;

    // ---- 2. rewards (quadrotor_multi.py:610-655)
    reward += c.rew_col * ((unique_any_nonzero && is_unique) ? -1.0f : 0.0f);
    reward += -1.0f * (c.control_dt * prox);
    if (OBST) reward += c.rew_col_obst * (obst_new ? -1.0f : 0.0f);
    if (__builtin_expect(P.rew_info != nullptr, 0) && valid)          // (:642-649) rewraw_spin, rewraw_quadcol, rew_proximity, rewraw_quadcol_obstacle
        P.rew_info[2 * gi + 1] = make_float4(-c.dt * norm3f(q.w[0], q.w[1], q.w[2]), (unique_any_nonzero && is_unique) ? -1.0f : 0.0f,
                                             -1.0f * (c.control_dt * prox), (OBST && obst_new) ? -1.0f : 0.0f);
    if (valid) { rew[gi] = reward; done[gi] = all_done ? 1 : 0; }      // final here: not carried (spilled) across the impulse / observation code

    if (OBST) scen_now = (q.flags & F_SCEN_OSTATIC) ? QS_SCENARIO_O_STATIC_SAME_GOAL : QS_SCENARIO_O_RANDOM;
    // distance_to_goal log: reached-goal flag from the mean of the last 5 entries, and the 1/3/5 s windows (:651-655, 762-767)
    if (valid) {
        float dlog = c.dt * dist;                                      // -rewraw_pos
        if (tick >= 5 && !(q.flags & F_REACHED)) {
            float m5 = (ring.x + ring.y + ring.z + ring.w + dlog) / 5.0f;
            float metric = (OBST && scen_now == QS_SCENARIO_O_STATIC_SAME_GOAL) ? 1.0f : c.approach_metric;
            if (m5 / c.dt < metric) q.flags |= F_REACHED;
        }
        P.plane[PL_DIST_RING][gi] = make_float4(ring.y, ring.z, ring.w, dlog);
        int steps_left = c.ep_len + 1 - tick;
        if (steps_left < 500) {                                         // == the prefetch condition (tick was incremented since)
            if (steps_left < 100) sums.x += dlog;
            if (steps_left < 300) sums.y += dlog;
            sums.z += dlog;
            P.plane[PL_DIST_SUMS][gi] = sums;
        }
    }

    // ---- 3. impulses (quadrotor_multi.py:659-698): rare, group-divergent
    bool flag = false;
    if (DOWNWASH && KG > 1) {
        // perform_downwash, aerodynamics/downwash.py:4-66: lane j accumulates the pushes of every source i in index order
        const float px0 = q.p[0], py0 = q.p[1], pz0 = q.p[2];
        // every drone publishes its position and body z axis; sources are read back as broadcast 16-byte loads
        __syncwarp(gmask);
        stage[2 * lane] = make_float4(px0, py0, pz0, 0.f);
        stage[2 * lane + 1] = make_float4(q.R[2], q.R[5], q.R[8], 0.f);
        __syncwarp(gmask);
        bool hit = false;
        QS_UNROLL(QS_DW_UNROLL)
        for (int i = 0; i < c.K; ++i) {
            const float4 sp = stage[2 * (base + i)];
            float rx = px0 - sp.x, ry = py0 - sp.y, rz = pz0 - sp.z;
            float d2 = rx * rx + ry * ry + rz * rz;
            // inside the wake cylinder (|relz| < 0.7, rxy < 0.1) means d^2 < 0.5: everything else is skipped on d^2 alone
            if (i != d && valid && d2 < 0.51f) {
                const float4 sz = stage[2 * (base + i) + 1];
                float dd = sqrtf(d2);
                float relz = rx * sz.x + ry * sz.y + rz * sz.z;
                float rxy = sqrtf(dd * dd - relz * relz);
                if (-0.7f < relz && relz < 0.f && rxy < 0.1f) {
                    float su[4];
                    rng_u4(g, SITE_DOWNWASH, i, 0xFF, 0, su);            // the source's own (a, w) jitter: same counter on every target
                    float acc = fmaxf(1e-6f, (6.0f / 17.0f) * (-10.0f * dd + 7.0f) + (-0.1f + 0.2f * su[0]));
                    float ow = fmaxf(1e-6f, 0.3f * (dd - 1.0f) * (dd - 1.0f) + (-0.01f + 0.02f * su[1]));
                    float u[4], t[4];
                    rng_u4(g, SITE_DOWNWASH, i, d, 0, u); rng_u4(g, SITE_DOWNWASH, i, d, 1, t);
                    float nx = sz.x + (-0.1f + 0.2f * u[0]), ny = sz.y + (-0.1f + 0.2f * u[1]), nz = sz.z + (-0.1f + 0.2f * u[2]);
                    float nm = norm3f(nx, ny, nz), den = (nm == 0.f) ? nm + 1e-6f : nm;
                    float wx = -1.f + 2.f * u[3], wy = -1.f + 2.f * t[0], wz = -1.f + 2.f * t[1];
                    float wm = norm3f(wx, wy, wz), wden = (wm == 0.f) ? wm + 1e-6f : wm;
                    q.v[0] += acc * (-nx / den) * c.control_dt; q.v[1] += acc * (-ny / den) * c.control_dt; q.v[2] += acc * (-nz / den) * c.control_dt;
                    q.w[0] += ow * (wx / wden) * c.control_dt; q.w[1] += ow * (wy / wden) * c.control_dt; q.w[2] += ow * (wz / wden) * c.control_dt;
                    hit = true;
                }
            }
        }
        flag = (__ballot_sync(QS_FULL, hit) & gmask) != 0u;
    }
    if (c.apply_force) {
        if (__builtin_expect(pair_ballot != 0u, 0)) {
            // new pairs in (i, j) lexicographic order; a drone in two pairs is updated twice (:674-677)
            for (int i = 0; i < c.K - 1; ++i) {
                uint32_t rowi = __shfl_sync(gmask, new_pairs, base + i) & ~((2u << i) - 1u);   // j > i
                while (rowi) {
                    int j = __ffs(rowi) - 1;
                    rowi &= rowi - 1;
                    float p1[3], p2[3], v1[3], v2[3], w1[3], w2[3];
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
                        p1[a] = __shfl_sync(gmask, q.p[a], base + i); p2[a] = __shfl_sync(gmask, q.p[a], base + j);
                        v1[a] = __shfl_sync(gmask, q.v[a], base + i); v2[a] = __shfl_sync(gmask, q.v[a], base + j);
                        w1[a] = __shfl_sync(gmask, q.w[a], base + i); w2[a] = __shfl_sync(gmask, q.w[a], base + j);
                    }
                    pair_impulse(g, i, j, p1, p2, v1, v2, w1, w2);
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
                        if (d == i) { q.v[a] = v1[a]; q.w[a] = w1[a]; }
                        if (d == j) { q.v[a] = v2[a]; q.w[a] = w2[a]; }
                    }
                }
            }
            flag = true;
        }
        if (__builtin_expect(OBST && obst_ballot, 0)) {
            if (obst_new) {
                float2 xy = P.obst_xy[(size_t)env * QS_MAX_OBSTACLES + obst_hit];
                float tp[3] = { q.p[0], q.p[1], q.p[2] }, tv[3] = { q.v[0], q.v[1], q.v[2] }, tw[3] = { q.w[0], q.w[1], q.w[2] };
                obstacle_impulse(c, g, d, tp, tv, tw, xy.x, xy.y);
#pragma unroll
                for (int a = 0; a < 3; ++a) { q.v[a] = tv[a]; q.w[a] = tw[a]; }
            }
            flag = true;
        }
        if (__builtin_expect((wall_ballot | ceil_ballot) != 0u, 0)) {
            if (new_wall || new_ceil) {
                float tv[3] = { q.v[0], q.v[1], q.v[2] }, tw[3] = { q.w[0], q.w[1], q.w[2] };
                if (new_wall) room_impulse(c, g, d, q.flags, tv, tw, true);
                if (new_ceil) room_impulse(c, g, d, q.flags, tv, tw, false);
#pragma unroll
                for (int a = 0; a < 3; ++a) { q.v[a] = tv[a]; q.w[a] = tw[a]; }
            }
            flag = true;
        }
    }
    q.colmask = rowmask;                                               // :568

    // ---- 4. scenario.step() (:701): goals may move.  The self observation below still belongs to the old goal unless an
    // impulse forces its recomputation (:711-712)
    float og[3] = { q.goal[0], q.goal[1], q.goal[2] };
    if (SCEN) {
        if (env < c.N) formation_scenario_step<KG>(c, g, d, valid && d == 0, gmask, lane, tick, sc_env, reinterpret_cast<float *>(P.scen + (size_t)env * (QS_SC_COUNT / 4)), stage, q.goal);
        if (flag) { og[0] = q.goal[0]; og[1] = q.goal[1]; og[2] = q.goal[2]; }
    }

    // ---- episode counters (leader lane) (:557-565, 578-581, 631-635)
    if (valid && d == 0) {
        int *ec = P.ecnt + env * EC_COUNT;
        if (col_tick > 0) {
            ec[EC_COL] += col_tick;
            if (settled) ec[EC_COL_SETTLE] += col_tick;
            if ((float)time_remain <= c.final_grace_steps) ec[EC_COL_FINAL] += col_tick;
        }
        if (n_obst_new > 0) { ec[EC_OBST] += n_obst_new; if (settled) ec[EC_OBST_SETTLE] += n_obst_new; }
        if (settled && (room_ballot | floor_ballot | wall_ballot | ceil_ballot)) {
            ec[EC_ROOM] += __popc(room_ballot); ec[EC_FLOOR] += __popc(floor_ballot);
            ec[EC_WALL] += __popc(wall_ballot); ec[EC_CEIL] += __popc(ceil_ballot);
        }
    }

    // ---- 5. observations (:703-720).  Self obs carries fresh sensor noise if any impulse fired (:711-712)
    float vs[3] = { q.v[0], q.v[1], q.v[2] };                          // self.vel snapshot, :705-709
    if (valid) {
        if (SCEN) { float t; t = q.goal[0]; q.goal[0] = og[0]; og[0] = t; t = q.goal[1]; q.goal[1] = og[1]; og[1] = t; t = q.goal[2]; q.goal[2] = og[2]; og[2] = t; }
        // fresh sensor noise only if an impulse forced the observation to be recomputed (:711-712); otherwise the draws made above
        SensorNoise sn;
        sn.n = sn.m = sn.l = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c.sense_noise) {
            if (__builtin_expect(flag, 0)) sn = sensor_noise(g, flag ? SITE_SENSOR_IMPULSE : SITE_SENSOR, d);
            else { sn.n = nz[nz_stride]; sn.m = nz[2 * nz_stride]; sn.l = nz[3 * nz_stride]; }
        }
        self_obs(c, sn, q, orow);
        if (SCEN) { q.goal[0] = og[0]; q.goal[1] = og[1]; q.goal[2] = og[2]; }
    }
    group_obs_tail<KG, OBST, false, SCEN>(c, ob_env, d, lane, gmask, valid, q, vs, orow, stage);
    // ---- 7. dones (:739-838): episode stats, then the env resets itself and returns the new episode's first observation
    const uint32_t done_ballot = __ballot_sync(QS_FULL, all_done && valid);
    if (__builtin_expect(done_ballot != 0u, 0)) {
        __syncwarp();
        if (term_obs != nullptr) {
            // terminal observation of the finished episode (rows of envs that go on are left untouched)
            for (int r = 0; r < warp_rows; ++r) {
                int src_lane = (r / c.K) * KG;                         // leader lane of that row's env
                if ((done_ballot >> src_lane) & 1u) {
                    const float *s = tile + (size_t)r * c.D;
                    float *t = term_obs + ((size_t)warp_env0 * c.K + r) * c.D;
                    for (int k = lane; k < c.D; k += 32) t[k] = s[k];
                }
            }
            __syncwarp();
        }
        if (all_done) {
            int *ec = P.ecnt + env * EC_COUNT;
            qs_stats *st = P.stats;
            {
                bool col = (q.flags & (F_COL_AGENT | F_COL_OBST)) != 0, reached = (q.flags & F_REACHED) != 0;
                uint32_t b_succ = __ballot_sync(gmask, !col && reached && valid) & gmask;
                uint32_t b_dead = __ballot_sync(gmask, !col && !reached && valid) & gmask;
                uint32_t b_col = __ballot_sync(gmask, col && valid) & gmask;
                float4 sums = valid ? P.plane[PL_DIST_SUMS][gi] : make_float4(0.f, 0.f, 0.f, 0.f);
                float inv_dt = 1.0f / c.dt;
                float m1 = inv_dt * sums.x / (float)min(100, tick), m3 = inv_dt * sums.y / (float)min(300, tick), m5 = inv_dt * sums.z / (float)min(500, tick);
                if (bad_ballot) {                                       // a diverged env must not poison the aggregates: its record and sums carry zeros
                    m1 = isfinite(m1) ? m1 : 0.f; m3 = isfinite(m3) ? m3 : 0.f; m5 = isfinite(m5) ? m5 : 0.f;
                }
                // per-episode record (infos[i]['episode_extra_stats'], :739-831): per-drone part, then the env row below
                if (valid) P.ep_agent[gi] = make_float4(m1, m3, m5, 0.f);
                const uint32_t b_ncol = __ballot_sync(gmask, (q.flags & F_COL_AGENT) && valid) & gmask;
                const uint32_t b_ocol = __ballot_sync(gmask, (q.flags & F_COL_OBST) && valid) & gmask;
#pragma unroll
                for (int off = KG / 2; off > 0; off >>= 1) {
                    m1 += __shfl_xor_sync(gmask, m1, off); m3 += __shfl_xor_sync(gmask, m3, off); m5 += __shfl_xor_sync(gmask, m5, off);
                }
                if (valid && d == 0) {
                    int *er = P.ep_rec + (size_t)env * QS_ER_COUNT;
                    er[QS_ER_SEQ] += 1;
                    er[QS_ER_SCENARIO] = OBST ? scen_now : (SCEN ? (int)sc_env[0].x : QS_SCENARIO_STATIC_SAME_GOAL);
#pragma unroll
                    for (int k = 0; k < 9; ++k) er[QS_ER_NUM_COLLISIONS + k] = ec[k];
                    er[QS_ER_AGENTS_SUCCESS] = __popc(b_succ); er[QS_ER_AGENTS_DEADLOCK] = __popc(b_dead); er[QS_ER_AGENTS_COLLIDED] = __popc(b_col);
                    er[QS_ER_AGENTS_NEIGHBOR_COL] = __popc(b_ncol); er[QS_ER_AGENTS_OBST_COL] = __popc(b_ocol);
                    er[QS_ER_EP_LEN] = tick; er[QS_ER_SUCCESS] = 0; er[QS_ER_NONFINITE] = bad_ballot ? 1 : 0;
                }
                if (valid && d == 0) {
                    atomicAdd((unsigned long long *)&st->episodes, 1ull);
                    atomicAdd((unsigned long long *)&st->num_collisions, (unsigned long long)ec[EC_COL]);
                    atomicAdd((unsigned long long *)&st->num_collisions_after_settle, (unsigned long long)ec[EC_COL_SETTLE]);
                    atomicAdd((unsigned long long *)&st->num_collisions_final_5s, (unsigned long long)ec[EC_COL_FINAL]);
                    atomicAdd((unsigned long long *)&st->num_collisions_with_room, (unsigned long long)ec[EC_ROOM]);
                    atomicAdd((unsigned long long *)&st->num_collisions_with_floor, (unsigned long long)ec[EC_FLOOR]);
                    atomicAdd((unsigned long long *)&st->num_collisions_with_wall, (unsigned long long)ec[EC_WALL]);
                    atomicAdd((unsigned long long *)&st->num_collisions_with_ceiling, (unsigned long long)ec[EC_CEIL]);
                    atomicAdd((unsigned long long *)&st->num_collisions_obst_quad, (unsigned long long)ec[EC_OBST]);
                    atomicAdd((unsigned long long *)&st->num_collisions_obst_quad_after_settle, (unsigned long long)ec[EC_OBST_SETTLE]);
                    atomicAdd((unsigned long long *)&st->agents_success, (unsigned long long)__popc(b_succ));
                    atomicAdd((unsigned long long *)&st->agents_deadlock, (unsigned long long)__popc(b_dead));
                    atomicAdd((unsigned long long *)&st->agents_collided, (unsigned long long)__popc(b_col));
                    if (bad_ballot) atomicAdd((unsigned long long *)&st->nonfinite_resets, 1ull);
                    if (reset_success != nullptr) reset_success[env] = 0;   // upstream reset() reports no success flag
                    atomicAdd(&st->distance_to_goal_1s, (double)m1);
                    atomicAdd(&st->distance_to_goal_3s, (double)m3);
                    atomicAdd(&st->distance_to_goal_5s, (double)m5);
                }
            }
            int scen = 0;
            if (bad_ballot) {                                           // do not let NaNs leak through the persistent noise state
                if (valid) { const float4 h = P.plane[PL_OU][gi]; q.ou[0] = h.x; q.ou[1] = h.y; q.ou[2] = h.z; q.ou[3] = h.w; }   // written above by this thread
#pragma unroll
                for (int m = 0; m < 4; ++m) q.ou[m] = isfinite(q.ou[m]) ? q.ou[m] : 0.f;
                if (valid) P.plane[PL_OU][gi] = make_float4(q.ou[0], q.ou[1], q.ou[2], q.ou[3]);
                if (!isfinite(vs[0] + vs[1] + vs[2])) { vs[0] = vs[1] = vs[2] = 0.f; }
            }
            group_reset<KG, OBST, SCEN>(c, P, g, env, d, valid, gmask, tile + (size_t)(lane / KG) * c.K * c.D, c.K * c.D,
                                        OBST ? ob_sm + (lane / KG) * c.M : nullptr, q, scen);
            if (valid) {                                                // the motor lag restarts at rest (quadrotor_dynamics.py:176-178)
                P.plane[PL_ROT_DAMP][gi] = make_float4(0.f, 0.f, 0.f, 0.f);
                P.plane[PL_CMDS_DAMP][gi] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            tick = 0;
            if (valid) {
                if (d == 0) {
#pragma unroll
                    for (int k = 0; k < EC_COUNT; ++k) ec[k] = 0;
                    ec[EC_SCENARIO] = scen;
                }
                P.plane[PL_DIST_RING][gi] = make_float4(0.f, 0.f, 0.f, 0.f);
                P.plane[PL_DIST_SUMS][gi] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            __threadfence_block();                                      // obstacle centres written by the leader lane
            __syncwarp(gmask);
            if (valid) {
                SensorNoise sn;
                sn.n = sn.m = sn.l = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c.sense_noise) sn = sensor_noise(g, SITE_SENSOR_RESET, d);
                self_obs(c, sn, q, orow);
            }
            // the new obstacle centres are in the warp's staged copy as well (written by the group's first lane inside the reset)
            group_obs_tail<KG, OBST, true>(c, ob_env, d, lane, gmask, valid, q, vs, orow, stage);   // stale self.vel, quadrotor_multi.py:477-481
        }
        __syncwarp();
    }

    // ---- write back
    if (valid) {
        store_drone<false>(P, gi, q, SCEN || all_done);   // the motor planes were written after the dynamics
        if (d == 0) { P.tick[env] = tick; P.svd_ctr[env] = svd; }
    }
    if (HOT) {
        // tiles with an env that finishes its episode in the NEXT step (the tick is already advanced / reset): listed for the hot blocks
        const uint32_t nb = __ballot_sync(QS_FULL, valid && d == 0 && tick >= c.ep_len);
        if (nb != 0u && lane == 0) {
            const int idx = atomicAdd(P.hot_cnt_next, 1);
            if (idx < P.hot_cap) { P.hot_list_next[idx] = wt; P.hot_flag_next[wt] = 1; }
        }
    }
    __syncwarp();
    if (warp_rows > 0) warp_store_tile(tile, obs + (size_t)warp_env0 * c.K * c.D, warp_rows * c.D, lane);
    __syncwarp();
    }   // warp-tile loop
}

// ----------------------------------------------------------------------------------------------------------------
// explicit reset (QuadrotorEnvMulti.reset through VecEnv.reset)
// ----------------------------------------------------------------------------------------------------------------
template <int KG, bool OBST, bool SCEN>
__global__ void __launch_bounds__(128) reset_kernel(const __grid_constant__ DevConst c, const __grid_constant__ DevPtrs P,
                                                    const uint8_t *__restrict__ env_mask, float *__restrict__ obs)
{
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp_in_block = threadIdx.x >> 5;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int env = tid / KG, d = tid % KG;
    const bool in_range = env < c.N && d < c.K;
    const bool valid = in_range && (env_mask == nullptr || env_mask[env] != 0);
    const int gi = env * c.K + d;
    const uint32_t gmask = group_mask<KG>(lane);
    constexpr int GPW = 32 / KG;
    const int rows_per_warp = GPW * c.K;
    float4 *stage = reinterpret_cast<float4 *>(smem) + (size_t)warp_in_block * 64;
    float *tile = smem + (size_t)(blockDim.x >> 5) * 256 + (size_t)warp_in_block * rows_per_warp * c.D;
    const int row = (lane / KG) * c.K + d;
    float *orow = tile + (size_t)row * c.D;

    Drone q;
    Rng g; g.k0 = c.key0; g.k1 = c.key1; g.gid = 0; g.step = c.rng_step;
    float vs[3] = { 0.f, 0.f, 0.f };
    if (env < c.N) g.gid = (uint32_t)(c.env_id_offset + env);          // every lane of the group: the reset draws cooperatively
    if (in_range) {
        load_drone(P, gi, q);
        vs[0] = q.v[0]; vs[1] = q.v[1]; vs[2] = q.v[2];                 // self.vel is not refreshed by reset (quadrotor_multi.py:477)
    } else {
#pragma unroll
        for (int a = 0; a < 3; ++a) { q.p[a] = 0.f; q.v[a] = 0.f; q.w[a] = 0.f; q.goal[a] = 0.f; }
#pragma unroll
        for (int a = 0; a < 9; ++a) q.R[a] = 0.f;
#pragma unroll
        for (int a = 0; a < 4; ++a) { q.rd[a] = q.cd[a] = q.ou[a] = 0.f; }
        q.flags = 0; q.colmask = 0;
    }
    int scen = 0;
    const bool grp = env < c.N && (env_mask == nullptr || env_mask[env] != 0);      // uniform over the env's lane group
    if (grp) group_reset<KG, OBST, SCEN>(c, P, g, env, d, valid, gmask, tile + (size_t)(lane / KG) * c.K * c.D, c.K * c.D, nullptr, q, scen);
    if (valid) {
        if (d == 0) {
            int *ec = P.ecnt + env * EC_COUNT;
#pragma unroll
            for (int k = 0; k < EC_COUNT; ++k) ec[k] = 0;
            ec[EC_SCENARIO] = scen;
            P.tick[env] = 0;
        }
        P.plane[PL_DIST_RING][gi] = make_float4(0.f, 0.f, 0.f, 0.f);
        P.plane[PL_DIST_SUMS][gi] = make_float4(0.f, 0.f, 0.f, 0.f);
        store_drone(P, gi, q, true);
    }
    __threadfence_block();
    __syncwarp();
    if (valid) {
        SensorNoise sn;
        if (c.sense_noise) sn = sensor_noise(g, SITE_SENSOR_RESET, d);
        else sn.n = sn.m = sn.l = make_float4(0.f, 0.f, 0.f, 0.f);
        self_obs(c, sn, q, orow);
    }
    group_obs_tail<KG, OBST, true>(c, P.obst_xy + (size_t)(env < c.N ? env : 0) * QS_MAX_OBSTACLES, d, lane, gmask, valid, q, vs, orow, stage);
    __syncwarp();
    // rows of envs that were not reset stay untouched: per-row masked copy
    const int warp_env0 = (tid - lane) / KG;
    const int warp_rows = max(0, min(GPW, c.N - warp_env0)) * c.K;
    for (int r = 0; r < warp_rows; ++r) {
        int e = warp_env0 + r / c.K;
        if (env_mask == nullptr || env_mask[e] != 0) {
            const float *s = tile + (size_t)r * c.D;
            float *t = obs + ((size_t)warp_env0 * c.K + r) * c.D;
            for (int k = lane; k < c.D; k += 32) t[k] = s[k];
        }
    }
}

// ----------------------------------------------------------------------------------------------------------------
// state pack / unpack (qs_get_state / qs_set_state)
// ----------------------------------------------------------------------------------------------------------------
struct StateView {
    float *pos, *vel, *rot, *omega, *rot_damp, *cmds_damp, *ou, *goal;
    int *flags; uint32_t *col_mask; int *tick, *svd_ctr; uint32_t *step_ctr; float *obst_xy;
    float *scenario;                    // formation scenarios: [N, QS_SC_COUNT]
    float *pid, *heading, *evader;      // fork mode
};

// fork-mode planes (fork_kernels.cuh): 6 float4 planes of PID state + (angle, ang_vel, -, -); per env evader + flags
enum { FP_PID0 = 0, FP_HEADING = 6, FP_COUNT = 7 };
struct ForkPtrs {
    float4 *plane[FP_COUNT];   // each [N*K]
    float2 *evader;            // [N]
    int *flags;                // [N]
};

}  // namespace qs
