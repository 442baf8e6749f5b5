// quadsim.cu -- C-ABI (include/quadsim.h) over the sm_100a kernels in quadsim_kernels.cuh.
// Host side: owns the device state planes, converts qs_config to the kernel constant block, picks the launch shape.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "launch.h"

namespace qs {

// ----------------------------------------------------------------------------------------------------------------
// kernels that do not depend on the lane-group width live in this translation unit
// ----------------------------------------------------------------------------------------------------------------
__global__ void state_io_kernel(DevConst c, DevPtrs P, ForkPtrs F, StateView v, int set)
{
    const size_t gi = (size_t)blockIdx.x * blockDim.x + threadIdx.x;      // 24 * gi exceeds 2^31 at the largest admitted batches
    const size_t nd = (size_t)c.N * c.K;
    if (gi < nd) {
        Drone q;
        load_drone(P, (int)gi, q);                                       // gi < nd <= 2^30 (validate())
        if (set) {
            if (v.pos) for (int a = 0; a < 3; ++a) q.p[a] = v.pos[3 * gi + a];
            if (v.vel) for (int a = 0; a < 3; ++a) q.v[a] = v.vel[3 * gi + a];
            if (v.omega) for (int a = 0; a < 3; ++a) q.w[a] = v.omega[3 * gi + a];
            if (v.rot) for (int a = 0; a < 9; ++a) q.R[a] = v.rot[9 * gi + a];
            if (v.rot_damp) for (int a = 0; a < 4; ++a) q.rd[a] = v.rot_damp[4 * gi + a];
            if (v.cmds_damp) for (int a = 0; a < 4; ++a) q.cd[a] = v.cmds_damp[4 * gi + a];
            if (v.ou) for (int a = 0; a < 4; ++a) q.ou[a] = v.ou[4 * gi + a];
            if (v.goal) for (int a = 0; a < 3; ++a) q.goal[a] = v.goal[3 * gi + a];
            if (v.flags) q.flags = (v.flags[gi] & ~F_SCEN_OSTATIC) | (q.flags & F_SCEN_OSTATIC);   // the episode's scenario bit is not caller state
            if (v.col_mask) q.colmask = v.col_mask[gi];
            store_drone(P, (int)gi, q, true);
        } else {
            if (v.pos) for (int a = 0; a < 3; ++a) v.pos[3 * gi + a] = q.p[a];
            if (v.vel) for (int a = 0; a < 3; ++a) v.vel[3 * gi + a] = q.v[a];
            if (v.omega) for (int a = 0; a < 3; ++a) v.omega[3 * gi + a] = q.w[a];
            if (v.rot) for (int a = 0; a < 9; ++a) v.rot[9 * gi + a] = q.R[a];
            if (v.rot_damp) for (int a = 0; a < 4; ++a) v.rot_damp[4 * gi + a] = q.rd[a];
            if (v.cmds_damp) for (int a = 0; a < 4; ++a) v.cmds_damp[4 * gi + a] = q.cd[a];
            if (v.ou) for (int a = 0; a < 4; ++a) v.ou[4 * gi + a] = q.ou[a];
            if (v.goal) for (int a = 0; a < 3; ++a) v.goal[3 * gi + a] = q.goal[a];
            if (v.flags) v.flags[gi] = q.flags;
            if (v.col_mask) v.col_mask[gi] = q.colmask;
        }
    }
    if (gi < nd && F.plane[0] != nullptr) {
        if (v.pid) {
            for (int k = 0; k < 6; ++k) {
                if (set) F.plane[FP_PID0 + k][gi] = make_float4(v.pid[24 * gi + 4 * k], v.pid[24 * gi + 4 * k + 1], v.pid[24 * gi + 4 * k + 2], v.pid[24 * gi + 4 * k + 3]);
                else { float4 x = F.plane[FP_PID0 + k][gi]; v.pid[24 * gi + 4 * k] = x.x; v.pid[24 * gi + 4 * k + 1] = x.y; v.pid[24 * gi + 4 * k + 2] = x.z; v.pid[24 * gi + 4 * k + 3] = x.w; }
            }
        }
        if (v.heading) {
            if (set) F.plane[FP_HEADING][gi] = make_float4(v.heading[3 * gi], v.heading[3 * gi + 1], v.heading[3 * gi + 2], 0.f);
            else { float4 x = F.plane[FP_HEADING][gi]; v.heading[3 * gi] = x.x; v.heading[3 * gi + 1] = x.y; v.heading[3 * gi + 2] = x.z; }
        }
    }
    if (gi < (size_t)c.N && F.evader != nullptr && v.evader) {
        if (set) F.evader[gi] = make_float2(v.evader[2 * gi], v.evader[2 * gi + 1]);
        else { float2 x = F.evader[gi]; v.evader[2 * gi] = x.x; v.evader[2 * gi + 1] = x.y; }
    }
    if (gi < (size_t)c.N) {
        if (set) {
            if (v.tick) P.tick[gi] = v.tick[gi];
            if (v.svd_ctr) P.svd_ctr[gi] = v.svd_ctr[gi];
            // step_ctr: the RNG launch counter belongs to the handle (host side, state_io below)
        } else {
            if (v.tick) v.tick[gi] = P.tick[gi];
            if (v.svd_ctr) v.svd_ctr[gi] = P.svd_ctr[gi];
            if (v.step_ctr) v.step_ctr[gi] = c.rng_step;                // one counter per handle, reported per env
        }
    }
    if (v.scenario && P.scen) {
        const size_t tot = (size_t)c.N * QS_SC_COUNT;
        float *rows = reinterpret_cast<float *>(P.scen);
        for (size_t k = gi; k < tot; k += (size_t)gridDim.x * blockDim.x) {
            if (set) rows[k] = v.scenario[k];
            else v.scenario[k] = rows[k];
        }
    }
    if (v.obst_xy) {
        const size_t tot = (size_t)c.N * QS_MAX_OBSTACLES;
        for (size_t k = gi; k < tot; k += (size_t)gridDim.x * blockDim.x) {
            if (set) P.obst_xy[k] = make_float2(v.obst_xy[2 * k], v.obst_xy[2 * k + 1]);
            else { float2 xy = P.obst_xy[k]; v.obst_xy[2 * k] = xy.x; v.obst_xy[2 * k + 1] = xy.y; }
        }
    }
}

// raw generator probe used by the tests to pin the RNG contract bit-for-bit against the oracle
__global__ void philox_probe_kernel(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *out, float *fout)
{
    uint4 r = philox4x32_10(c0, c1, c2, c3, k0, k1);
    out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
    fout[0] = u23(r.x); fout[1] = u23(r.y);
    box_muller(r.x, r.y, fout[2], fout[3]);
    box_muller(r.z, r.w, fout[4], fout[5]);
}

// every rotation starts as the identity so that an env that was never reset is still a valid state
__global__ void init_identity_kernel(DevPtrs P, int nd)
{
    int gi = blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= nd) return;
    P.plane[PL_W_R0][gi] = make_float4(0.f, 1.f, 0.f, 0.f);      // omega.z, R00 R01 R02
    P.plane[PL_R1][gi] = make_float4(0.f, 1.f, 0.f, 0.f);        // R10 R11 R12 R20
    P.plane[PL_R2_FLAGS][gi] = make_float4(0.f, 1.f, 0.f, 0.f);  // R21 R22 flags colmask
}

}  // namespace qs

using namespace qs;

struct qs_env {
    qs_config cfg;
    DevConst dc;
    DevPtrs dp;
    ForkConst fc;
    ForkPtrs fp;
    bool fork;
    int A;                  // action dim
    int feat;               // upstream step kernel specialisation (bit 0 obstacles, bit 1 downwash, bit 2 formation scenarios)
    int device;
    int KG;                 // lanes per env
    int block;              // threads per block
    int grid;
    size_t smem_bytes;
    void *slab;             // one allocation for all device state
    size_t slab_bytes;
    // pinned host staging + device io buffers for the *_host entry points
    float *h_act, *h_obs, *h_rew, *h_term; uint8_t *h_done, *h_succ;
    float *d_act, *d_obs, *d_rew, *d_term; uint8_t *d_done, *d_succ;
    // qs_step_host pipeline: env chunks alternate between two internal streams so that the D2H of one chunk overlaps the H2D and
    // the kernel of the next
    cudaStream_t cs[2]; cudaEvent_t ev_in, ev_out[2]; bool pipe_ready;
    long long launches;
    // reset-first scheduling of the upstream step kernel (DevPtrs::hot_*): three rotating buffers in the slab
    int *hot_list[3], *hot_cnt[3], *hot_flag[3];
    int hot_cap, hot_blocks; unsigned hot_phase; bool hot;
    size_t hot_bytes;       // the three buffers back to back from hot_cnt[0]
    uint32_t rng_step;      // Philox counter word 1: +1 per step / reset call (+ fork.substeps per fork step); the same for every env of the handle
    bool host_ready;        // staging buffers of the *_host entry points are allocated
    std::string err;
};

static thread_local std::string g_create_err;

static int fail(qs_env *e, int code, const std::string &msg)
{
    if (e) e->err = msg; else g_create_err = msg;
    return code;
}

#define QS_CUDA(e, call)                                                                               \
    do {                                                                                               \
        cudaError_t _r = (call);                                                                       \
        if (_r != cudaSuccess) return fail(e, QS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_r)); \
    } while (0)

// makes `device` current for the scope of an entry point and restores the caller's device afterwards
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit DeviceGuard(int device)
    {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != device) switched = cudaSetDevice(device) == cudaSuccess;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

static int pow2_at_least(int k) { int p = 1; while (p < k) p <<= 1; return p; }

static void fill_const(const qs_config &c, DevConst &d)
{
    memset(&d, 0, sizeof(d));
    d.N = c.num_envs; d.K = c.num_agents; d.scenario = c.scenario; d.obs_repr = c.obs_repr;
    d.nbr_type = c.neighbor_obs_type; d.V = c.neighbor_visible_num; d.use_obstacles = c.use_obstacles;
    d.use_downwash = c.use_downwash; d.apply_force = c.apply_collision_force; d.sense_noise = c.sense_noise;
    d.ep_len = c.ep_len; d.sim_steps = c.sim_steps; d.svd_period = c.svd_period;
    d.obst_L = c.obst_area_len; d.obst_W = c.obst_area_wid; d.M = c.num_obstacles;
    if (c.env_mode == QS_MODE_FORK) {
        d.S = (c.obs_repr == QS_OBS_CDIST_CDISTDOT_DIST_DISTDOT_SANGLE_ANGLEDOT || c.obs_repr == QS_OBS_CDIST_CDISTDOT_NDIST_DISTDOT_NSANGLE_ANGLEDOT) ? 7 : 6;
        int W = 0;
        switch (c.neighbor_obs_type) {
            case QS_NEIGHBOR_DIST_ANGLE: W = 2; break;
            case QS_NEIGHBOR_DIST_SANGLE: case QS_NEIGHBOR_DIST_ANGLE_HEADING: case QS_NEIGHBOR_NDIST_NSANGLE: W = 3; break;
            case QS_NEIGHBOR_DIST_SANGLE_SHEADING: W = 5; break;
            default: break;
        }
        d.D = d.S + W * c.neighbor_visible_num;
    } else {
        d.S = c.obs_repr == QS_OBS_XYZ_VXYZ_R_OMEGA_FLOOR ? 19 : (c.obs_repr == QS_OBS_XYZ_VXYZ_R_OMEGA_WALL ? 24 : 18);
        d.D = d.S + (c.neighbor_obs_type == QS_NEIGHBOR_POS_VEL ? 6 * c.neighbor_visible_num : 0) + (c.use_obstacles ? 9 : 0);
    }
    d.key0 = (uint32_t)c.seed; d.key1 = (uint32_t)(c.seed >> 32);
    d.env_id_offset = c.env_id_offset;
    d.dt = (float)c.dt;
    d.hx = (float)(c.room_dims[0] / 2); d.hy = (float)(c.room_dims[1] / 2); d.hz = (float)c.room_dims[2];
    d.room_l = (float)c.room_dims[0]; d.room_w = (float)c.room_dims[1]; d.room_h = (float)c.room_dims[2];
    d.gravity = (float)c.gravity; d.mass = (float)c.mass; d.inv_mass = (float)(1.0 / c.mass);
    for (int a = 0; a < 3; ++a) { d.inertia[a] = (float)c.inertia[a]; d.inv_inertia[a] = (float)(1.0 / c.inertia[a]); }
    for (int m = 0; m < 4; ++m) {
        d.thrust_max[m] = (float)c.thrust_max[m]; d.torque_max[m] = (float)c.torque_max[m];
        d.pcx[m] = (float)c.prop_cross[m][0]; d.pcy[m] = (float)c.prop_cross[m][1]; d.pcz[m] = (float)c.prop_cross[m][2];
        d.ccw[m] = (float)c.prop_ccw[m];
    }
    d.arm = (float)c.arm; d.tau_up = (float)c.motor_tau_up; d.tau_down = (float)c.motor_tau_down; d.lin = (float)c.motor_linearity;
    d.vel_damp = (float)c.vel_damp; d.damp_wq = (float)c.damp_omega_quadratic; d.omega_max = (float)c.omega_max; d.mu = (float)c.floor_mu;
    d.ou_theta = (float)c.ou_theta; d.ou_sigma = (float)c.ou_sigma;
    d.s_pos = (float)c.sense_pos_std; d.s_vel = (float)c.sense_vel_std; d.s_gyro = (float)c.sense_gyro_std;
    d.rew_pos = (float)c.rew_pos; d.rew_effort = (float)c.rew_effort; d.rew_crash = (float)c.rew_crash;
    d.rew_orient = (float)c.rew_orient; d.rew_spin = (float)c.rew_spin; d.rew_col = (float)c.rew_quadcol_bin;
    d.rew_col_smooth = (float)c.rew_quadcol_bin_smooth_max; d.rew_col_obst = (float)c.rew_quadcol_bin_obst;
    d.thr_col = (float)(c.collision_hitbox_radius * c.arm); d.thr_fall = (float)(c.collision_falloff_radius * c.arm);
    d.thr_obst = (float)(c.arm + c.obst_size / 2.0); d.obst_rad = (float)(c.obst_size / 2.0); d.sdf_res = (float)c.sdf_resolution;
    d.spawn_box = (float)c.spawn_box; d.spawn_min_z = (float)c.spawn_min_z; d.approach_metric = (float)c.approach_goal_metric;
    double control_freq = std::floor(1.0 / c.dt + 0.5) / c.sim_steps;      // sim_freq / sim_steps (quadrotor_single.py:160)
    d.grace_steps = (float)(1.5 * control_freq);                           // quadrotor_multi.py:156
    d.final_grace_steps = (float)(5.0 * control_freq);                     // quadrotor_multi.py:160
    d.control_dt = (float)(1.0 / control_freq);                            // quadrotor_multi.py:91
    d.control_freq = (float)control_freq;
    for (int a = 0; a < 3; ++a) d.cube_dim[a] = c.cube_dim[a] > 0 ? c.cube_dim[a] : 1;
    d.small_angle = (std::sqrt(3.0) * c.omega_max * c.dt * 0.5 <= 0.25) ? 1 : 0;
    d.lin_one = (c.motor_linearity == 1.0) ? 1 : 0;
    d.no_omega_damp = (c.damp_omega_quadratic == 0.0) ? 1 : 0;
}

static void fill_fork(const qs_config &c, ForkConst &f)
{
    memset(&f, 0, sizeof(f));
    const qs_fork_config &s = c.fork;
    f.substeps = s.substeps;
    f.capture_radius = (float)s.capture_radius; f.rew_existence = (float)s.rew_existence; f.rew_captor = (float)s.rew_captor;
    f.rew_helper = (float)s.rew_helper; f.max_angular_rate = (float)s.max_angular_rate; f.chaser_speed = (float)s.chaser_speed;
    f.ev_vmax = (float)s.evader_v_max; f.ev_dt = (float)s.evader_dt; f.ev_arena = (float)s.evader_arena;
    f.spawn_ring = (float)s.spawn_ring; f.ev_rmin = (float)s.evader_r_min; f.ev_rspan = (float)s.evader_r_span;
    for (int i = 0; i < 12; ++i) {
        for (int k = 0; k < 3; ++k) f.pid[i][k] = (float)s.pid[i][k];
        f.pid[i][3] = s.pid[i][3] > 0 ? (float)s.pid[i][3] : INFINITY;      // saturation disabled -> +inf (branch-free clamp)
        f.pid[i][4] = s.pid[i][4] > 0 ? (float)s.pid[i][4] : -1.0f;         // anti-windup disabled -> empty interval
    }
    f.rate_scale = (float)s.rate_out_scale;
    for (int i = 0; i < 4; ++i) for (int k = 0; k < 4; ++k) f.mixer[i][k] = (float)s.mixer[i][k];
    f.mass = (float)s.ctrl_mass; f.g = (float)s.ctrl_g; f.inv_kf4 = (float)(1.0 / (s.ctrl_kf * 4.0));
    f.min_rpm = (float)s.ctrl_min_rpm; f.inv_rpm_span = (float)(1.0 / (s.ctrl_max_rpm - s.ctrl_min_rpm));
    f.half_len = (float)(c.room_dims[0] / 2.0);
    const double PI = 3.14159265358979323846;
    const double w = 2.0 * std::tan((s.cam_fov_deg / 2.0) * PI / 180.0) * s.cam_focal_length;      // sensor width, :289
    f.cam_r = (float)(s.cam_target_size / 2.0);
    // u_px = u * res / w + noise  ->  u / f = (x_y / x_x) + noise * w / (res * f)
    f.cam_noise_tan = (s.cam_resolution > 0 && s.cam_focal_length > 0) ? (float)(s.cam_pixel_noise * w / (s.cam_resolution * s.cam_focal_length)) : 0.f;
    f.cam_num = s.cam_num > 0 ? s.cam_num : 1;
    f.cam_seg = (float)(2.0 * PI / f.cam_num); f.cam_inv_seg = (float)(f.cam_num / (2.0 * PI));
}

static int validate(const qs_config *c, std::string &why)
{
    if (c->num_envs >= 1 && c->num_agents >= 1 && (long long)c->num_envs * 32 > (1ll << 30)) { why = "num_envs too large for 32-bit lane indices (<= 2^25)"; return 0; }
    if (c->env_mode == QS_MODE_FORK) {
        if (c->api_version != QS_API_VERSION) { why = "api_version mismatch"; return 0; }
        if (c->num_envs < 1) { why = "num_envs < 1"; return 0; }
        if (c->num_agents < 1 || c->num_agents > QS_MAX_AGENTS) { why = "num_agents out of [1, 32]"; return 0; }
        if (c->scenario != QS_SCENARIO_DYNAMIC_REPULSIVE) { why = "fork mode supports quads_mode dynamic_repulsive only"; return 0; }
        if (c->obs_repr < QS_OBS_CDIST_CDISTDOT_DIST_DISTDOT_ANGLE_ANGLEDOT || c->obs_repr > QS_OBS_CDIST_CDISTDOT_NDIST_DISTDOT_NSANGLE_ANGLEDOT) { why = "fork mode needs a fork obs_repr"; return 0; }
        if (c->neighbor_obs_type != QS_NEIGHBOR_NONE && (c->neighbor_obs_type < QS_NEIGHBOR_DIST_ANGLE || c->neighbor_obs_type > QS_NEIGHBOR_NDIST_NSANGLE)) { why = "fork mode needs a fork neighbor_obs_type"; return 0; }
        if (c->neighbor_obs_type == QS_NEIGHBOR_NDIST_NSANGLE && (c->fork.cam_num < 1 || !(c->fork.cam_focal_length > 0) || !(c->fork.cam_target_size > 0))) { why = "bad camera parameters"; return 0; }
        if (c->neighbor_visible_num < 0 || c->neighbor_visible_num > c->num_agents - 1) { why = "neighbor_visible_num out of range"; return 0; }
        if (c->use_obstacles || c->use_downwash || c->apply_collision_force) { why = "fork mode: obstacles / downwash / collision forces are off in the reference (quadrotor_multi_rewards.py:106-119,203) and not built"; return 0; }
        if (c->fork.substeps < 1 || c->fork.substeps > 64) { why = "fork.substeps out of [1, 64]"; return 0; }
        if (c->sim_steps < 1 || c->sim_steps > 16 || !(c->dt > 0) || c->svd_period < 1 || c->ep_len < 1) { why = "bad sim_steps / dt / svd_period / ep_len"; return 0; }
        if (!(c->mass > 0) || !(c->inertia[0] > 0) || !(c->inertia[1] > 0) || !(c->inertia[2] > 0)) { why = "bad mass / inertia"; return 0; }
        return 1;
    }
    if (c->env_mode != QS_MODE_UPSTREAM) { why = "unknown env_mode"; return 0; }
    if (c->scenario == QS_SCENARIO_DYNAMIC_REPULSIVE) { why = "dynamic_repulsive needs env_mode fork"; return 0; }
    if (c->api_version != QS_API_VERSION) { why = "api_version mismatch"; return 0; }
    if (c->num_envs < 1) { why = "num_envs < 1"; return 0; }
    if (c->num_agents < 1 || c->num_agents > QS_MAX_AGENTS) { why = "num_agents out of [1, 32]"; return 0; }
    if (c->neighbor_visible_num < 0 || c->neighbor_visible_num > c->num_agents - 1) { why = "neighbor_visible_num out of range"; return 0; }
    if (c->neighbor_obs_type != QS_NEIGHBOR_NONE && c->neighbor_obs_type != QS_NEIGHBOR_POS_VEL) { why = "unsupported neighbor_obs_type"; return 0; }
    if (c->obs_repr < 0 || c->obs_repr > QS_OBS_XYZ_VXYZ_R_OMEGA_WALL) { why = "unsupported obs_repr"; return 0; }
    if (c->sim_steps < 1 || c->sim_steps > 16 || !(c->dt > 0)) { why = "bad sim_steps / dt"; return 0; }
    if (c->svd_period < 1 || c->ep_len < 1) { why = "bad svd_period / ep_len"; return 0; }
    if (c->use_obstacles) {
        if (c->scenario == QS_SCENARIO_STATIC_SAME_GOAL) { why = "use_obstacles needs an obstacle scenario"; return 0; }
        int cells = c->obst_area_len * c->obst_area_wid;
        if (cells < 1 || cells > 64 || c->num_obstacles < 0 || c->num_obstacles > QS_MAX_OBSTACLES) { why = "obstacle grid must have <= 64 cells"; return 0; }
        if (cells - c->num_obstacles < c->num_agents) { why = "not enough free cells for the drones"; return 0; }
    } else {
        const int sc = c->scenario, K = c->num_agents;
        const bool formation = sc == QS_SCENARIO_STATIC_SAME_GOAL || (sc >= QS_SCENARIO_STATIC_DIFF_GOAL && sc <= QS_SCENARIO_RUN_AWAY);
        if (!formation) { why = "obstacle scenario without use_obstacles"; return 0; }
        // a sphere of n < 3 drones still has 3 goal rows (scenarios/utils.py:77-80): scenarios permuting stored rows need rows == drones
        if (sc == QS_SCENARIO_SWAP_GOALS && K < 3) { why = "swap_goals needs num_agents >= 3"; return 0; }
        if (sc == QS_SCENARIO_SWARM_VS_SWARM && K < 2) { why = "swarm_vs_swarm needs num_agents >= 2"; return 0; }
        if (sc == QS_SCENARIO_RUN_AWAY && K < 2) { why = "run_away needs num_agents >= 2"; return 0; }
        if (sc == QS_SCENARIO_MIX && K == 2) { why = "mix needs num_agents == 1 or >= 3"; return 0; }
    }
    if (!(c->mass > 0) || !(c->inertia[0] > 0) || !(c->inertia[1] > 0) || !(c->inertia[2] > 0)) { why = "bad mass / inertia"; return 0; }
    return 1;
}

static const KgLaunchers &launchers(int KG)
{
    switch (KG) {
        case 1: return launchers_kg1();
        case 2: return launchers_kg2();
        case 4: return launchers_kg4();
        case 8: return launchers_kg8();
        case 16: return launchers_kg16();
        default: return launchers_kg32();
    }
}

static void free_host_buffers(qs_env *e)
{
    if (e->h_act) cudaFreeHost(e->h_act);
    if (e->h_obs) cudaFreeHost(e->h_obs);
    if (e->h_rew) cudaFreeHost(e->h_rew);
    if (e->h_done) cudaFreeHost(e->h_done);
    if (e->d_act) cudaFree(e->d_act);
    if (e->d_obs) cudaFree(e->d_obs);
    if (e->d_rew) cudaFree(e->d_rew);
    if (e->d_done) cudaFree(e->d_done);
    e->h_act = e->h_obs = e->h_rew = nullptr; e->h_done = nullptr;
    e->d_act = e->d_obs = e->d_rew = nullptr; e->d_done = nullptr;
    e->host_ready = false;
}

// staging buffers of the *_host entry points, allocated on first use (all or nothing)
static int ensure_host_buffers(qs_env *e)
{
    if (e->host_ready) return QS_OK;
    const size_t nd = (size_t)e->cfg.num_envs * e->cfg.num_agents, D = (size_t)e->dc.D;
    cudaError_t r = cudaSuccess;
    if (r == cudaSuccess) r = cudaMallocHost(&e->h_act, nd * e->A * sizeof(float));
    if (r == cudaSuccess) r = cudaMallocHost(&e->h_obs, nd * D * sizeof(float));
    if (r == cudaSuccess) r = cudaMallocHost(&e->h_rew, nd * sizeof(float));
    if (r == cudaSuccess) r = cudaMallocHost(&e->h_done, nd);
    if (r == cudaSuccess) r = cudaMalloc(&e->d_act, nd * e->A * sizeof(float));
    if (r == cudaSuccess) r = cudaMalloc(&e->d_obs, nd * D * sizeof(float));
    if (r == cudaSuccess) r = cudaMalloc(&e->d_rew, nd * sizeof(float));
    if (r == cudaSuccess) r = cudaMalloc(&e->d_done, nd);
    if (r != cudaSuccess) {
        free_host_buffers(e);
        return fail(e, QS_ERR_CUDA, std::string("host staging buffers: ") + cudaGetErrorString(r));
    }
    e->host_ready = true;
    return QS_OK;
}

// the qs_config field a QS_PARAM_* key sets (nullptr for an unknown key)
static double *param_field(qs_config &c, int key)
{
    switch (key) {
        case QS_PARAM_REW_POS: return &c.rew_pos;
        case QS_PARAM_REW_EFFORT: return &c.rew_effort;
        case QS_PARAM_REW_CRASH: return &c.rew_crash;
        case QS_PARAM_REW_ORIENT: return &c.rew_orient;
        case QS_PARAM_REW_SPIN: return &c.rew_spin;
        case QS_PARAM_REW_QUADCOL_BIN: return &c.rew_quadcol_bin;
        case QS_PARAM_REW_QUADCOL_BIN_SMOOTH_MAX: return &c.rew_quadcol_bin_smooth_max;
        case QS_PARAM_REW_QUADCOL_BIN_OBST: return &c.rew_quadcol_bin_obst;
        case QS_PARAM_CAPTURE_RADIUS: return &c.fork.capture_radius;
        default: return nullptr;
    }
}

// ---- snapshots (include/quadsim.h) -------------------------------------------------------------------------------------------
// Every qs_config field except the reserved words, in declaration order: qs_restore compares field by field (padding bytes carry
// no meaning) so that its message can name the first field that differs.  Arrays compare as a whole.
#define QS_CONFIG_FIELDS(X)                                                                                                      \
    X(api_version) X(num_envs) X(num_agents) X(scenario) X(obs_repr) X(neighbor_obs_type) X(neighbor_visible_num)             \
    X(use_obstacles) X(use_downwash) X(apply_collision_force) X(sense_noise) X(ep_len) X(sim_steps) X(svd_period)               \
    X(obst_area_len) X(obst_area_wid) X(num_obstacles) X(env_mode) X(cube_dim) X(seed) X(env_id_offset) X(dt) X(room_dims)     \
    X(gravity) X(mass) X(inertia) X(thrust_max) X(torque_max) X(prop_cross) X(prop_ccw) X(arm) X(motor_tau_up)                 \
    X(motor_tau_down) X(motor_linearity) X(vel_damp) X(damp_omega_quadratic) X(omega_max) X(floor_mu) X(ou_theta) X(ou_sigma) \
    X(sense_pos_std) X(sense_vel_std) X(sense_gyro_std) X(rew_pos) X(rew_effort) X(rew_crash) X(rew_orient) X(rew_spin)       \
    X(rew_quadcol_bin) X(rew_quadcol_bin_smooth_max) X(rew_quadcol_bin_obst) X(collision_hitbox_radius)                        \
    X(collision_falloff_radius) X(spawn_box) X(spawn_min_z) X(obst_size) X(sdf_resolution) X(approach_goal_metric)             \
    X(fork.substeps) X(fork.capture_radius) X(fork.rew_existence) X(fork.rew_captor) X(fork.rew_helper)                        \
    X(fork.max_angular_rate) X(fork.chaser_speed) X(fork.evader_v_max) X(fork.evader_dt) X(fork.evader_arena)                   \
    X(fork.spawn_ring) X(fork.evader_r_min) X(fork.evader_r_span) X(fork.pid) X(fork.rate_out_scale) X(fork.mixer)             \
    X(fork.ctrl_mass) X(fork.ctrl_g) X(fork.ctrl_kf) X(fork.ctrl_min_rpm) X(fork.ctrl_max_rpm) X(fork.cam_focal_length)       \
    X(fork.cam_target_size) X(fork.cam_pixel_noise) X(fork.cam_fov_deg) X(fork.cam_resolution) X(fork.cam_num)

#define QS_FIELD_BYTES(f) + sizeof(((const qs_config *)nullptr)->f)
static_assert(0 QS_CONFIG_FIELDS(QS_FIELD_BYTES) + 3 * sizeof(int32_t) == sizeof(qs_config),
              "QS_CONFIG_FIELDS must list every qs_config field but reserved0, fork.reserved and fork.reserved2");
#undef QS_FIELD_BYTES

static const char *first_config_difference(const qs_config &a, const qs_config &b)
{
#define QS_CMP_FIELD(f) if (memcmp(&a.f, &b.f, sizeof(a.f)) != 0) return #f;
    QS_CONFIG_FIELDS(QS_CMP_FIELD)
#undef QS_CMP_FIELD
    return nullptr;
}

// the formation scenarios keep a per-env scenario row (DevPtrs::scen); static_same_goal, the obstacle scenarios and fork mode do not
static bool has_scenario_rows(const qs_config &c)
{
    return !c.use_obstacles && c.env_mode == QS_MODE_UPSTREAM && c.scenario != QS_SCENARIO_STATIC_SAME_GOAL;
}

// Sections of a snapshot, in blob order.  Sizes follow from N, K and the mode alone (never from the slab's alignment or the launch
// shape); a section the mode does not have is 0 bytes.
enum { SEC_PLANES = 0, SEC_TICK = SEC_PLANES + PL_COUNT, SEC_SVD, SEC_ECNT, SEC_OBST, SEC_SCEN, SEC_EP_REC, SEC_EP_AGENT, SEC_STATS,
       SEC_FPLANES, SEC_EVADER = SEC_FPLANES + FP_COUNT, SEC_FFLAGS, SEC_COUNT };

// Every section but the stats is env-major: env e's part is the `row` bytes at e * row (for the per-drone sections the rows of its
// K drones; the episode counters are [N, EC_COUNT], indexed env * EC_COUNT + k), so the part of an env range is one contiguous slice.
// The stats are one qs_stats for the whole handle (row 0).
struct SnapSection { void *dev; size_t bytes, row; };

// the section table of a snapshot of a handle created with `c`, device pointers unset
static void snapshot_sections(const qs_config &c, SnapSection s[SEC_COUNT])
{
    const size_t N = (size_t)c.num_envs, K = (size_t)c.num_agents;
    auto env_major = [&](int i, size_t row) { s[i] = { nullptr, N * row, row }; };
    for (int i = 0; i < SEC_COUNT; ++i) s[i] = { nullptr, 0, 0 };
    for (int p = 0; p < PL_COUNT; ++p) env_major(SEC_PLANES + p, K * sizeof(float4));
    env_major(SEC_TICK, sizeof(int));
    env_major(SEC_SVD, sizeof(int));
    env_major(SEC_ECNT, EC_COUNT * sizeof(int));
    if (c.use_obstacles) env_major(SEC_OBST, QS_MAX_OBSTACLES * sizeof(float2));
    if (has_scenario_rows(c)) env_major(SEC_SCEN, QS_SC_COUNT * sizeof(float));
    env_major(SEC_EP_REC, QS_ER_COUNT * sizeof(int));
    env_major(SEC_EP_AGENT, K * sizeof(float4));
    s[SEC_STATS] = { nullptr, sizeof(qs_stats), 0 };
    if (c.env_mode == QS_MODE_FORK) {
        for (int p = 0; p < FP_COUNT; ++p) env_major(SEC_FPLANES + p, K * sizeof(float4));
        env_major(SEC_EVADER, sizeof(float2));
        env_major(SEC_FFLAGS, sizeof(int));
    }
}

// the section table of the handle, with its device pointers
static void snapshot_sections(const qs_env *e, SnapSection s[SEC_COUNT])
{
    snapshot_sections(e->cfg, s);
    void *dev[SEC_COUNT] = {};
    for (int p = 0; p < PL_COUNT; ++p) dev[SEC_PLANES + p] = e->dp.plane[p];
    dev[SEC_TICK] = e->dp.tick; dev[SEC_SVD] = e->dp.svd_ctr; dev[SEC_ECNT] = e->dp.ecnt; dev[SEC_OBST] = e->dp.obst_xy;
    dev[SEC_SCEN] = e->dp.scen; dev[SEC_EP_REC] = e->dp.ep_rec; dev[SEC_EP_AGENT] = e->dp.ep_agent; dev[SEC_STATS] = e->dp.stats;
    for (int p = 0; p < FP_COUNT; ++p) dev[SEC_FPLANES + p] = e->fp.plane[p];
    dev[SEC_EVADER] = e->fp.evader; dev[SEC_FFLAGS] = e->fp.flags;
    for (int i = 0; i < SEC_COUNT; ++i) if (s[i].bytes) s[i].dev = dev[i];
}

static std::string section_name(int i)
{
    static const char *const names[] = { "tick", "svd_ctr", "episode counters", "obst_xy", "scenario", "ep_rec", "ep_agent", "stats" };
    if (i < SEC_TICK) return "state plane " + std::to_string(i - SEC_PLANES);
    if (i < SEC_FPLANES) return names[i - SEC_TICK];
    if (i < SEC_EVADER) return "fork plane " + std::to_string(i - SEC_FPLANES);
    return i == SEC_EVADER ? "evader" : "fork flags";
}

static const uint32_t SNAP_MAGIC = 0x4E535351u;     // the bytes "QSSN"

struct SnapHeader {
    uint32_t magic, version;
    uint64_t config_size;
    qs_config cfg;
    uint32_t rng_step, sections;
    uint64_t section_bytes[SEC_COUNT];
};
static_assert(offsetof(SnapHeader, cfg) == 16, "include/quadsim.h documents the configuration at offset 16");
static_assert(sizeof(qs_config) % 8 == 0, "the snapshot header has no padding");

// Magic, version, length and sizeof(qs_config) of a blob; copies its header to *h.  On failure `why` names the check first.
static int read_header(const void *src_host, size_t bytes, SnapHeader *h, std::string &why)
{
    const char *src = (const char *)src_host;
    uint32_t magic = 0, version = 0;
    if (bytes >= 8) { memcpy(&magic, src, 4); memcpy(&version, src + 4, 4); }
    if (magic != SNAP_MAGIC) { why = "magic: not a simulator snapshot"; return QS_ERR_SHAPE; }
    if (version != QS_SNAPSHOT_VERSION) {
        why = "version: snapshot format " + std::to_string(version) + ", this library reads " + std::to_string(QS_SNAPSHOT_VERSION);
        return QS_ERR_SHAPE;
    }
    if (bytes < sizeof(SnapHeader)) { why = "bytes: " + std::to_string(bytes) + " is shorter than the header"; return QS_ERR_SHAPE; }
    memcpy(h, src, sizeof(*h));
    if (h->config_size != sizeof(qs_config)) {
        why = "config_size: the snapshot's qs_config has " + std::to_string(h->config_size) + " bytes, this library's " +
              std::to_string(sizeof(qs_config));
        return QS_ERR_SHAPE;
    }
    return QS_OK;
}

// The header's section table against the expected one; *total = the blob length it implies.
static int check_sections(const SnapHeader &h, const SnapSection sec[SEC_COUNT], size_t *total, std::string &why)
{
    if (h.sections != SEC_COUNT) { why = "sections: " + std::to_string(h.sections) + ", expected " + std::to_string((int)SEC_COUNT); return QS_ERR_SHAPE; }
    size_t need = sizeof(SnapHeader);
    for (int i = 0; i < SEC_COUNT; ++i) {
        if (h.section_bytes[i] != sec[i].bytes) {
            why = "section " + section_name(i) + ": " + std::to_string(h.section_bytes[i]) + " bytes, expected " + std::to_string(sec[i].bytes);
            return QS_ERR_SHAPE;
        }
        need += sec[i].bytes;
    }
    *total = need;
    return QS_OK;
}

#define QS_STATS_FIELDS(X)                                                                                                       \
    X(episodes) X(num_collisions) X(num_collisions_after_settle) X(num_collisions_final_5s) X(num_collisions_with_room)          \
    X(num_collisions_with_floor) X(num_collisions_with_wall) X(num_collisions_with_ceiling) X(num_collisions_obst_quad)         \
    X(num_collisions_obst_quad_after_settle) X(agents_success) X(agents_deadlock) X(agents_collided) X(nonfinite_resets)         \
    X(episodes_success) X(distance_to_goal_1s) X(distance_to_goal_3s) X(distance_to_goal_5s) X(reward_sum)

#define QS_FIELD_BYTES(f) + sizeof(((const qs_stats *)nullptr)->f)
static_assert(0 QS_STATS_FIELDS(QS_FIELD_BYTES) == sizeof(qs_stats), "QS_STATS_FIELDS must list every qs_stats field");
#undef QS_FIELD_BYTES

static void add_stats(qs_stats &a, const qs_stats &b)
{
#define QS_ADD_FIELD(f) a.f += b.f;
    QS_STATS_FIELDS(QS_ADD_FIELD)
#undef QS_ADD_FIELD
}

extern "C" {

size_t qs_config_size(void) { return sizeof(qs_config); }
size_t qs_stats_size(void) { return sizeof(qs_stats); }
int qs_api_version(void) { return QS_API_VERSION; }
const char *qs_last_error(const qs_env *env) { return env ? env->err.c_str() : g_create_err.c_str(); }

int qs_create(const qs_config *cfg, int device, qs_env **out)
{
    if (!cfg || !out) return fail(nullptr, QS_ERR_NULL, "qs_create: null argument");
    *out = nullptr;
    std::string why;
    if (!validate(cfg, why)) return fail(nullptr, QS_ERR_BAD_CONFIG, "qs_create: " + why);
    int ndev = 0;
    cudaError_t r = cudaGetDeviceCount(&ndev);
    if (r != cudaSuccess || ndev == 0) return fail(nullptr, QS_ERR_CUDA, std::string("qs_create: no CUDA device (") + cudaGetErrorString(r) + ")");
    if (device < 0 || device >= ndev) return fail(nullptr, QS_ERR_BAD_CONFIG, "qs_create: bad device index");
    DeviceGuard guard(device);

    qs_env *e = new qs_env();
    e->cfg = *cfg; e->device = device; e->launches = 0; e->host_ready = false; e->rng_step = 0;
    e->h_act = e->h_obs = e->h_rew = e->h_term = nullptr; e->h_done = e->h_succ = nullptr;
    e->d_act = e->d_obs = e->d_rew = e->d_term = nullptr; e->d_done = e->d_succ = nullptr;
    e->pipe_ready = false;
    fill_const(*cfg, e->dc);
    e->fork = cfg->env_mode == QS_MODE_FORK;
    e->A = e->fork ? 2 : 4;
    const bool scen_feat = has_scenario_rows(*cfg);
    e->feat = (cfg->use_obstacles ? 1 : 0) | ((cfg->use_downwash && cfg->num_agents > 1) ? 2 : 0) | (scen_feat ? 4 : 0);
    fill_fork(*cfg, e->fc);
    memset(&e->fp, 0, sizeof(e->fp));
    const int N = cfg->num_envs, K = cfg->num_agents;
    e->KG = pow2_at_least(K);
    const long long lanes = (long long)N * e->KG;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    // small batches: 64-thread blocks so that every SM gets work; large batches: 128
    e->block = (lanes < (long long)sms * 2 * 128) ? 64 : 128;
    if (const char *tb = getenv("QS_BLOCK")) { int v = atoi(tb); if ((v == 32 || v == 64 || v == 128 || v == 256) && v <= QS_STEP_MAXTHREADS) e->block = v; }   // tuning knob (the step kernels are compiled for <= QS_STEP_MAXTHREADS threads)
    if (e->block < e->KG) e->block = e->KG;
    e->grid = (int)((lanes + e->block - 1) / e->block);
    const int warps = e->block / 32 > 0 ? e->block / 32 : 1;
    const int rows_per_warp = (32 / e->KG) * K;
    // exchange buffers + observation tiles (+ the staged obstacle centres of the upstream step kernel)
    const size_t tiles_floats = (((size_t)warps * 256 + (size_t)warps * rows_per_warp * e->dc.D) + 3) & ~(size_t)3;
    // staged per warp-tile behind the tiles: the obstacle centres, or (formation scenarios, never with obstacles) the scenario rows
    const size_t obst_floats = cfg->use_obstacles ? (size_t)warps * (32 / e->KG) * cfg->num_obstacles * 2
                                                  : (scen_feat ? (size_t)warps * (32 / e->KG) * QS_SC_COUNT : 0);
    // per-thread scratch slots of the step kernel: 4 float4 (the step's 16 pre-generated normals) + 3 ints (per-env scalars)
    const size_t park_floats = e->fork ? 0 : (size_t)19 * e->block;
    e->smem_bytes = (((tiles_floats + obst_floats + 3) & ~(size_t)3) + park_floats) * sizeof(float);
    if (e->smem_bytes > 200 * 1024) { delete e; return fail(nullptr, QS_ERR_BAD_CONFIG, "qs_create: observation tile does not fit in shared memory"); }

    // one slab: planes, per-env scalars, obstacle centres, stats
    const size_t nd = (size_t)N * K;
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    size_t off = 0, plane_off[PL_COUNT];
    for (int p = 0; p < PL_COUNT; ++p) { plane_off[p] = off; off += align(nd * sizeof(float4)); }
    size_t o_tick = off; off += align((size_t)N * sizeof(int));
    size_t o_svd = off; off += align((size_t)N * sizeof(int));
    size_t o_step = off; off += align((size_t)N * sizeof(uint32_t));
    size_t o_ecnt = off; off += align((size_t)N * EC_COUNT * sizeof(int));
    size_t o_obst = off; off += align((cfg->use_obstacles ? (size_t)N * QS_MAX_OBSTACLES : 1) * sizeof(float2));
    size_t o_scen = off; off += align((scen_feat ? (size_t)N * QS_SC_COUNT : 1) * sizeof(float));
    size_t o_erec = off; off += align((size_t)N * QS_ER_COUNT * sizeof(int));
    size_t o_eagent = off; off += align(nd * sizeof(float4));
    size_t o_stats = off; off += align(sizeof(qs_stats));
    const int n_wt = (N + (32 / e->KG) - 1) / (32 / e->KG);              // warp-tiles
    e->hot_cap = 128; e->hot_blocks = e->hot_cap / warps;
    size_t o_hot[3];
    for (int b3 = 0; b3 < 3; ++b3) { o_hot[b3] = off; off += align((size_t)(e->hot_cap + 64 + n_wt) * sizeof(int)); }
    e->hot_bytes = off - o_hot[0];
    size_t fplane_off[FP_COUNT] = {0}, o_evader = 0, o_fflags = 0;
    if (e->fork) {
        for (int p = 0; p < FP_COUNT; ++p) { fplane_off[p] = off; off += align(nd * sizeof(float4)); }
        o_evader = off; off += align((size_t)N * sizeof(float2));
        o_fflags = off; off += align((size_t)N * sizeof(int));
    }
    e->slab_bytes = off;
    r = cudaMalloc(&e->slab, off);
    if (r != cudaSuccess) { delete e; return fail(nullptr, QS_ERR_CUDA, std::string("qs_create: cudaMalloc: ") + cudaGetErrorString(r)); }
    r = cudaMemset(e->slab, 0, off);
    if (r != cudaSuccess) { cudaFree(e->slab); delete e; return fail(nullptr, QS_ERR_CUDA, std::string("qs_create: cudaMemset: ") + cudaGetErrorString(r)); }
    char *b = (char *)e->slab;
    for (int p = 0; p < PL_COUNT; ++p) e->dp.plane[p] = (float4 *)(b + plane_off[p]);
    e->dp.tick = (int *)(b + o_tick); e->dp.svd_ctr = (int *)(b + o_svd);
    (void)o_step;
    e->dp.ecnt = (int *)(b + o_ecnt); e->dp.obst_xy = (float2 *)(b + o_obst); e->dp.stats = (qs_stats *)(b + o_stats);
    e->dp.scen = scen_feat ? (float4 *)(b + o_scen) : nullptr;
    e->dp.ep_rec = (int *)(b + o_erec); e->dp.ep_agent = (float4 *)(b + o_eagent);
    for (int b3 = 0; b3 < 3; ++b3) {                                    // [count (64 ints: own cache line) | list | flags]
        e->hot_cnt[b3] = (int *)(b + o_hot[b3]); e->hot_list[b3] = e->hot_cnt[b3] + 64; e->hot_flag[b3] = e->hot_list[b3] + e->hot_cap;
    }
    e->hot_phase = 0;
    // reset-first scheduling pays where a reset is expensive (obstacle map generation, formation scenarios): cfg3 101.5 -> 98.8 us, mix
    // 108.7 -> 105.4 us; with the cheap static_same_goal reset it costs 1 % (cfg2 77.4 -> 78.0 us) and with 32-lane groups 5 % (cfg4
    // 109.4 -> 114.6 us: one env per warp, the listed tiles are 4x as many) -- profiles/README.md round 2.  Compiled out there (HOT_OK).
    e->hot = !e->fork && (e->feat & 5) != 0 && e->KG < 32;
    if (const char *hv = getenv("QS_HOT")) e->hot = e->hot && atoi(hv) != 0;   // tuning knob: 0 = plain block order
    if (e->fork) {
        for (int p = 0; p < FP_COUNT; ++p) e->fp.plane[p] = (float4 *)(b + fplane_off[p]);
        e->fp.evader = (float2 *)(b + o_evader); e->fp.flags = (int *)(b + o_fflags);
    }
    init_identity_kernel<<<(int)((nd + 127) / 128), 128>>>(e->dp, (int)nd);
    r = cudaDeviceSynchronize();
    if (r != cudaSuccess) { cudaFree(e->slab); delete e; return fail(nullptr, QS_ERR_CUDA, std::string("qs_create: state init: ") + cudaGetErrorString(r)); }
    launchers(e->KG).prepare(e->feat, e->smem_bytes, e->block, e->fork);
    r = cudaGetLastError();
    if (r != cudaSuccess) { cudaFree(e->slab); delete e; return fail(nullptr, QS_ERR_CUDA, std::string("qs_create: ") + cudaGetErrorString(r)); }
    *out = e;
    return QS_OK;
}

int qs_destroy(qs_env *e)
{
    if (!e) return QS_ERR_NULL;
    DeviceGuard guard(e->device);
    cudaFree(e->slab);
    free_host_buffers(e);
    if (e->h_term) cudaFreeHost(e->h_term);
    if (e->h_succ) cudaFreeHost(e->h_succ);
    if (e->d_term) cudaFree(e->d_term);
    if (e->d_succ) cudaFree(e->d_succ);
    if (e->pipe_ready) {
        for (int i = 0; i < 2; ++i) { cudaStreamDestroy(e->cs[i]); cudaEventDestroy(e->ev_out[i]); }
        cudaEventDestroy(e->ev_in);
    }
    delete e;
    return QS_OK;
}

int qs_num_envs(const qs_env *e) { return e ? e->cfg.num_envs : QS_ERR_NULL; }
int qs_num_agents(const qs_env *e) { return e ? e->cfg.num_agents : QS_ERR_NULL; }
int qs_obs_dim(const qs_env *e) { return e ? e->dc.D : QS_ERR_NULL; }
int qs_act_dim(const qs_env *e) { return e ? e->A : QS_ERR_NULL; }
int64_t qs_launch_count(const qs_env *e) { return e ? e->launches : 0; }

int qs_reset(qs_env *e, const uint8_t *env_mask, float *obs, void *stream)
{
    if (!e || !obs) return fail(e, QS_ERR_NULL, "qs_reset: null argument");
    DeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    const LaunchShape shape = { e->grid, e->block, e->smem_bytes };
    e->dc.rng_step = e->rng_step;
    if (e->fork) launchers(e->KG).fork_reset(shape, s, e->dc, e->fc, e->dp, e->fp, env_mask, obs);
    else launchers(e->KG).reset(e->feat, shape, s, e->dc, e->dp, env_mask, obs);
    e->launches += 1;
    e->rng_step += 1u;
    QS_CUDA(e, cudaGetLastError());
    return QS_OK;
}

// One step of envs [e0, e0 + n) of the handle: the same kernels on offset views of the state (environments are independent, and the
// RNG is keyed by the global env id, so a step done in chunks is bitwise the step done at once).  e0 must be a multiple of 32.
static void launch_step_range(qs_env *e, int e0, int n, cudaStream_t s, const float *actions, float *obs, float *rew, uint8_t *done,
                              float *terminal_obs, uint8_t *reset_success)
{
    const int K = e->cfg.num_agents;
    const size_t r0 = (size_t)e0 * K;
    DevConst c = e->dc;
    DevPtrs P = e->dp;
    c.N = n; c.env_id_offset += e0; c.rng_step = e->rng_step;
    for (int p = 0; p < PL_COUNT; ++p) P.plane[p] += r0;
    if (P.rew_info) P.rew_info += 2 * r0;
    P.tick += e0; P.svd_ctr += e0; P.ecnt += (size_t)e0 * EC_COUNT; P.ep_rec += (size_t)e0 * QS_ER_COUNT; P.ep_agent += r0;
    if (e->cfg.use_obstacles) P.obst_xy += (size_t)e0 * QS_MAX_OBSTACLES;
    if (P.scen) P.scen += (size_t)e0 * (QS_SC_COUNT / 4);
    const int grid = (int)(((long long)n * e->KG + e->block - 1) / e->block);
    const size_t D = (size_t)e->dc.D;
    actions += r0 * e->A; obs += r0 * D; rew += r0; done += r0;
    if (terminal_obs) terminal_obs += r0 * D;
    if (reset_success) reset_success += e0;
    if (e->fork) {
        ForkPtrs F = e->fp;
        for (int p = 0; p < FP_COUNT; ++p) F.plane[p] += r0;
        F.evader += e0; F.flags += e0;
        launchers(e->KG).fork_step({ grid, e->block, e->smem_bytes }, s, c, e->fc, P, F, (const float2 *)actions, obs, rew, done, terminal_obs,
                                   reset_success);
    } else {
        int g2 = grid;
        if (e->hot && e0 == 0 && n == e->cfg.num_envs) {                // full-range launches only: tile ids are relative to the launch
            const unsigned ph = e->hot_phase++;
            const int cur = ph % 3, nxt = (ph + 1) % 3, clr = (ph + 2) % 3;
            P.hot_list_cur = e->hot_list[cur]; P.hot_cnt_cur = e->hot_cnt[cur]; P.hot_flag_cur = e->hot_flag[cur];
            P.hot_list_next = e->hot_list[nxt]; P.hot_cnt_next = e->hot_cnt[nxt]; P.hot_flag_next = e->hot_flag[nxt];
            P.hot_cnt_clear = e->hot_cnt[clr];
            P.hot_cap = e->hot_cap; P.hot_blocks = e->hot_blocks;
            g2 += e->hot_blocks;
        }
        launchers(e->KG).step(e->feat, { g2, e->block, e->smem_bytes }, s, c, P, (const float4 *)actions, obs, rew, done, terminal_obs,
                              reset_success);
    }
    e->launches += 1;
}

int qs_step(qs_env *e, const float *actions, float *obs, float *rew, uint8_t *done, float *terminal_obs, uint8_t *reset_success,
            void *stream)
{
    if (!e || !actions || !obs || !rew || !done) return fail(e, QS_ERR_NULL, "qs_step: null argument");
    if (((size_t)actions & 15) != 0) return fail(e, QS_ERR_SHAPE, "qs_step: actions must be 16-byte aligned");
    DeviceGuard guard(e->device);
    launch_step_range(e, 0, e->cfg.num_envs, (cudaStream_t)stream, actions, obs, rew, done, terminal_obs, reset_success);
    e->rng_step += e->fork ? (uint32_t)e->cfg.fork.substeps : 1u;
    QS_CUDA(e, cudaGetLastError());
    return QS_OK;
}

// true if `p` is page-locked host memory the copy engines can reach directly (cudaHostAlloc / cudaHostRegister /
// torch pin_memory); pageable buffers go through the handle's pinned staging area instead.
static bool is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

int qs_reset_host(qs_env *e, float *obs_host, void *stream)
{
    if (!e || !obs_host) return fail(e, QS_ERR_NULL, "qs_reset_host: null argument");
    DeviceGuard guard(e->device);
    int rc = ensure_host_buffers(e);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t nd = (size_t)e->cfg.num_envs * e->cfg.num_agents, D = (size_t)e->dc.D;
    rc = qs_reset(e, nullptr, e->d_obs, stream);
    if (rc) return rc;
    const bool direct = is_pinned(obs_host);
    QS_CUDA(e, cudaMemcpyAsync(direct ? obs_host : e->h_obs, e->d_obs, nd * D * sizeof(float), cudaMemcpyDeviceToHost, s));
    QS_CUDA(e, cudaStreamSynchronize(s));
    if (!direct) memcpy(obs_host, e->h_obs, nd * D * sizeof(float));
    return QS_OK;
}

int qs_step_host(qs_env *e, const float *actions_host, float *obs_host, float *rew_host, uint8_t *done_host,
                 float *terminal_obs_host, uint8_t *reset_success_host, void *stream)
{
    if (!e || !actions_host || !obs_host || !rew_host || !done_host) return fail(e, QS_ERR_NULL, "qs_step_host: null argument");
    DeviceGuard guard(e->device);
    int rc = ensure_host_buffers(e);
    if (rc) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)e->cfg.num_envs, nd = N * e->cfg.num_agents, D = (size_t)e->dc.D, A = (size_t)e->A;
    if (terminal_obs_host && !(e->d_term && e->h_term)) {                // device + pinned pair: all or nothing
        cudaError_t r = e->d_term ? cudaSuccess : cudaMalloc(&e->d_term, nd * D * sizeof(float));
        if (r == cudaSuccess) r = cudaMemsetAsync(e->d_term, 0, nd * D * sizeof(float), s);
        if (r == cudaSuccess) r = cudaMallocHost(&e->h_term, nd * D * sizeof(float));
        if (r != cudaSuccess) {
            if (e->d_term) cudaFree(e->d_term);
            e->d_term = nullptr; e->h_term = nullptr;
            return fail(e, QS_ERR_CUDA, std::string("qs_step_host: terminal-observation buffers: ") + cudaGetErrorString(r));
        }
    }
    if (reset_success_host && !(e->d_succ && e->h_succ)) {
        cudaError_t r = e->d_succ ? cudaSuccess : cudaMalloc(&e->d_succ, N);
        if (r == cudaSuccess) r = cudaMemsetAsync(e->d_succ, 0, N, s);
        if (r == cudaSuccess) r = cudaMallocHost(&e->h_succ, N);
        if (r != cudaSuccess) {
            if (e->d_succ) cudaFree(e->d_succ);
            e->d_succ = nullptr; e->h_succ = nullptr;
            return fail(e, QS_ERR_CUDA, std::string("qs_step_host: reset-success buffers: ") + cudaGetErrorString(r));
        }
    }
    // page-locked caller buffers are DMA'd directly; pageable ones are staged through the handle's pinned buffers
    const bool pa = is_pinned(actions_host), po = is_pinned(obs_host), pr = is_pinned(rew_host), pd = is_pinned(done_host);
    const bool pt = terminal_obs_host && is_pinned(terminal_obs_host), ps = reset_success_host && is_pinned(reset_success_host);
    if (!pa) memcpy(e->h_act, actions_host, nd * A * sizeof(float));
    const float *src_act = pa ? actions_host : e->h_act;
    float *dst_obs = po ? obs_host : e->h_obs, *dst_rew = pr ? rew_host : e->h_rew;
    uint8_t *dst_done = pd ? done_host : e->h_done;
    // Large batches: the step is PCIe-bound (D2H of the observations), so the env range is cut into chunks that alternate between two
    // internal streams -- while chunk i's observations travel to the host, chunk i+1's actions arrive and its kernel runs.  Chunks are
    // >= 8192 envs (a kernel launch below that is latency-bound) and start at multiples of 32 envs (16-byte alignment of every view).
    int chunks = (int)(N / 8192);
    if (chunks > 8) chunks = 8;
    if (const char *pc = getenv("QS_HOST_CHUNKS")) chunks = atoi(pc);      // tuning knob / tests
    if (chunks < 1) chunks = 1;
    if (chunks > 1 && !e->pipe_ready) {
        cudaError_t r = cudaSuccess;
        for (int i = 0; i < 2 && r == cudaSuccess; ++i) { r = cudaStreamCreateWithFlags(&e->cs[i], cudaStreamNonBlocking); if (r == cudaSuccess) r = cudaEventCreateWithFlags(&e->ev_out[i], cudaEventDisableTiming); }
        if (r == cudaSuccess) r = cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming);
        if (r != cudaSuccess) return fail(e, QS_ERR_CUDA, std::string("qs_step_host: pipeline streams: ") + cudaGetErrorString(r));
        e->pipe_ready = true;
    }
    float *d_term = terminal_obs_host ? e->d_term : nullptr;
    uint8_t *d_succ = reset_success_host ? e->d_succ : nullptr;
    if (chunks == 1) {
        QS_CUDA(e, cudaMemcpyAsync(e->d_act, src_act, nd * A * sizeof(float), cudaMemcpyHostToDevice, s));
        launch_step_range(e, 0, (int)N, s, e->d_act, e->d_obs, e->d_rew, e->d_done, d_term, d_succ);
        QS_CUDA(e, cudaMemcpyAsync(dst_rew, e->d_rew, nd * sizeof(float), cudaMemcpyDeviceToHost, s));
        QS_CUDA(e, cudaMemcpyAsync(dst_done, e->d_done, nd, cudaMemcpyDeviceToHost, s));
        QS_CUDA(e, cudaMemcpyAsync(dst_obs, e->d_obs, nd * D * sizeof(float), cudaMemcpyDeviceToHost, s));
    } else {
        const size_t K = (size_t)e->cfg.num_agents;
        QS_CUDA(e, cudaEventRecord(e->ev_in, s));                       // work queued on the caller's stream comes first
        QS_CUDA(e, cudaStreamWaitEvent(e->cs[0], e->ev_in, 0));
        QS_CUDA(e, cudaStreamWaitEvent(e->cs[1], e->ev_in, 0));
        const size_t per = (((N + chunks - 1) / chunks) + 31) & ~(size_t)31;
        int i = 0;
        for (size_t e0 = 0; e0 < N; e0 += per, ++i) {
            const size_t n = (e0 + per <= N) ? per : N - e0, r0 = e0 * K, rows = n * K;
            cudaStream_t t = e->cs[i & 1];
            QS_CUDA(e, cudaMemcpyAsync(e->d_act + r0 * A, src_act + r0 * A, rows * A * sizeof(float), cudaMemcpyHostToDevice, t));
            launch_step_range(e, (int)e0, (int)n, t, e->d_act, e->d_obs, e->d_rew, e->d_done, d_term, d_succ);
            QS_CUDA(e, cudaMemcpyAsync(dst_obs + r0 * D, e->d_obs + r0 * D, rows * D * sizeof(float), cudaMemcpyDeviceToHost, t));
            QS_CUDA(e, cudaMemcpyAsync(dst_rew + r0, e->d_rew + r0, rows * sizeof(float), cudaMemcpyDeviceToHost, t));
            QS_CUDA(e, cudaMemcpyAsync(dst_done + r0, e->d_done + r0, rows, cudaMemcpyDeviceToHost, t));
        }
        for (int k = 0; k < 2; ++k) { QS_CUDA(e, cudaEventRecord(e->ev_out[k], e->cs[k])); QS_CUDA(e, cudaStreamWaitEvent(s, e->ev_out[k], 0)); }
    }
    e->rng_step += e->fork ? (uint32_t)e->cfg.fork.substeps : 1u;        // every chunk of this step drew from the same counter
    QS_CUDA(e, cudaGetLastError());
    if (reset_success_host) QS_CUDA(e, cudaMemcpyAsync(ps ? reset_success_host : e->h_succ, e->d_succ, N, cudaMemcpyDeviceToHost, s));
    QS_CUDA(e, cudaStreamSynchronize(s));
    if (!po) memcpy(obs_host, e->h_obs, nd * D * sizeof(float));
    if (!pr) memcpy(rew_host, e->h_rew, nd * sizeof(float));
    if (!pd) memcpy(done_host, e->h_done, nd);
    if (reset_success_host && !ps) memcpy(reset_success_host, e->h_succ, N);
    if (terminal_obs_host) {
        // terminal observations are only needed for envs that finished (rare): copy them after looking at `done`
        const uint8_t *dn = pd ? done_host : e->h_done;
        bool any = false;
        for (size_t i = 0; i < nd && !any; i += (size_t)e->cfg.num_agents) any = dn[i] != 0;
        if (any) {
            QS_CUDA(e, cudaMemcpyAsync(pt ? terminal_obs_host : e->h_term, e->d_term, nd * D * sizeof(float), cudaMemcpyDeviceToHost, s));
            QS_CUDA(e, cudaStreamSynchronize(s));
            if (!pt) memcpy(terminal_obs_host, e->h_term, nd * D * sizeof(float));
        }
    }
    return QS_OK;
}

static int state_io(qs_env *e, const qs_state_view *view, void *stream, int set)
{
    if (!e || !view) return fail(e, QS_ERR_NULL, "qs_get/set_state: null argument");
    DeviceGuard guard(e->device);
    StateView v;
    v.pos = view->pos; v.vel = view->vel; v.rot = view->rot; v.omega = view->omega; v.rot_damp = view->rot_damp;
    v.cmds_damp = view->cmds_damp; v.ou = view->ou; v.goal = view->goal; v.flags = view->flags; v.col_mask = view->col_mask;
    v.tick = view->tick; v.svd_ctr = view->svd_ctr; v.step_ctr = view->step_ctr;
    v.obst_xy = e->cfg.use_obstacles ? view->obst_xy : nullptr;      // obstacle storage exists only with use_obstacles
    v.scenario = e->dp.scen ? view->scenario : nullptr;
    v.pid = e->fork ? view->pid : nullptr; v.heading = e->fork ? view->heading : nullptr; v.evader = e->fork ? view->evader : nullptr;
    const size_t nd = (size_t)e->cfg.num_envs * e->cfg.num_agents;
    if (set && view->step_ctr) {                                        // the handle's RNG launch counter = entry 0 of the (device) array
        uint32_t h = 0;
        QS_CUDA(e, cudaMemcpyAsync(&h, view->step_ctr, sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        QS_CUDA(e, cudaStreamSynchronize((cudaStream_t)stream));
        e->rng_step = h;
    }
    e->dc.rng_step = e->rng_step;
    state_io_kernel<<<(int)((nd + 127) / 128), 128, 0, (cudaStream_t)stream>>>(e->dc, e->dp, e->fp, v, set);
    e->launches += 1;
    QS_CUDA(e, cudaGetLastError());
    return QS_OK;
}
int qs_get_state(qs_env *e, const qs_state_view *view, void *stream) { return state_io(e, view, stream, 0); }
int qs_set_state(qs_env *e, const qs_state_view *view, void *stream) { return state_io(e, view, stream, 1); }

int qs_set_param(qs_env *e, int key, double value)
{
    if (!e) return QS_ERR_NULL;
    double *field = param_field(e->cfg, key);
    if (!field) return fail(e, QS_ERR_BAD_CONFIG, "qs_set_param: unknown key");
    *field = value;
    fill_const(e->cfg, e->dc);
    fill_fork(e->cfg, e->fc);
    return QS_OK;
}

int qs_set_reward_info(qs_env *e, float *rew_info)
{
    if (!e) return QS_ERR_NULL;
    if (((size_t)rew_info & 15) != 0) return fail(e, QS_ERR_SHAPE, "qs_set_reward_info: buffer must be 16-byte aligned");
    e->dp.rew_info = reinterpret_cast<float4 *>(rew_info);
    return QS_OK;
}

int qs_episode_stats(qs_env *e, qs_stats *out, int reset, void *stream)
{
    if (!e || !out) return fail(e, QS_ERR_NULL, "qs_episode_stats: null argument");
    DeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    QS_CUDA(e, cudaMemcpyAsync(out, e->dp.stats, sizeof(qs_stats), cudaMemcpyDeviceToHost, s));
    if (reset) QS_CUDA(e, cudaMemsetAsync(e->dp.stats, 0, sizeof(qs_stats), s));
    QS_CUDA(e, cudaStreamSynchronize(s));
    return QS_OK;
}

int qs_episode_records(qs_env *e, int32_t *env_rec, float *agent_rec, void *stream)
{
    if (!e) return fail(e, QS_ERR_NULL, "qs_episode_records: null handle");
    DeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)e->cfg.num_envs, nd = N * e->cfg.num_agents;
    if (env_rec) QS_CUDA(e, cudaMemcpyAsync(env_rec, e->dp.ep_rec, N * QS_ER_COUNT * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    if (agent_rec) QS_CUDA(e, cudaMemcpyAsync(agent_rec, e->dp.ep_agent, nd * sizeof(float4), cudaMemcpyDeviceToDevice, s));
    return QS_OK;
}

int qs_episode_records_host(qs_env *e, int32_t *env_rec_host, float *agent_rec_host, void *stream)
{
    if (!e) return fail(e, QS_ERR_NULL, "qs_episode_records_host: null handle");
    DeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t N = (size_t)e->cfg.num_envs, nd = N * e->cfg.num_agents;
    if (env_rec_host) QS_CUDA(e, cudaMemcpyAsync(env_rec_host, e->dp.ep_rec, N * QS_ER_COUNT * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (agent_rec_host) QS_CUDA(e, cudaMemcpyAsync(agent_rec_host, e->dp.ep_agent, nd * sizeof(float4), cudaMemcpyDeviceToHost, s));
    QS_CUDA(e, cudaStreamSynchronize(s));
    return QS_OK;
}

size_t qs_snapshot_size(const qs_env *e)
{
    if (!e) return 0;
    SnapSection sec[SEC_COUNT];
    snapshot_sections(e, sec);
    size_t n = sizeof(SnapHeader);
    for (int i = 0; i < SEC_COUNT; ++i) n += sec[i].bytes;
    return n;
}

int qs_snapshot(qs_env *e, void *dst_host, size_t bytes, void *stream)
{
    if (!e || !dst_host) return fail(e, QS_ERR_NULL, "qs_snapshot: null argument");
    const size_t need = qs_snapshot_size(e);
    if (bytes < need)
        return fail(e, QS_ERR_SHAPE, "qs_snapshot: the buffer has " + std::to_string(bytes) + " bytes, the snapshot " + std::to_string(need));
    DeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    SnapSection sec[SEC_COUNT];
    snapshot_sections(e, sec);
    SnapHeader h;
    memset(&h, 0, sizeof(h));
    h.magic = SNAP_MAGIC; h.version = QS_SNAPSHOT_VERSION; h.config_size = sizeof(qs_config);
    h.cfg = e->cfg; h.rng_step = e->rng_step; h.sections = SEC_COUNT;
    for (int i = 0; i < SEC_COUNT; ++i) h.section_bytes[i] = sec[i].bytes;
    memcpy(dst_host, &h, sizeof(h));
    char *p = (char *)dst_host + sizeof(h);
    for (int i = 0; i < SEC_COUNT; ++i) {
        if (!sec[i].bytes) continue;
        QS_CUDA(e, cudaMemcpyAsync(p, sec[i].dev, sec[i].bytes, cudaMemcpyDeviceToHost, s));
        p += sec[i].bytes;
    }
    QS_CUDA(e, cudaStreamSynchronize(s));
    return QS_OK;
}

int qs_restore(qs_env *e, const void *src_host, size_t bytes, void *stream)
{
    if (!e || !src_host) return fail(e, QS_ERR_NULL, "qs_restore: null argument");
    // everything is checked before the first copy: a rejected snapshot leaves the handle as it was
    const char *src = (const char *)src_host;
    SnapHeader h;
    std::string why;
    if (int rc = read_header(src, bytes, &h, why)) return fail(e, rc, "qs_restore: " + why);
    qs_config want = e->cfg;                                            // the qs_set_param values come from the snapshot
    for (int k = 0; k < QS_PARAM_COUNT; ++k) *param_field(want, k) = *param_field(h.cfg, k);
    if (const char *f = first_config_difference(want, h.cfg))
        return fail(e, QS_ERR_BAD_CONFIG, std::string("qs_restore: ") + f + ": the snapshot's configuration differs from the handle's");
    SnapSection sec[SEC_COUNT];
    snapshot_sections(e, sec);
    size_t need = 0;
    if (int rc = check_sections(h, sec, &need, why)) return fail(e, rc, "qs_restore: " + why);
    if (bytes != need)
        return fail(e, QS_ERR_SHAPE, "qs_restore: bytes: the blob has " + std::to_string(bytes) + ", a snapshot of this handle " + std::to_string(need));
    DeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    const char *p = src + sizeof(SnapHeader);
    for (int i = 0; i < SEC_COUNT; ++i) {
        if (!sec[i].bytes) continue;
        QS_CUDA(e, cudaMemcpyAsync(sec[i].dev, p, sec[i].bytes, cudaMemcpyHostToDevice, s));
        p += sec[i].bytes;
    }
    // reset-first lists as qs_create leaves them: zero counts and flags make every warp-tile a regular block's (the hot blocks find
    // no listed tile and return), and the step results do not depend on the schedule
    QS_CUDA(e, cudaMemsetAsync(e->hot_cnt[0], 0, e->hot_bytes, s));
    QS_CUDA(e, cudaStreamSynchronize(s));
    e->cfg = want;
    e->rng_step = h.rng_step;
    e->hot_phase = 0;
    fill_const(e->cfg, e->dc);
    fill_fork(e->cfg, e->fc);
    return QS_OK;
}

int qs_restore_shards(qs_env *e, const void *const *blobs, const size_t *bytes, int count, void *stream)
{
    if (!e) return QS_ERR_NULL;
    if (count < 1) return fail(e, QS_ERR_SHAPE, "qs_restore_shards: count: " + std::to_string(count) + ", at least one snapshot is needed");
    if (!blobs || !bytes) return fail(e, QS_ERR_NULL, "qs_restore_shards: null argument");
    // every blob is checked before the first copy: a rejected call leaves the handle as it was
    const int64_t lo = e->cfg.env_id_offset, hi = lo + e->cfg.num_envs;
    std::vector<SnapHeader> hs((size_t)count);
    for (int i = 0; i < count; ++i) {
        const std::string at = "qs_restore_shards: blob " + std::to_string(i) + ": ";
        if (!blobs[i]) return fail(e, QS_ERR_NULL, at + "null pointer");
        SnapHeader &h = hs[i];
        std::string why;
        if (int rc = read_header(blobs[i], bytes[i], &h, why)) return fail(e, rc, at + why);
        if (h.cfg.num_envs < 1) return fail(e, QS_ERR_SHAPE, at + "num_envs: " + std::to_string(h.cfg.num_envs));
        // the env range may differ from the handle's; the qs_set_param values come from the snapshots and must agree among them
        qs_config want = e->cfg;
        want.num_envs = h.cfg.num_envs; want.env_id_offset = h.cfg.env_id_offset;
        for (int k = 0; k < QS_PARAM_COUNT; ++k) *param_field(want, k) = *param_field(h.cfg, k);
        if (const char *f = first_config_difference(want, h.cfg))
            return fail(e, QS_ERR_BAD_CONFIG, at + f + ": the snapshot's configuration differs from the handle's");
        if (i > 0) {
            qs_config first = hs[0].cfg;
            first.num_envs = h.cfg.num_envs; first.env_id_offset = h.cfg.env_id_offset;
            if (const char *f = first_config_difference(first, h.cfg))
                return fail(e, QS_ERR_BAD_CONFIG, at + f + ": differs from blob 0's (qs_set_param values must agree among the shards)");
            if (h.rng_step != hs[0].rng_step)
                return fail(e, QS_ERR_BAD_CONFIG, at + "rng_step: " + std::to_string(h.rng_step) + ", blob 0's " + std::to_string(hs[0].rng_step) +
                                                  " (the shards of one run stand at the same step)");
        }
        SnapSection sec[SEC_COUNT];
        snapshot_sections(h.cfg, sec);
        size_t need = 0;
        if (int rc = check_sections(h, sec, &need, why)) return fail(e, rc, at + why);
        if (bytes[i] != need)
            return fail(e, QS_ERR_SHAPE, at + "bytes: the blob has " + std::to_string(bytes[i]) + ", its header describes " + std::to_string(need));
    }
    // env ranges: disjoint, and together covering [lo, hi); blobs outside it are ignored
    auto range = [&](int i) { return std::make_pair((int64_t)hs[i].cfg.env_id_offset, (int64_t)hs[i].cfg.env_id_offset + hs[i].cfg.num_envs); };
    auto span = [](std::pair<int64_t, int64_t> r) { return "[" + std::to_string(r.first) + ", " + std::to_string(r.second) + ")"; };
    std::vector<int> order((size_t)count);
    for (int i = 0; i < count; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return range(a).first < range(b).first; });
    for (int j = 1; j < count; ++j) {
        const int a = order[j - 1], b = order[j];
        if (range(b).first < range(a).second)
            return fail(e, QS_ERR_SHAPE, "qs_restore_shards: env range: blob " + std::to_string(b) + " " + span(range(b)) + " overlaps blob " +
                                         std::to_string(a) + " " + span(range(a)));
    }
    int64_t covered = lo;                                               // [lo, covered) is in some blob
    for (int j = 0; j < count && covered < hi; ++j) {
        const auto r = range(order[j]);
        if (r.second <= covered) continue;
        if (r.first > covered) break;
        covered = r.second;
    }
    if (covered < hi)
        return fail(e, QS_ERR_SHAPE, "qs_restore_shards: env range: gap: env " + std::to_string(covered) + " of the handle's " +
                                     span({ lo, hi }) + " is in no snapshot");

    DeviceGuard guard(e->device);
    cudaStream_t s = (cudaStream_t)stream;
    SnapSection dst[SEC_COUNT];
    snapshot_sections(e, dst);
    // qs_stats: the sum of the blobs whose first env is in this handle's range, so that over all handles every blob counts once
    qs_stats stats;
    memset(&stats, 0, sizeof(stats));
    bool have_stats = false;
    for (int i = 0; i < count; ++i) {
        const auto r = range(i);
        const int64_t a = std::max(lo, r.first), b = std::min(hi, r.second);     // envs of blob i that this handle holds
        SnapSection sec[SEC_COUNT];
        snapshot_sections(hs[i].cfg, sec);
        const char *p = (const char *)blobs[i] + sizeof(SnapHeader);
        for (int k = 0; k < SEC_COUNT; ++k) {
            if (!sec[k].bytes) continue;
            if (sec[k].row == 0) {                                      // SEC_STATS
                if (r.first >= lo && r.first < hi) {
                    qs_stats x;
                    memcpy(&x, p, sizeof(x));
                    if (have_stats) add_stats(stats, x); else stats = x;
                    have_stats = true;
                }
            } else if (a < b) {
                const size_t row = sec[k].row;
                QS_CUDA(e, cudaMemcpyAsync((char *)dst[k].dev + (size_t)(a - lo) * row, p + (size_t)(a - r.first) * row, (size_t)(b - a) * row,
                                           cudaMemcpyHostToDevice, s));
            }
            p += sec[k].bytes;
        }
    }
    QS_CUDA(e, cudaMemcpyAsync(e->dp.stats, &stats, sizeof(stats), cudaMemcpyHostToDevice, s));
    QS_CUDA(e, cudaMemsetAsync(e->hot_cnt[0], 0, e->hot_bytes, s));    // reset-first lists as qs_restore leaves them
    QS_CUDA(e, cudaStreamSynchronize(s));
    for (int k = 0; k < QS_PARAM_COUNT; ++k) *param_field(e->cfg, k) = *param_field(hs[0].cfg, k);
    e->rng_step = hs[0].rng_step;
    e->hot_phase = 0;
    fill_const(e->cfg, e->dc);
    fill_fork(e->cfg, e->fc);
    return QS_OK;
}

// test hook: raw generator output (pins the RNG contract against the oracle); not part of the reference surface
int qs_philox_probe(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t *out4, float *fout6)
{
    uint32_t *d = nullptr; float *f = nullptr;
    if (cudaMalloc(&d, 16) != cudaSuccess || cudaMalloc(&f, 24) != cudaSuccess) return QS_ERR_CUDA;
    philox_probe_kernel<<<1, 1>>>(c0, c1, c2, c3, k0, k1, d, f);
    cudaError_t r = cudaMemcpy(out4, d, 16, cudaMemcpyDeviceToHost);
    if (r == cudaSuccess) r = cudaMemcpy(fout6, f, 24, cudaMemcpyDeviceToHost);
    cudaFree(d); cudaFree(f);
    return r == cudaSuccess ? QS_OK : QS_ERR_CUDA;
}

}  // extern "C"
