/*
 * quadsim.h -- C-ABI of the B200-native batched quadrotor-swarm simulator.
 *
 * This is the drop-in boundary for the reference's per-control-step hot path.  The reference
 * (priban42/quad-swarm-rl-stable-baselines3) is pure Python, so "the FFI a maintainer would bind"
 * is a ctypes binding (shown in INTEGRATION.md).  Every entry point below names the reference
 * interface it replaces (paths relative to the reference root):
 *
 *   qs_create / qs_destroy   QuadrotorEnvMulti.__init__            gym_art/quadrotor_multi/quadrotor_multi.py:27-228
 *                            SubprocVecEnvCustom.__init__/close    swarm_rl/env_wrappers/subproc_vec_env_custom.py:112-139,190-201
 *   qs_reset                 QuadrotorEnvMulti.reset               gym_art/quadrotor_multi/quadrotor_multi.py:440-519
 *                            SubprocVecEnvCustom.reset             swarm_rl/env_wrappers/subproc_vec_env_custom.py:155-164
 *   qs_step                  QuadrotorEnvMulti.step                gym_art/quadrotor_multi/quadrotor_multi.py:521-842
 *                            SubprocVecEnvCustom.step_async/_wait  swarm_rl/env_wrappers/subproc_vec_env_custom.py:141-153
 *                            (+ the worker auto-reset,             swarm_rl/env_wrappers/subproc_vec_env_custom.py:35-52)
 *   qs_step_host / qs_reset_host   the same two calls with HOST buffers (what SB3's numpy rollout loop sees)
 *   qs_get_state/qs_set_state      envs[i].dynamics.{pos,vel,rot,omega,...} attribute access
 *                                  (gym_art/quadrotor_multi/quadrotor_dynamics.py:180-191)
 *   qs_set_param             rew_coeff updates / set_capture_radius  quadrotor_multi.py:101-112, quadrotor_multi_rewards.py:210-211
 *   qs_episode_stats         infos[i]['episode_extra_stats'] summed over a rollout   gym_art/quadrotor_multi/quadrotor_multi.py:739-831
 *   qs_episode_records       infos[i]['episode_extra_stats'] per finished episode    (same lines)
 *   qs_set_reward_info       infos[i]['rewards'] of every step        gym_art/quadrotor_multi/quadrotor_single.py:69-84, quadrotor_multi.py:642-649
 *                            infos[i]['goal_dist'] (fork env)         gym_art/quadrotor_multi/quadrotor_single_rewards.py:457
 *
 * Conventions
 *   - plain C types only; all device pointers are raw CUDA device addresses (e.g. torch tensor.data_ptr()).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Nothing in qs_step /
 *     qs_reset allocates, synchronises or touches the host; the *_host variants copy through pinned staging
 *     buffers owned by the handle and synchronise the stream before returning.
 *   - every call returns 0 on success or a negative qs_status; qs_last_error() gives a message.
 *   - a handle is bound to one device and is not thread-safe (reference analogue: one process per env).
 *   - N = num_envs on this device, K = num_agents, D = qs_obs_dim(), A = qs_act_dim().
 *     Agent-major flattening is the reference VecEnv's: row = env * K + agent
 *     (swarm_rl/env_wrappers/subproc_vec_env_custom.py:145-147, 250-262).
 */
#ifndef QUADSIM_H_
#define QUADSIM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QS_API_VERSION 2
#define QS_MAX_AGENTS 32      /* drones per env handled by the warp-group kernels */
#define QS_MAX_OBSTACLES 64

typedef enum qs_status {
    QS_OK = 0,
    QS_ERR_BAD_CONFIG = -1,
    QS_ERR_CUDA = -2,
    QS_ERR_SHAPE = -3,
    QS_ERR_NULL = -4,
    QS_ERR_UNSUPPORTED = -5
} qs_status;

/* quads_mode values that run on the device (gym_art/quadrotor_multi/scenarios/) */
enum { QS_SCENARIO_STATIC_SAME_GOAL = 0,      /* scenarios/static_same_goal.py */
       QS_SCENARIO_O_MIX = 1,                 /* scenarios/mix.py with obstacles: o_random | o_static_same_goal per episode */
       QS_SCENARIO_O_RANDOM = 2,              /* scenarios/obstacles/o_random.py */
       QS_SCENARIO_O_STATIC_SAME_GOAL = 3,    /* scenarios/obstacles/o_static_same_goal.py */
       QS_SCENARIO_DYNAMIC_REPULSIVE = 4,     /* scenarios/dynamic_repulsive.py (fork mode: pursuit of a repelled evader) */
       /* formation scenarios of the upstream env (scenarios/base.py:42-173, one of 8 formations per episode) */
       QS_SCENARIO_STATIC_DIFF_GOAL = 5,      /* scenarios/static_diff_goal.py */
       QS_SCENARIO_DYNAMIC_SAME_GOAL = 6,     /* scenarios/dynamic_same_goal.py: a new common goal every 4-6 s */
       QS_SCENARIO_DYNAMIC_DIFF_GOAL = 7,     /* scenarios/dynamic_diff_goal.py: a new formation + centre every 4-6 s */
       QS_SCENARIO_SWAP_GOALS = 8,            /* scenarios/swap_goals.py: goals reshuffled every 4-6 s */
       QS_SCENARIO_DYNAMIC_FORMATIONS = 9,    /* scenarios/dynamic_formations.py: formation size breathing every step */
       QS_SCENARIO_MIX = 10,                  /* scenarios/mix.py without obstacles: one of the 9 (K = 1: 5) modes per episode */
       QS_SCENARIO_EP_LISSAJOUS3D = 11,       /* scenarios/ep_lissajous3D.py: common goal integrating a Lissajous velocity */
       QS_SCENARIO_EP_RAND_BEZIER = 12,       /* scenarios/ep_rand_bezier.py: common goal along random quadratic Bezier arcs */
       QS_SCENARIO_SWARM_VS_SWARM = 13,       /* scenarios/swarm_vs_swarm.py: two half-swarms exchanging formation centres */
       QS_SCENARIO_RUN_AWAY = 14 };           /* scenarios/run_away.py: every second drones 0 and 1 take over the goals of two random others (K >= 2) */

/* per-env state of the formation scenarios (the reference's QuadrotorScenario object, scenarios/base.py:9-35), as a row of
 * QS_SC_COUNT floats in qs_state_view.scenario.  Integers are stored as exactly representable floats. */
enum { QS_SC_SCENARIO = 0,    /* the scenario of the current episode (differs from qs_config.scenario under mix) */
       QS_SC_FORMATION = 1,   /* index into QUADS_FORMATION_LIST, scenarios/utils.py:25-26 */
       QS_SC_SIZE = 2,        /* formation_size */
       QS_SC_LAYER_DIST = 3,
       QS_SC_HIGHEST = 4,     /* highest_formation_size */
       QS_SC_LOWEST = 5,      /* lowest_formation_size */
       QS_SC_CENTER = 6,      /* formation_center xyz (6..8) */
       QS_SC_CTL_STEPS = 9,   /* control_step_for_sec: goals change when tick % this == 0 */
       QS_SC_INCREASE = 10,   /* dynamic_formations: growing (1) or shrinking (0) */
       QS_SC_SPEED = 11,      /* dynamic_formations: control_speed */
       QS_SC_AUX = 12,        /* 12..20: swarm_vs_swarm goal_center_1, goal_center_2 | ep_rand_bezier control points P0 P1 P2 */
       QS_SC_COUNT = 24 };

/* env_mode: which of the reference's two live env variants the handle reproduces */
enum { QS_MODE_UPSTREAM = 0,   /* gym_art/quadrotor_multi/quadrotor_multi.py + quadrotor_single.py (RawControl, 4 motor thrusts) */
       QS_MODE_FORK = 1 };     /* quadrotor_multi_rewards.py + quadrotor_single_rewards.py: PID pre-controller, 2-D action,
                                  `substeps` control steps per call, capture reward (what swarm_rl/sb_train.py trains on) */

/* obs_repr (gym_art/quadrotor_multi/quad_utils.py:30-38, get_state.py:226-292) */
enum { QS_OBS_XYZ_VXYZ_R_OMEGA = 0, QS_OBS_XYZ_VXYZ_R_OMEGA_FLOOR = 1, QS_OBS_XYZ_VXYZ_R_OMEGA_WALL = 2,
       /* fork 2-D representations (get_state.py:7-103), QS_MODE_FORK only */
       QS_OBS_CDIST_CDISTDOT_DIST_DISTDOT_ANGLE_ANGLEDOT = 3,   /* 6 floats, get_state.py:37-69 */
       QS_OBS_CDIST_CDISTDOT_DIST_DISTDOT_SANGLE_ANGLEDOT = 4,  /* 7 floats, get_state.py:71-103 */
       QS_OBS_AW_AWDOT_DIST_DISTDOT_ANGLE_ANGLEDOT = 5,         /* 6 floats, get_state.py:7-35 */
       QS_OBS_CDIST_CDISTDOT_NDIST_DISTDOT_NSANGLE_ANGLEDOT = 6 }; /* 7 floats, get_state.py:190-224: distance and bearing of the goal as
                                                                     the camera model measures them (pixel noise, best of n cameras) */

/* neighbor_obs_type (quad_utils.py:40-58) */
enum { QS_NEIGHBOR_NONE = 0, QS_NEIGHBOR_POS_VEL = 1,
       /* fork types (quadrotor_multi_rewards.py:326-358), QS_MODE_FORK only */
       QS_NEIGHBOR_DIST_ANGLE = 2,      /* [|dp|, bearing - heading] */
       QS_NEIGHBOR_DIST_SANGLE = 3,     /* [|dp|, cos, sin of the relative bearing] */
       QS_NEIGHBOR_DIST_ANGLE_HEADING = 4,    /* + heading_j - heading_i wrapped (:372-376) */
       QS_NEIGHBOR_DIST_SANGLE_SHEADING = 5,  /* + cos, sin of the relative heading (:377-382) */
       QS_NEIGHBOR_NDIST_NSANGLE = 6 };       /* camera model: [noisy dist clipped to 0..10, cos, sin of the noisy bearing]
                                                 (simulate_camera_measurement_vect, quadrotor_multi_rewards.py:238-324,338-347,370-371) */

/* noise source: counter-based Philox on the device (production) */
enum { QS_SENSE_NOISE_NONE = 0, QS_SENSE_NOISE_DEFAULT = 1 };

/* qs_set_param keys */
enum { QS_PARAM_REW_POS = 0, QS_PARAM_REW_EFFORT, QS_PARAM_REW_CRASH, QS_PARAM_REW_ORIENT, QS_PARAM_REW_SPIN,
       QS_PARAM_REW_QUADCOL_BIN, QS_PARAM_REW_QUADCOL_BIN_SMOOTH_MAX, QS_PARAM_REW_QUADCOL_BIN_OBST,
       QS_PARAM_CAPTURE_RADIUS,   /* set_capture_radius, quadrotor_multi_rewards.py:210-211 */
       QS_PARAM_COUNT };

/* Constants of the fork's pre-controller and pursuit task, evaluated once on the host from the reference's
 * construction-time code (fork_model.py) -- only read when env_mode == QS_MODE_FORK. */
typedef struct qs_fork_config {
    int32_t substeps;             /* control steps per step() call: 8, quadrotor_multi_rewards.py:633 */
    int32_t reserved;
    double capture_radius;        /* initial_capture_radius, quadrotor_multi_rewards.py:205-208 */
    double rew_existence;         /* -0.1  (:744) */
    double rew_captor;            /* 100   (:741) */
    double rew_helper;            /* 100   (:743) */
    double max_angular_rate;      /* pi*80/180 rad/s, Controller/Controller.py:31 */
    double chaser_speed;          /* 0.2 m/s, Controller/Controller.py:89 */
    double evader_v_max;          /* 0.5,  scenarios/dynamic_repulsive.py:31 */
    double evader_dt;             /* 1/200, :32 */
    double evader_arena;          /* 5,    :35 */
    double spawn_ring;            /* 0.5,  :75 */
    double evader_r_min;          /* 2,    :79 */
    double evader_r_span;         /* 3,    :79 */
    /* 12 PIDs in cascade order: position x,y,z; velocity x,y,z; attitude x,y,z; rate x,y,z.
     * Columns: kp, kd, ki, saturation (<=0: none), antiwindup (<=0: none).  Controller/Pid.py:7-26 and the
     * initialize_pids() of Position/Velocity/Attitude/RateController.py. */
    double pid[12][5];
    double rate_out_scale;        /* 800, Controller/RateController.py:84-86 */
    double mixer[4][4];           /* allocation_matrix_inv [motor][roll,pitch,yaw,throttle], Controller/Mixer.py:31-65 */
    double ctrl_mass;             /* ModelParams.mass 0.028, Controller/MultirotorModel.py:14 */
    double ctrl_g;                /* 9.81 */
    double ctrl_kf;               /* 1.25e-9 */
    double ctrl_min_rpm;          /* 1170 */
    double ctrl_max_rpm;          /* 13000 */
    /* camera model of the ndist / nsangle neighbour observations (swarm_rl/global_cfg.py:12-17) */
    double cam_focal_length;      /* focal_length_cam 0.035 m */
    double cam_target_size;       /* neighbour_size_cam 0.2 m */
    double cam_pixel_noise;       /* pixel_noise_cam (std, px); sb_train.py:136 sets 0 */
    double cam_fov_deg;           /* 70  (quadrotor_multi_rewards.py:286) */
    double cam_resolution;        /* 640 (:287) */
    int32_t cam_num;              /* n_cameras 3 */
    int32_t reserved2;
} qs_fork_config;

/*
 * Flat, POD configuration.  Host code evaluates the reference's construction-time Python once
 * (quad_models.py / inertia.py / quadrotor_dynamics.py:106-168 / quadrotor_single.py:139-234) and
 * passes the resulting constants here.  Doubles on purpose: the library rounds to fp32 itself.
 */
typedef struct qs_config {
    int32_t api_version;          /* must be QS_API_VERSION */
    int32_t num_envs;             /* N, environments on this device */
    int32_t num_agents;           /* K <= QS_MAX_AGENTS */
    int32_t scenario;             /* QS_SCENARIO_* */
    int32_t obs_repr;             /* QS_OBS_* */
    int32_t neighbor_obs_type;    /* QS_NEIGHBOR_* */
    int32_t neighbor_visible_num; /* resolved: 0..K-1 (reference's -1 means K-1) */
    int32_t use_obstacles;        /* quadrotor_multi.py:128-140 */
    int32_t use_downwash;         /* quadrotor_multi.py:663-668 */
    int32_t apply_collision_force;/* quadrotor_multi.py:227 */
    int32_t sense_noise;          /* QS_SENSE_NOISE_* (quadrotor_single.py:236-247) */
    int32_t ep_len;               /* int(ep_time / (dt * sim_steps)), quadrotor_single.py:158 */
    int32_t sim_steps;            /* physics sub-steps per control step (2) */
    int32_t svd_period;           /* sub-steps between re-orthonormalisations (quadrotor_dynamics.py:554-558) */
    int32_t obst_area_len;        /* int(obst_spawn_area[0]) */
    int32_t obst_area_wid;        /* int(obst_spawn_area[1]) */
    int32_t num_obstacles;        /* int(density * area), quadrotor_multi.py:138 */
    int32_t env_mode;             /* QS_MODE_* */
    int32_t cube_dim[3];          /* cube formation: int(np.power(n, 1/3)) for n = K, K/2, K - K/2 (scenarios/base.py:101-102); evaluated
                                     on the host with numpy like the reference, because the last-ulp rounding of that power decides
                                     e.g. int(27 ** (1/3)) == 2 */
    int32_t reserved0;
    uint64_t seed;                /* Philox key */
    int64_t env_id_offset;        /* global id of local env 0 (multi-GPU sharding keeps streams G-independent) */

    double dt;                    /* 1 / sim_freq = 0.005 */
    double room_dims[3];          /* length, width, height -> box [-L/2,L/2]x[-W/2,W/2]x[0,H] */
    double gravity;               /* 9.81 */
    /* QuadrotorDynamics.update_model, quadrotor_dynamics.py:106-168 */
    double mass;
    double inertia[3];
    double thrust_max[4];
    double torque_max[4];
    double prop_cross[4][3];      /* np.cross(prop_pos, [0,0,1]) */
    double prop_ccw[4];
    double arm;                   /* ||motor_xyz[:2]||, also the numba floor threshold (quadrotor_dynamics.py:385) */
    double motor_tau_up;          /* 4*dt/(damp_time_up+1e-6) */
    double motor_tau_down;
    double motor_linearity;
    double vel_damp;
    double damp_omega_quadratic;
    double omega_max;             /* 40 */
    double floor_mu;              /* 0.6 */
    double ou_theta;              /* 0.15  (numba_utils.py:77-105) */
    double ou_sigma;              /* 0.2 * thrust_noise_ratio */
    /* SensorNoise defaults, sensor_noise.py:69-76 */
    double sense_pos_std;         /* 0.005 */
    double sense_vel_std;         /* 0.01 */
    double sense_gyro_std;        /* 0.000175 */
    /* reward coefficients, quadrotor_multi.py:101-112 */
    double rew_pos, rew_effort, rew_crash, rew_orient, rew_spin;
    double rew_quadcol_bin, rew_quadcol_bin_smooth_max, rew_quadcol_bin_obst;
    /* collisions, quadrotor_multi.py:164-165 */
    double collision_hitbox_radius;   /* x arm */
    double collision_falloff_radius;  /* x arm */
    /* reset, quadrotor_single.py:215-218,406-418 */
    double spawn_box;             /* 2.0 (0.1 with obstacles) */
    double spawn_min_z;           /* 0.75 */
    /* obstacles, obstacles/obstacles.py:8-14 */
    double obst_size;             /* diameter */
    double sdf_resolution;        /* 0.1 */
    double approach_goal_metric;  /* scenarios/base.py:35 (0.5); o_static_same_goal uses 1.0 */
    qs_fork_config fork;          /* QS_MODE_FORK only */
} qs_config;

/* SoA view used by qs_get_state / qs_set_state.  Every pointer is a DEVICE pointer to a dense
 * row-major array, or NULL to skip that field.  Shapes: [N*K, c] unless noted. */
typedef struct qs_state_view {
    float *pos;          /* [N*K,3] */
    float *vel;          /* [N*K,3] */
    float *rot;          /* [N*K,9] row-major body->world */
    float *omega;        /* [N*K,3] body frame */
    float *rot_damp;     /* [N*K,4] thrust_rot_damp */
    float *cmds_damp;    /* [N*K,4] thrust_cmds_damp */
    float *ou;           /* [N*K,4] OU thrust-noise state */
    float *goal;         /* [N*K,3] */
    int32_t *flags;      /* [N*K]   bit0 on_floor, bit1 crashed_floor, bit2 crashed_wall, bit3 crashed_ceiling,
                                    bit4 prev_new_wall, bit5 prev_new_ceiling, bit6 prev_new_room, bit7 prev_obst_hit;
                                    higher bits are internal (bit 15: the obstacle scenario of the episode, kept by qs_set_state) */
    uint32_t *col_mask;  /* [N*K]   previous-step collision row (bit j set: pair (i,j) collided last step) */
    int32_t *tick;       /* [N]     per-env episode tick */
    int32_t *svd_ctr;    /* [N]     sub-steps since the last re-orthonormalisation */
    uint32_t *step_ctr;  /* [N]     RNG launch counter of the HANDLE (steps + resets so far; a fork step counts fork.substeps), reported
                                    per env.  qs_set_state reads entry 0 and sets the handle's counter (DESIGN.md "RNG contract") */
    float *obst_xy;      /* [N, QS_MAX_OBSTACLES, 2] obstacle centres (first num_obstacles valid) */
    float *scenario;     /* [N, QS_SC_COUNT] formation-scenario state (QS_SC_*); only for the formation scenarios */
    /* fork mode (NULL / ignored otherwise) */
    float *pid;          /* [N*K,24] (last_error, integral) of the 12 PIDs in cascade order */
    float *heading;      /* [N*K,3]  pre_controller.angle, pre_controller.angular_velocity, env.heading snapshot
                                     (refreshed in step only, quadrotor_multi_rewards.py:647) */
    float *evader;       /* [N,2]    Scenario_dynamic_repulsive.pos */
} qs_state_view;

/* Per-rollout aggregate of the reference's per-episode 'episode_extra_stats' (quadrotor_multi.py:739-831):
 * sums over all episodes that finished since the last qs_episode_stats(reset=1). */
typedef struct qs_stats {
    int64_t episodes;
    int64_t num_collisions;
    int64_t num_collisions_after_settle;
    int64_t num_collisions_final_5s;
    int64_t num_collisions_with_room;
    int64_t num_collisions_with_floor;
    int64_t num_collisions_with_wall;
    int64_t num_collisions_with_ceiling;
    int64_t num_collisions_obst_quad;
    int64_t num_collisions_obst_quad_after_settle;
    int64_t agents_success;       /* sum over episodes of #agents with no collision and reached goal */
    int64_t agents_deadlock;
    int64_t agents_collided;
    int64_t nonfinite_resets;     /* envs force-reset because a NaN/Inf appeared in their state */
    int64_t episodes_success;     /* fork mode: episodes that ended with the target caught (reset_info["success"]) */
    double  distance_to_goal_1s;  /* sum over episodes and agents of the per-agent mean distance in the last 1 s */
    double  distance_to_goal_3s;
    double  distance_to_goal_5s;
    double  reward_sum;           /* sum of all per-agent rewards of finished episodes */
} qs_stats;

/* Per-episode record: what the reference puts in infos[i]['episode_extra_stats'] when an episode ends
 * (quadrotor_multi.py:739-831, quadrotor_multi_rewards.py:886-978).  One row of QS_ER_COUNT int32 per env, describing the LAST
 * episode that env finished, plus one float4 per drone.  QS_ER_SEQ counts the episodes the env has finished since creation, so
 * a reader can tell a fresh record from an old one; the VecEnv layer reads the rows of the envs whose done flag is set. */
enum { QS_ER_SEQ = 0,                 /* episodes finished by this env so far (0: no record yet) */
       QS_ER_SCENARIO = 1,            /* QS_SCENARIO_* of the finished episode -> the f'{scenario_name}/...' keys */
       QS_ER_NUM_COLLISIONS = 2,      /* num_collisions */
       QS_ER_COLLISIONS_AFTER_SETTLE = 3,
       QS_ER_COLLISIONS_FINAL_5S = 4,
       QS_ER_COLLISIONS_ROOM = 5, QS_ER_COLLISIONS_FLOOR = 6, QS_ER_COLLISIONS_WALL = 7, QS_ER_COLLISIONS_CEILING = 8,
       QS_ER_COLLISIONS_OBST = 9,     /* num_collisions_obst_quad */
       QS_ER_COLLISIONS_OBST_AFTER_SETTLE = 10,
       QS_ER_AGENTS_SUCCESS = 11,     /* metric/agent_success_rate * K */
       QS_ER_AGENTS_DEADLOCK = 12,    /* metric/agent_deadlock_rate * K */
       QS_ER_AGENTS_COLLIDED = 13,    /* metric/agent_col_rate * K */
       QS_ER_AGENTS_NEIGHBOR_COL = 14,/* metric/agent_neighbor_col_rate * K */
       QS_ER_AGENTS_OBST_COL = 15,    /* metric/agent_obst_col_rate * K */
       QS_ER_EP_LEN = 16,             /* control steps of the episode */
       QS_ER_SUCCESS = 17,            /* fork mode: reset_info["success"]; upstream: 0 */
       QS_ER_NONFINITE = 18,          /* the episode was cut because a NaN/Inf appeared */
       QS_ER_COUNT = 20 };
/* per-drone part: { distance_to_goal_1s, distance_to_goal_3s, distance_to_goal_5s, 0 } of the finished episode.  The fork env
 * never fills its distance log (quadrotor_multi_rewards.py:797 is commented out), so there the three are NaN as in the reference. */

typedef struct qs_env qs_env;

size_t      qs_config_size(void);     /* sizeof(qs_config), for binding self-checks */
size_t      qs_stats_size(void);
int         qs_api_version(void);
const char *qs_last_error(const qs_env *env);   /* env may be NULL: last creation error */

int qs_create(const qs_config *cfg, int device, qs_env **out);
int qs_destroy(qs_env *env);

int qs_num_envs(const qs_env *env);
int qs_num_agents(const qs_env *env);
int qs_obs_dim(const qs_env *env);
int qs_act_dim(const qs_env *env);
/* number of kernels the library has launched since creation (bench.py's gpu_launches claim) */
int64_t qs_launch_count(const qs_env *env);

/* reset all envs (env_mask == NULL) or those with env_mask[e] != 0 (device uint8 [N]); writes obs [N*K,D]
 * (rows of envs that were not reset are left untouched). */
int qs_reset(qs_env *env, const uint8_t *env_mask, float *obs, void *stream);

/* One control step for every env.
 *   actions      [N*K,A] device float32 (raw policy output; clipped inside like RawControl.step)
 *   obs          [N*K,D] device float32: next observation; for envs that finished, the observation after
 *                        the automatic reset (quadrotor_multi.py:836, subproc_vec_env_custom.py:43-46)
 *   rew          [N*K]   device float32
 *   done         [N*K]   device uint8 (all K agents of a finished env are 1, quadrotor_multi.py:838)
 *   terminal_obs [N*K,D] device float32 or NULL: last observation of the finished episode (rows of unfinished
 *                        envs untouched) -> infos[i]["terminal_observation"]
 *   reset_success [N]    device uint8 or NULL: for envs that finished this step, reset_info["success"] of the episode
 *                        that ended (fork mode: the target was caught, quadrotor_multi_rewards.py:625-627; upstream
 *                        mode: 0); entries of unfinished envs are untouched -> VecEnv.reset_infos
 * In QS_MODE_FORK one call advances every env by fork.substeps control steps (fewer if the episode ends inside,
 * quadrotor_multi_rewards.py:633,986-987), A = 2, and the reward is the last executed sub-step's (:634).
 */
int qs_step(qs_env *env, const float *actions, float *obs, float *rew, uint8_t *done,
            float *terminal_obs, uint8_t *reset_success, void *stream);

/* Same, HOST buffers.  H2D of actions and D2H of obs/rew/done happen inside; the call returns after the stream has
 * drained.  Page-locked buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory) are DMA'd directly, pageable ones
 * are staged through pinned buffers owned by the handle (one extra host memcpy each way). */
int qs_reset_host(qs_env *env, float *obs_host, void *stream);
int qs_step_host(qs_env *env, const float *actions_host, float *obs_host, float *rew_host,
                 uint8_t *done_host, float *terminal_obs_host /* nullable */, uint8_t *reset_success_host /* nullable */,
                 void *stream);

int qs_get_state(qs_env *env, const qs_state_view *view, void *stream);
int qs_set_state(qs_env *env, const qs_state_view *view, void *stream);

/* scalar parameter update (QS_PARAM_*), takes effect from the next step */
int qs_set_param(qs_env *env, int key, double value);

/* copies the aggregate episode statistics to *out (host); synchronises `stream`.  reset != 0 zeroes them. */
int qs_episode_stats(qs_env *env, qs_stats *out, int reset, void *stream);

/* Per-episode records (QS_ER_*).  env_rec: int32 [N, QS_ER_COUNT]; agent_rec: float [N*K, 4]; either may be NULL.
 * qs_episode_records copies device-to-device on `stream` without synchronising; the _host variant copies to host memory and
 * returns after the stream has drained. */
int qs_episode_records(qs_env *env, int32_t *env_rec, float *agent_rec, void *stream);
int qs_episode_records_host(qs_env *env, int32_t *env_rec_host, float *agent_rec_host, void *stream);

/* Per-step reward breakdown (optional, off by default).  rew_info: device float [N*K, QS_RI_COUNT], 16-byte aligned, owned by
 * the caller; from the next qs_step on every step writes, per drone, the RAW reward terms of the reference's
 * infos[i]["rewards"] (each already multiplied by dt where the reference does: quadrotor_single.py:69-84): the weighted entries are
 * raw * rew_coeff (Python side).  Fork mode writes infos[i]['goal_dist'] (quadrotor_single_rewards.py:457) into slot 0 and zeros
 * elsewhere -- its 'rewards' dict is empty in the reference.  NULL switches the output off again. */
enum { QS_RI_RAW_POS = 0,           /* rewraw_pos = rewraw_main; fork mode: goal_dist */
       QS_RI_RAW_ACTION = 1, QS_RI_RAW_CRASH = 2, QS_RI_RAW_ORIENT = 3, QS_RI_RAW_SPIN = 4,
       QS_RI_RAW_QUADCOL = 5,       /* rewraw_quadcol: -1 / 0 */
       QS_RI_PROXIMITY = 6,         /* rew_proximity */
       QS_RI_RAW_QUADCOL_OBST = 7,  /* rewraw_quadcol_obstacle: -1 / 0 */
       QS_RI_COUNT = 8 };
int qs_set_reward_info(qs_env *env, float *rew_info);

/* Snapshots: the whole simulator state of a handle as one self-describing HOST blob, for checkpoints and exact resumes
 * (reference: the env side of SB3 model.save / CheckpointCallback, which the reference cannot restore at all).  A step after
 * qs_restore is bitwise the step the snapshotted handle would have taken next.
 *   Layout (native byte order): uint32 magic "QSSN" | uint32 QS_SNAPSHOT_VERSION | uint64 sizeof(qs_config) | at offset 16 the
 *   handle's current qs_config, qs_set_param changes included | uint32 RNG launch counter | uint32 section count | uint64 bytes of
 *   every section | the sections, dense, in a fixed order: the state planes; per-env tick, svd counter, episode counters; obstacle
 *   centres [N, QS_MAX_OBSTACLES] (use_obstacles only); scenario rows (formation scenarios only); episode records (env rows, drone
 *   rows); qs_stats; fork mode: the PID / heading planes, evader, per-env fork flags.  A section absent in the mode has size 0.
 *   Section sizes depend on N, K and the mode only, never on the launch shape, so a snapshot restores into any handle created
 *   with the same qs_config, seed and env_id_offset included: a shard restores into its own handle only (qs_restore_shards below
 *   moves envs across shard boundaries).
 *   Not stored: the launch count, the reset-first scheduling lists (qs_restore empties them, as qs_create leaves them), the
 *   staging buffers of the *_host calls, and the qs_set_reward_info pointer (the target handle keeps its own).
 * Both calls take pinned or pageable host memory and return after `stream` has drained.  qs_snapshot writes
 * qs_snapshot_size(env) bytes (`bytes` may be larger).  qs_restore needs `bytes` equal to the target's size; it checks the header
 * and every qs_config field except the qs_set_param ones (those are taken from the snapshot) before it copies anything, and on a
 * mismatch returns QS_ERR_SHAPE (blob: magic, version, sizes) or QS_ERR_BAD_CONFIG (configuration) with the first differing
 * field named in qs_last_error, leaving the handle untouched. */
#define QS_SNAPSHOT_VERSION 1
size_t qs_snapshot_size(const qs_env *env);                                   /* 0 for NULL */
int    qs_snapshot(qs_env *env, void *dst_host, size_t bytes, void *stream);
int    qs_restore(qs_env *env, const void *src_host, size_t bytes, void *stream);

/* Resharded resume: loads this handle's envs, global ids [env_id_offset, env_id_offset + num_envs), from `count` snapshots
 * (blobs[i], bytes[i] bytes each) that qs_snapshot took on handles of any size -- the rank files of a run saved on another number of
 * GPUs.  Every env is independent and its random stream is keyed by (global env id, RNG launch counter), so the steps after the call
 * are bitwise the steps the old shards would have taken.
 *   Checks, on every blob before the first copy: magic, version, sizeof(qs_config), the section table against the blob's own num_envs,
 *   K and mode, and bytes[i] equal to the length it implies; every qs_config field equal to the handle's except num_envs,
 *   env_id_offset and the qs_set_param fields (those must agree among the blobs and are taken from them, as qs_restore does); the
 *   same RNG launch counter in every blob; env ranges that do not overlap and together cover the handle's range.  Blobs whose range
 *   does not meet the handle's are ignored, so every new shard may pass the full list of old ones.  On a failure the handle is
 *   untouched and the call returns QS_ERR_SHAPE (blob layout, env ranges, count < 1) or QS_ERR_BAD_CONFIG (configuration, RNG
 *   counter) with the first problem named in qs_last_error (the field, or the first env no blob covers); QS_ERR_NULL for NULL arrays.
 *   Copies: one cudaMemcpyAsync per section per blob, of the slice of the envs this handle holds (every section is env-major).
 *   The handle's qs_stats become the sum, in blob order, of the stats of the blobs whose first env lies in its range: summed over
 *   the new handles, the totals are the old ones, each counted once.  The reset-first lists are emptied as qs_restore does.
 * Pinned or pageable host memory; returns after `stream` has drained.  restore_shards of one blob into a handle of the blob's own
 * range is qs_restore. */
int    qs_restore_shards(qs_env *env, const void *const *blobs, const size_t *bytes, int count, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* QUADSIM_H_ */
