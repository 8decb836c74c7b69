/*
 * gpd.h — C ABI of the B200-native batched quadrotor simulator (libgpd_b200.so).
 *
 * Drop-in boundary for the Physics.DYN hot path of komxun/gym-pybullet-drones-routing.
 * The reference is pure Python (no FFI of its own); each entry point below names the
 * reference interface it replaces (paths relative to gym_pybullet_drones/ in the reference).
 * INTEGRATION.md shows the ctypes stub a reference maintainer would add.
 *
 * Conventions
 *   - plain C: pointers and sizes only, no CUDA/torch types. `stream` is a cudaStream_t
 *     passed as void* (NULL = the legacy default stream).
 *   - every function returns 0 on success or a negative gpd_status; the message is read
 *     with gpd_last_error() (thread-local). Nothing ever calls exit().
 *   - "dev" pointers are CUDA device memory on the handle's device, owned by the caller
 *     (PyTorch tensors in the Python host code). The library owns only its persistent
 *     per-drone state allocated in gpd_create(). No hidden allocation or sync in gpd_step().
 *   - Real = float (GPD_F32) or double (GPD_F64), fixed per handle.
 *   - E = num_envs, N = num_drones, A = action width, B = ctrl_freq/2 (action ring length),
 *     W = obs row width: 12 + A*B for the RL envs (float32), 20 for the Ctrl env (Real).
 *   - quaternions are xyzw (pybullet order).
 *   - a handle is not thread-safe; distinct handles are independent. Calls are asynchronous
 *     on `stream`.
 */
#ifndef GPD_H
#define GPD_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPD_VERSION 200            /* 0.2.0 */
#define GPD_MAX_DRONES_PER_ENV 256 /* one thread block owns whole envs */

typedef enum gpd_status {
    GPD_OK = 0,
    GPD_ERR_INVALID = -1,    /* bad argument / unsupported configuration */
    GPD_ERR_CUDA = -2,       /* a CUDA runtime call failed */
    GPD_ERR_NO_DEVICE = -3,  /* no usable CUDA device: there is NO CPU fallback */
    GPD_ERR_ALLOC = -4
} gpd_status;

/* utils/enums.py:3-8 */
typedef enum gpd_drone_model { GPD_CF2X = 0, GPD_CF2P = 1, GPD_RACE = 2 } gpd_drone_model;
typedef enum gpd_precision { GPD_F32 = 0, GPD_F64 = 1 } gpd_precision;
/* utils/enums.py:35-41 (+ CtrlAviary.py:140 raw RPM with clip to [0, MAX_RPM]) */
typedef enum gpd_action_type {
    GPD_ACT_RPM = 0, GPD_ACT_PID = 1, GPD_ACT_VEL = 2, GPD_ACT_ONE_D_RPM = 3, GPD_ACT_ONE_D_PID = 4,
    GPD_ACT_CTRL_RPM = 5,   /* CtrlAviary: raw RPM, clipped to [0, MAX_RPM] (CtrlAviary.py:140) */
    GPD_ACT_CTRL_VEL = 6    /* VelocityAviary: (vx, vy, vz, speed fraction) tracked by DSLPIDControl (VelocityAviary.py:129-170) */
} gpd_action_type;
/* envs/CtrlAviary.py (+ envs/VelocityAviary.py: same observation/reward shape), envs/HoverAviary.py, envs/MultiHoverAviary.py */
typedef enum gpd_env_kind { GPD_ENV_CTRL = 0, GPD_ENV_HOVER = 1, GPD_ENV_MULTIHOVER = 2 } gpd_env_kind;
/* DYN-form force models (BaseAviary.py:715-811 recast for Physics.DYN; see DESIGN.md) */
enum { GPD_PHY_GND = 1, GPD_PHY_DRAG = 2, GPD_PHY_DW = 4 };

/* Replaces BaseAviary._parseURDFParameters (BaseAviary.py:982-1014) + derived constants
 * (BaseAviary.py:74,117-128). Filled on the host in float64 exactly as the reference does;
 * the device never recomputes them. ROTOR_XYZ: CoM offsets of rotor links 0-3 (cf2x.urdf:42-78). */
typedef struct gpd_drone_params {
    int32_t model;
    int32_t _pad;
    double M, L, THRUST2WEIGHT;
    double J[3], J_INV[3];
    double KF, KM;
    double COLLISION_H, COLLISION_R, COLLISION_Z_OFFSET;
    double MAX_SPEED_KMH, GND_EFF_COEFF, PROP_RADIUS;
    double DRAG_COEFF[3];
    double DW_COEFF_1, DW_COEFF_2, DW_COEFF_3;
    double G, GRAVITY, HOVER_RPM, MAX_RPM, MAX_THRUST, MAX_XY_TORQUE, MAX_Z_TORQUE, GND_EFF_H_CLIP;
    double ROTOR_XYZ[4][3];
} gpd_drone_params;

/* Replaces DSLPIDControl.__init__ (control/DSLPIDControl.py:37-60) and BaseControl.__init__
 * (control/BaseControl.py:35-39): gains, PWM map, mixer, the controller's own GRAVITY and KF. */
typedef struct gpd_pid_params {
    double P_FOR[3], I_FOR[3], D_FOR[3];
    double P_TOR[3], I_TOR[3], D_TOR[3];
    double PWM2RPM_SCALE, PWM2RPM_CONST, MIN_PWM, MAX_PWM;
    double MIXER[4][3];
    double GRAVITY, KF;
} gpd_pid_params;

/* Replaces the constructor arguments of BaseAviary/BaseRLAviary/HoverAviary/MultiHoverAviary/CtrlAviary
 * (BaseAviary.py:25-40, BaseRLAviary.py:16-29) plus the batch axis. */
typedef struct gpd_config {
    int32_t device;             /* CUDA device ordinal */
    int32_t precision;          /* gpd_precision */
    int64_t num_envs;           /* E */
    int32_t num_drones;         /* N, 1..GPD_MAX_DRONES_PER_ENV */
    int32_t pyb_freq;           /* BaseAviary.py:78 */
    int32_t ctrl_freq;          /* BaseAviary.py:77; pyb_freq % ctrl_freq must be 0 (BaseAviary.py:79-80) */
    int32_t env_kind;           /* gpd_env_kind */
    int32_t action_type;        /* gpd_action_type */
    int32_t physics_flags;      /* OR of GPD_PHY_* ; 0 = Physics.DYN */
    int32_t auto_reset;         /* 1: envs whose terminated|truncated fired are reset inside gpd_step (SB3 VecEnv contract) */
    int32_t threads_per_block;  /* physics threads per CTA (multiple of 32, <= 256); 0 = chosen by the library: a measured
                                 * default per shape, then the block size with the fewest waves for launches of 2-4 waves.
                                 * A pure scheduling choice: results are bit-identical for every value. */
    double episode_len_sec;     /* HoverAviary.py:52 */
    double speed_limit;         /* BaseRLAviary.py:95 (ActionType.VEL) */
    const double* target_pos;   /* host [N][3]: HoverAviary.py:51 / MultiHoverAviary.py:71; NULL for the Ctrl env */
    gpd_drone_params drone;
    gpd_pid_params pid;         /* used by the PID-family action types (BaseRLAviary.py:73-78) */
} gpd_config;

typedef struct gpd_sim gpd_sim;

int gpd_version(void);
const char* gpd_last_error(void);
/* number of visible CUDA devices, or a negative gpd_status */
int gpd_device_count(void);

/* BaseAviary.__init__ (BaseAviary.py:25-216). State starts at the reference's default initial poses
 * (BaseAviary.py:194-207) unless gpd_set_init_poses() is called; step counters 0; action ring zero. */
int gpd_create(const gpd_config* cfg, gpd_sim** out);
void gpd_destroy(gpd_sim* sim);

int gpd_obs_width(const gpd_sim* sim);     /* W */
int gpd_action_width(const gpd_sim* sim);  /* A */
int gpd_substeps(const gpd_sim* sim);      /* PYB_STEPS_PER_CTRL, BaseAviary.py:81 */

/* initial_xyzs / initial_rpys (BaseAviary.py:194-207). Host float64 arrays, [N][3] when per_env == 0
 * (every env identical, as in the reference) or [E][N][3] when per_env == 1. Takes effect at the next reset. */
int gpd_set_init_poses(gpd_sim* sim, const double* xyz, const double* rpy, int per_env);

/* TARGET_POS after construction (HoverAviary.py:51; MultiHoverAviary.py:71 TARGET_POS = INIT_XYZS + [0,0,1/(i+1)]).
 * Host float64 [N][3] (per_env == 0, every env shares the targets — the reference) or [E][N][3] (per_env == 1: envs that
 * start from their own poses are rewarded and terminated against their own targets). Drains the device. */
int gpd_set_targets(gpd_sim* sim, const double* target_pos, int per_env);

/* BaseAviary.reset (BaseAviary.py:220-255, _housekeeping :451-477) for the envs with env_mask[e] != 0
 * (dev uint8 [E]; NULL = all). The action ring and the in-env controllers are NOT reset
 * (BaseRLAviary.py:153-154,76). Writes the observation of every env into obs_out; the ring part of it is
 * taken from obs_prev (the previous observation buffer; NULL = all-zero ring, the state after __init__). */
int gpd_reset(gpd_sim* sim, const uint8_t* env_mask, const void* obs_prev, void* obs_out, void* stream);

/*
 * BaseAviary.step (BaseAviary.py:259-383): _preprocessAction (BaseRLAviary.py:160-239, CtrlAviary.py:140),
 * PYB_STEPS_PER_CTRL substeps of _dynamics/_integrateQ (BaseAviary.py:815-889) with the optional DYN-form
 * force models, _computeObs (BaseRLAviary.py:307-319 / CtrlAviary.py:117), _computeReward/_computeTerminated/
 * _computeTruncated (HoverAviary.py:68-117, MultiHoverAviary.py:84-130), step_counter += S.
 *   actions   dev [E][N][A]: float32 for the RL envs (the SB3 dtype, BaseRLAviary.py:156); Real for GPD_ACT_CTRL_RPM/_VEL
 *   obs_prev  dev, the observation written by the previous gpd_step/gpd_reset on this handle: the RL observation
 *             carries the action ring (BaseRLAviary.py:317-318), so the shifted history is read from it.
 *             NULL = all-zero ring. Ignored for the Ctrl env. Must not alias obs_out.
 *             FP32 single-drone KIN sims with an RPM-type action and no force model (GPD_STATE_IN_OBS=0 turns this off)
 *             keep position and velocity ONLY in the kin part of the latest observation (kin[0..2], kin[6..8]: the
 *             float32 state itself): the next step reads them from there, so an in-place edit of the returned observation
 *             is an edit of the env's state. A step whose obs_prev is neither the handle's latest obs_out nor the buffer
 *             given to gpd_note_latest_obs takes its state from the handle's own copy instead, like every other handle.
 *   obs_out   dev [E][N][W]: float32 (RL) / Real (Ctrl)
 *   reward    dev [E] Real (NULL allowed); terminated/truncated dev [E] uint8 (NULL allowed)
 *   terminal_kin dev [E][N][12] float32 or NULL: with auto_reset, the 12 kinematic observation entries of a
 *             finished env BEFORE its reset (its ring part equals the one in obs_out, which survives reset) —
 *             enough to rebuild SB3's infos[i]["terminal_observation"]. Rows of unfinished envs are untouched.
 */
int gpd_step(gpd_sim* sim, const void* actions, const void* obs_prev, void* obs_out,
             void* reward, uint8_t* terminated, uint8_t* truncated, void* terminal_kin, void* stream);

/*
 * Chained stepping (default OFF).  BaseAviary.step calls are strictly ordered (BaseAviary.py:259-383 returns before the
 * next call starts); gpd_step keeps that order on its stream: a step kernel starts only after ALL earlier work of the
 * stream has completed and its results are visible.  A caller whose step inputs do not depend on the work enqueued just
 * before the step — a pre-computed action schedule, an action repeated over k steps (frame skip), several independent
 * env sets stepped in rotation on one stream — may turn chaining on: consecutive gpd_step launches of the stream are then
 * launched programmatically (the next kernel starts while the previous one drains) and each tile of a handle waits only
 * for ITS OWN previous step (one 64-bit word per tile), so results are bit-identical to unchained stepping.
 * CONTRACT while chaining is on: `actions` (and every other input that is not this handle's own state or its previous
 * observation) must have been complete BEFORE the previous kernel of the stream was enqueued; never chain a step behind
 * the kernel that computes its actions (a policy network).  The library itself never chains the first step after
 * gpd_reset / gpd_set_state / gpd_set_* on a handle, nor a step issued on a different stream than the handle's last one.
 * No effect on shapes the library runs without per-tile sequencing (launches of more than ~4 waves).
 */
int gpd_set_step_chaining(gpd_sim* sim, int enable);

/* Host-buffer variant of gpd_step for numpy-style call sites (the reference's own step() signature): copies
 * `actions` from host memory, runs gpd_step on internal device buffers (an internal obs ping-pong pair), copies
 * obs/reward/terminated/truncated back and synchronises `stream`. Host pointers may be pageable or pinned.
 * terminal_kin may be NULL. */
int gpd_step_host(gpd_sim* sim, const void* actions, void* obs_out, void* reward,
                  uint8_t* terminated, uint8_t* truncated, void* terminal_kin, void* stream);
int gpd_reset_host(gpd_sim* sim, const uint8_t* env_mask, void* obs_out, void* stream);

/*
 * Host mirror of the RL observation: the numpy-facing step without the echo.
 *
 * 83 % of an RL observation row is the action ring (BaseRLAviary.py:187,307-319) — values the HOST sent. gpd_step_host
 * ships them back over PCIe every step (19.3 MB per 65,536-env HoverAviary step); gpd_step_mirror ships only what the
 * device computed (12 kinematic floats per drone, reward, terminated, truncated: 54 B per env, 3.5 MB) and keeps the host
 * observation in a FEATURE-MAJOR log in pinned host memory, log[row][col] (row = observation feature, col = drone):
 *     obs(e, n, j) of the current step = log[(first_row + j) * row_len + col0 + e*N + n],   j = 0 .. W-1
 * i.e. a strided view of shape (E, N, W) with element strides (N, 1, row_len) — the transpose of a dense [W][D] block.
 * A step slides the window by A rows: the 12 kin rows land (one contiguous device-to-host copy) on the rows the oldest ring
 * entry and the old kin rows occupied, the newest action is written by the host itself (transposed from `actions` while the
 * device works) behind the window. When the window reaches the end of the log it is rebuilt at row 0 from the device
 * observation (one W-row copy every (rows - W) / A steps); the same rebuild re-synchronises a mirror that went stale because
 * gpd_step / gpd_reset advanced the device chain without it. A view returned by step t stays intact until step t+1 begins.
 *
 *   gpd_mirror_alloc   pinned (cudaHostAlloc), zero-filled log of rows x row_len floats; gpd_mirror_free releases it
 *   gpd_mirror_attach  binds a log to a handle: rows >= W + A, row_len >= col0 + E*N. Several handles (env pools stepping
 *                      in lockstep) may share one log through different col0: their windows stay aligned and ONE strided
 *                      view covers all pools. RL envs only (the Ctrl observation has no ring: gpd_step_host).
 *   gpd_step_mirror    actions: host [E][N][A] float32 (pinned or pageable). d_obs_prev / d_obs_out: the DEVICE observation
 *                      chain exactly as in gpd_step (caller-owned, so tensor-path and numpy-path steps share one chain);
 *                      d_obs_out == NULL selects the handle's internal ping-pong. reward (Real) / terminated / truncated /
 *                      terminal_kin: host arrays, any may be NULL. *first_row receives the window's first row after the step.
 *                      Synchronises `stream`. _begin enqueues the device work and returns; _end writes the newest action into
 *                      the log (`actions` must stay valid until then), synchronises and publishes the window — several pools
 *                      on their own streams overlap one pool's H2D with another's D2H.
 *   gpd_reset_mirror   BaseAviary.reset for env_mask (HOST uint8 [E] or NULL = all): the ring survives (BaseRLAviary.py:153-154),
 *                      the window does not move, its 12 kin rows are refreshed.
 *
 * Zero-copy step: the log is mapped into the device's address space; when reward / terminated / truncated / terminal_kin are
 * pinned host arrays too (cudaHostAlloc, cudaHostRegister, torch's pin_memory) the step kernel itself writes the kin rows and
 * those arrays over PCIe, and reads `actions` from host memory if it is pinned (pageable actions are staged with one copy):
 * one kernel launch per step, no separate copy operations. Arrays the device cannot address fall back to staging + copies;
 * the results are the same either way.
 */
int gpd_mirror_alloc(int64_t rows, int64_t row_len, float** log_out);
int gpd_mirror_free(float* log);
int gpd_mirror_attach(gpd_sim* sim, float* log, int64_t rows, int64_t row_len, int64_t col0);
int64_t gpd_mirror_row(const gpd_sim* sim);
int gpd_step_mirror(gpd_sim* sim, const void* actions, const void* d_obs_prev, void* d_obs_out, void* reward,
                    uint8_t* terminated, uint8_t* truncated, void* terminal_kin, int64_t* first_row, void* stream);
int gpd_step_mirror_begin(gpd_sim* sim, const void* actions, const void* d_obs_prev, void* d_obs_out, void* reward,
                          uint8_t* terminated, uint8_t* truncated, void* terminal_kin, void* stream);
int gpd_step_mirror_end(gpd_sim* sim, int64_t* first_row, void* stream);
int gpd_reset_mirror(gpd_sim* sim, const uint8_t* env_mask, const void* d_obs_prev, void* d_obs_out, int64_t* first_row,
                     void* stream);

/* BaseAviary._getDroneStateVector (BaseAviary.py:541-561) for every drone + the hidden integrator state.
 *   state20 dev [E][N][20] Real: pos3 quat4 rpy3 vel3 ang_v3 last_clipped_action4
 *   rpy_rates dev [E][N][3] Real (BaseAviary.py:477,874); pid_state dev [E][N][9] Real: integral_pos_e3,
 *   integral_rpy_e3, last_rpy3 (DSLPIDControl.py:73-78); step_counter dev [E] int32. Any pointer may be NULL.
 * gpd_set_state reads pos, quat, vel, ang_v, last_clipped_action from state20 (rpy is derived). Together they
 * checkpoint/resume a simulation bit-exactly.
 * FP32 KIN sims with an RPM-type action and no force model keep ang_v and last_clipped_action only in the observation
 * row: gpd_get_state (and a masked gpd_reset) re-derive them, bit-exactly, from the observation buffer most recently
 * passed as obs_out - the same buffer the next gpd_step needs intact as obs_prev. */
int gpd_get_state(gpd_sim* sim, void* state20, void* rpy_rates, void* pid_state, int32_t* step_counter, void* stream);
/* Tells the library which device buffer now holds the latest observation (a caller that copied it elsewhere and is about to
 * release the buffer it passed as obs_out). Only FP32 KIN sims with an RPM-type action and no force model read it back;
 * for the single-drone ones it then carries the position and velocity the next step starts from (see gpd_step). */
int gpd_note_latest_obs(gpd_sim* sim, const void* obs);
int gpd_set_state(gpd_sim* sim, const void* state20, const void* rpy_rates, const void* pid_state,
                  const int32_t* step_counter, void* stream);

/* DSLPIDControl.computeControl (control/DSLPIDControl.py:82-145) for n independent controllers.
 * All arrays dev Real: cur_pos[n][3] cur_quat[n][4] cur_vel[n][3] target_pos[n][3]; target_rpy/target_vel/
 * target_rpy_rates [n][3] or NULL (= zeros, the reference's defaults); pid_state[n][9] in/out;
 * rpm_out[n][4]; pos_e_out[n][3] and yaw_e_out[n] optional. (cur_ang_vel is unused by the reference.) */
int gpd_pid_compute(int device, int precision, const gpd_pid_params* pid, int64_t n, double control_timestep,
                    const void* cur_pos, const void* cur_quat, const void* cur_vel, const void* target_pos,
                    const void* target_rpy, const void* target_vel, const void* target_rpy_rates,
                    void* pid_state, void* rpm_out, void* pos_e_out, void* yaw_e_out, void* stream);

/* Force models, unit-test entry points on raw arrays (dev Real):
 *   BaseAviary._groundEffect (BaseAviary.py:715-750): rpm[n][4] pos[n][3] quat[n][4] -> out[n][4] (+z LINK-frame
 *     force per rotor), applied[n] uint8 = the |roll|,|pitch| < pi/2 gate (BaseAviary.py:742)
 *   BaseAviary._drag (BaseAviary.py:754-781): rpm[n][4] quat[n][4] vel[n][3] -> out[n][3] (body frame)
 *   BaseAviary._downwash (BaseAviary.py:785-811): pos[E][N][3] -> out[E][N] (summed body-z force) */
int gpd_force_ground_effect(int device, int precision, const gpd_drone_params* d, int64_t n, const void* rpm,
                            const void* pos, const void* quat, void* out, uint8_t* applied, void* stream);
int gpd_force_drag(int device, int precision, const gpd_drone_params* d, int64_t n, const void* rpm,
                   const void* quat, const void* vel, void* out, void* stream);
int gpd_force_downwash(int device, int precision, const gpd_drone_params* d, int64_t num_envs, int32_t num_drones,
                       const void* pos, void* out, void* stream);

/* examples/pid.py:127-147 as one launch: n_ctrl_steps iterations of { env.step(action);
 * action = DSLPIDControl.computeControlFromState(obs, target = [waypoints[wp][0:2], INIT_XYZS z],
 * target_rpy = INIT_RPYS); wp = (wp + 1) % n_wp } with the controller in the kernel (Ctrl env only).
 *   waypoints dev [n_wp][3] Real; wp_counters dev [E][N] int32 in/out; action dev [E][N][4] Real in/out
 *   (the RPM applied by the next step; zeros at start, examples/pid.py:130). */
int gpd_rollout_pid(gpd_sim* sim, int32_t n_ctrl_steps, const void* waypoints, int32_t n_wp,
                    int32_t* wp_counters, void* action, void* stream);

/* K = n_steps control steps of BaseAviary.step with a given action schedule, in one launch.  Equivalent to
 * K calls of gpd_step with actions[k], each reading the previous one's observation. The differences:
 * only the final observation is written, and the per-step outputs land in rows of [K]-major arrays.
 *   actions      dev [K][E][N][A], dtype as gpd_step; 16-byte aligned
 *   obs_prev     as gpd_step (ring source of step 0; NULL = all-zero ring; ignored for the Ctrl env)
 *   obs_out      dev [E][N][W]: the observation after step K-1; must not alias obs_prev; 16-byte aligned
 *   reward       dev [K][E] Real or NULL;  terminated / truncated dev [K][E] uint8 or NULL
 *   traj         dev or NULL: the device-computed part of each step's observation, i.e. what gpd_step would
 *                have written there:
 *                [K][E][N][12] float32 (RL envs: kin) or [K][E][N][20] Real (Ctrl env: the whole row)
 *   terminal_kin dev [K][E][N][12] float32 or NULL: gpd_step's terminal_kin, per step (auto_reset, RL envs); rows of
 *                steps where the env did not finish are left untouched
 * Every configuration gpd_create accepts is supported. Auto-reset, episode statistics, counters and DSLPID
 * state advance exactly as over K steps. The rollout is never launched programmatically behind a chained step, nor a
 * step behind it; it allocates nothing and does not synchronise (graph-capturable). obs_out becomes the latest observation
 * (gpd_get_state, the next gpd_step's obs_prev, a host mirror's rebuild). GPD_ERR_INVALID for n_steps < 1, a NULL
 * actions / obs_out, aliased buffers, or actions / observations / traj / terminal_kin that are not 16-byte aligned. */
int gpd_rollout(gpd_sim* sim, int32_t n_steps, const void* actions, const void* obs_prev, void* obs_out,
                void* reward, uint8_t* terminated, uint8_t* truncated, void* traj, void* terminal_kin, void* stream);

/* Diagnostics: number of CTAs of a step launch, and an optional device buffer [grid][8] of uint64 that every step
 * launch fills with per-CTA phase timestamps in ns (%globaltimer): 0 CTA start, 1 previous kernel complete (PDL wait
 * passed), 2 state+action arrived, 3 substeps done, 4 physics outputs stored, 5 history tile landed in shared memory
 * (TMA load), 6 TMA store consumed shared memory, 7 block barrier passed. NULL (default) disables it. */
int gpd_grid_size(const gpd_sim* sim);
int gpd_set_timeline_buffer(gpd_sim* sim, unsigned long long* dev_buf);

/* Failure detection: number of drones whose position, quaternion, velocity or body rates hold a NaN/Inf (a DYN drone has
 * no ground and no RPM clip for ActionType.RPM — BaseRLAviary.py:192 — so bad actions diverge without bound).
 * Scans the persistent state; off the step path. Synchronises `stream`. */
int gpd_count_nonfinite(gpd_sim* sim, long long* out_host, void* stream);

/* Episode statistics kept on the device when auto_reset is on (what SB3's Monitor reports in the
 * single-process reference, examples/learn.py:53-57,142-146). out (host) = { episodes, sum_return, sum_length,
 * sum_return_sq, min_return, max_return, env_steps, terminated_episodes }. Synchronises `stream`.
 * clear != 0 zeroes the accumulators afterwards.
 * nccl_comm: an ncclComm_t (as void*) or NULL. NULL = this handle's statistics. With a communicator the result is
 * JOB-WIDE on every rank: one ncclAllGather of the 8 doubles + a rank-ordered combine on the device (sums added, min/max
 * over the ranks that finished an episode) — the only collective of the whole design, off the step path. libnccl.so.2 is
 * bound at run time (dlopen; the copy already loaded in the process is reused), never linked. */
int gpd_episode_stats(gpd_sim* sim, double out[8], int clear, void* nccl_comm, void* stream);

/* Communicator plumbing for callers without one (the Python host code: torch.distributed does not expose its ncclComm_t):
 * rank 0 calls gpd_nccl_unique_id and broadcasts the 128 bytes by any means; every rank then calls gpd_nccl_comm_init. */
#define GPD_NCCL_UNIQUE_ID_BYTES 128
int gpd_nccl_unique_id(char id_out[GPD_NCCL_UNIQUE_ID_BYTES]);
int gpd_nccl_comm_init(const char id[GPD_NCCL_UNIQUE_ID_BYTES], int rank, int world_size, int device, void** comm_out);
int gpd_nccl_comm_destroy(void* comm);

/* BaseAviary._getAdjacencyMatrix (BaseAviary.py:658-675) of every env from the current positions:
 * out dev [E][N][N] Real, 1 on the diagonal and where ||pos_i - pos_j|| < neighbourhood_radius, else 0. */
int gpd_adjacency(gpd_sim* sim, double neighbourhood_radius, void* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPD_H */
