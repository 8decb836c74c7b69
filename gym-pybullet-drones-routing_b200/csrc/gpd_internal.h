// gpd_internal.h — host/device shared declarations of libgpd_b200 (not part of the public ABI).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gpd.h"

namespace gpd {

enum { GPD_MAX_DEVICES = 64, GPD_BULK_MAX_TPC = 2 };

// per-block episode-statistics partials: sums {episodes, return, length, return^2, env_steps, terminated} and the
// min/max episode return as order-preserving int32 images of float32
struct StatSlot {
    double s[6];
    int32_t mn, mx;
};

template <typename R> struct Vec4;
template <> struct Vec4<float> { using type = float4; };
template <> struct Vec4<double> { using type = double4; };

// Drone constants in the compute type, plus the float64 originals the FP32 path needs for its
// cancellation-free rotor prologue (DESIGN.md "FP32 mode").
template <typename R>
struct DevDrone {
    // ---- hot: everything the lean (plain DYN, RPM action) kernel reads, packed into the first constant-bank lines ----
    int model;
    int _pad;
    double KF_d, KM_d, GRAVITY_d, L_d, ARM_d, HOVER_RPM_d, MAX_RPM_d;
    R GRAVITY, MAX_RPM;
    R DT_INV_M, DT_JINV[3]; // FP32 mode: PYB_TIMESTEP/M and PYB_TIMESTEP*J^-1 (filled by gpd_create)
    R DT_EULER[3];          // FP32 mode: PYB_TIMESTEP*J^-1[k]*(J[k+2]-J[k+1]), the gyroscopic coefficients of the diagonal J
    R J[3], JINV[3];
    R M, L, ARM;            // ARM = L/sqrt(2)  (BaseAviary.py:847-848)
    R INV_M;                // RN(1/M), for div_by_const (FP64 kernels)
    R KF, KM;
    // ---- cold: force models ----
    R GND_EFF_COEFF, PROP_RADIUS, GND_EFF_H_CLIP;
    R ROTOR[4][3];
    R DRAG[3];
    R DW1, DW2, DW3;
    R DW1_NEG_PR2_16;       // -DW1 * (PROP_RADIUS / 4)^2, folded on the host in double (FP32 downwash pair)
};

template <typename R>
struct DevPid {
    R P_FOR[3], I_FOR[3], D_FOR[3], P_TOR[3], I_TOR[3], D_TOR[3];
    R PWM2RPM_SCALE, PWM2RPM_CONST, MIN_PWM, MAX_PWM;
    R MIXER[4][3];
    R GRAVITY, KF4;         // KF4 = 4*KF of the controller's own model (DSLPIDControl.py:198)
};

// Persistent per-drone state, SoA of 16-byte vectors (D = E*N drones):
//   sP = (pos.x, pos.y, pos.z, rates.x)   sQ = quat xyzw   sV = (vel.x, vel.y, vel.z, rates.y)   sWz = rates.z
//   aux_av = (ang_v.xyz, 0), aux_rpm = last_clipped_action   (outputs kept so gpd_get_state is exact).
//   Lean FP32 KIN sims (StepArgs::skip_aux) do not write them per step: both are bit-exact functions of the observation
//   row (kin[9..11]; newest ring slot + counter) and are re-derived on demand; *aux_auth says which copy is authoritative.
//   pid[k*D + d], k = 0..8
//   Chained-state handles (StepArgs::state_in_obs): the bulk step keeps position and velocity only in the kin part of the
//   latest observation row (kin[0..2], kin[6..8]: the float32 state itself), rates and episode return in StepArgs::sR =
//   (rates.xyz, ep_ret); a tile whose flag (tile_seq[4 * tile + 1]) is set holds its state so, and launch_state_sync writes
//   it back into sP / sV / sWz / ep_ret for every other reader or writer of the state.
template <typename R>
struct SimPtrs {
    typename Vec4<R>::type* sP;
    typename Vec4<R>::type* sQ;
    typename Vec4<R>::type* sV;
    R* sWz;
    typename Vec4<R>::type* aux_av;
    typename Vec4<R>::type* aux_rpm;
    int32_t* aux_auth;      // [1] 1 = the aux arrays are authoritative (after reset-all / gpd_set_state), 0 = derive from the obs row
    R* pid;
    int32_t* counter;       // [E] BaseAviary.step_counter
    float* ep_ret;          // [E] running episode return (auto_reset only)
    StatSlot* stat_slots;   // [grid] per-block statistics partials (fire-and-forget atomics, no contention)
    const typename Vec4<R>::type* init_pos;   // [N] or [D]  (xyz, 0)
    const typename Vec4<R>::type* init_quat;  // [N] or [D]
    const typename Vec4<R>::type* target;     // [N] or [D] (xyz, 0)
};

template <typename R>
struct StepArgs {
    // hot scalars first (constant-bank locality: the kernel entry stalls on every distinct 64-byte line it touches)
    int64_t D;              // total drones
    int64_t E;
    int N, S, A, B, W;
    int DPB, EPB;           // drones / envs per block
    int env_kind, action_type, phy, auto_reset, init_per_env;
    int32_t max_counter;    // largest step_counter with step_counter/PYB_FREQ <= EPISODE_LEN_SEC (HoverAviary.py:114)
    int32_t copy_threads;   // last threads of the block: they only move the action history (RL envs)
    int32_t use_tma;        // history moved by TMA tensor copies (needs obs_prev and float4-granular rows)
    int32_t tma_bytes;      // shared-memory bytes reserved for the TMA tile (multiple of 128)
    int32_t tma_bytes_box;  // bytes one TMA box transfers: DPB * (B-1-2*tma_edge) * 16
    int32_t skip_aux;          // lean FP32 KIN sims: ang_v / last_clipped_action live in the observation row, not in aux_*
    int32_t pdl_trigger_early; // PDL: release the dependent launch at CTA start (small grids) or after this CTA's stores
    int32_t tma_edge_bytes; // shared-memory bytes of one edge box (DPB*16 rounded up to 128)
    int32_t tma_edge;       // 1: rows are 32-byte aligned, the box skips the first and last shifted slot (written by the drone's thread)
    R dt, ctrl_dt, speed_limit;
    const void* actions;
    const float* obs_prev;
    void* obs_out;
    R* reward;
    uint8_t* terminated;
    uint8_t* truncated;
    float* terminal_kin;
    const uint8_t* reset_mask;   // reset kernel only
    unsigned long long* timeline; // diagnostics: [grid][8] phase timestamps (ns, %globaltimer) or nullptr
    float* kin_t;           // host-mirror export: feature-major copy [12][kin_ld] of the kinematic observation part, or nullptr
    int64_t kin_ld;         // row stride of kin_t: D for the device staging, the log's row length when the rows ARE the pinned host log
    unsigned long long* tile_seq;   // per-CTA step sequencing, one 64-bit word per tile at a 32-byte stride (tile_claim_and_wait)
    int32_t tile_dep;       // 1: a CTA waits only for ITS OWN tile's previous step (per-CTA flag) instead of the whole grid
    int32_t target_per_env; // 1: p.target holds D entries (per-env MultiHover targets), else N
    int32_t cta0;           // block-index offset of a step launch: always 0 (dropping it from gpd::step_kernel measured 1 % slower on C4)
    int32_t out_plain;      // bulk path, per call: reward / terminated / truncated are not all 16-byte aligned -> plain stores by the threads
    int32_t tpc;            // bulk path, per call: tiles per CTA (0/1 = one; chained launches may take GPD_BULK_MAX_TPC)
    int32_t tile_end;       // bulk path, per call: first tile not covered by this launch
    int32_t bulk_direct;    // bulk path: what bypasses shared memory (0 nothing, 1 the small per-env arrays, 2 the state vectors too)
    int32_t state_in_obs;   // lean FP32 single-drone sims on the bulk kernel: position / velocity chained through the observation (SimPtrs)
    SimPtrs<R> p;
    DevDrone<R> drone;
    DevPid<R> pid;
    double pyb_freq, episode_len;
    // after everything the other kernels read, so that their parameter layout does not depend on it
    typename Vec4<R>::type* sR;   // [D] chained-state handles only: (rates.x, rates.y, rates.z, ep_ret)
};

// gpd_plan's own arguments, a separate kernel parameter so that StepArgs (every other kernel's parameter layout) is unchanged.
// D / E count the copies: E = source envs * n_samples, D = E * N.  Outputs as in include/gpd.h.
template <typename R>
struct PlanArgs {
    int64_t D, E;
    int32_t n_samples;
    R gamma;
    const R* targets;       // [E_src][N][3] or nullptr (the handle's own)
    R* returns;             // [E]
    int32_t* done_step;     // [E] or nullptr
    R* reward;              // [K][E] or nullptr
    float* final_kin;       // [D][12] or nullptr
};

// gpd_plan_grad's own arguments (PlanArgs' copy counts and return outputs, the gradient and the tape)
template <typename R>
struct PlanGradArgs {
    int64_t D, E;
    int32_t n_samples;
    R gamma;
    const R* targets;       // [E_src][N][3] or nullptr (the handle's own)
    R* returns;             // [E]
    int32_t* done_step;     // [E] or nullptr
    R* grad;                // [K][D][A]
    R* tape;                // [K][13][D]: each copy drone's state at the start of every control step
};

struct LaunchCfg {
    int threads;
    int64_t grid;
    size_t smem;
    int pdl;                // launch step kernels with programmatic stream serialization
};

// implemented once per precision in gpd_f32.cu / gpd_f64.cu
// step-kernel code variants (template axis KIND of gpd::step_kernel)
enum { GPD_K_FORCES = 0, GPD_K_LEAN = 1, GPD_K_PID = 2 };

template <typename R> int step_blocks_per_sm(int action_type, int phy, int N, int A, int W, int env_kind, int threads, size_t smem);
template <typename R> cudaError_t launch_step(const StepArgs<R>& a, const LaunchCfg& lc, const CUtensorMap* tm_prev,
                                              const CUtensorMap* tm_out, const CUtensorMap* tm_edge, cudaStream_t st);
template <typename R> int step_bulk_blocks_per_sm(int action_type, int phy, int N, int threads, size_t smem);
template <typename R> cudaError_t launch_step_bulk(const StepArgs<R>& a, const LaunchCfg& lc, cudaStream_t st);
template <typename R> cudaError_t launch_reset(const StepArgs<R>& a, const LaunchCfg& lc, cudaStream_t st);
template <typename R> cudaError_t launch_get_state(const StepArgs<R>& a, const float* obs_latest, R* state20, R* rpy_rates, R* pid_state,
                                                   int32_t* counter, cudaStream_t st);
template <typename R> cudaError_t launch_set_state(const StepArgs<R>& a, const R* state20, const R* rpy_rates,
                                                   const R* pid_state, const int32_t* counter, cudaStream_t st);
template <typename R> cudaError_t launch_pid(const DevPid<R>& c, int64_t n, R dt, const R* cur_pos, const R* cur_quat,
                                             const R* cur_vel, const R* target_pos, const R* target_rpy,
                                             const R* target_vel, const R* target_rates, R* pid_state, R* rpm_out,
                                             R* pos_e_out, R* yaw_e_out, cudaStream_t st);
template <typename R> cudaError_t launch_ground_effect(const DevDrone<R>& d, int64_t n, const R* rpm, const R* pos,
                                                       const R* quat, R* out, uint8_t* applied, cudaStream_t st);
template <typename R> cudaError_t launch_drag(const DevDrone<R>& d, int64_t n, const R* rpm, const R* quat,
                                              const R* vel, R* out, cudaStream_t st);
template <typename R> cudaError_t launch_downwash(const DevDrone<R>& d, int64_t E, int N, const R* pos, R* out,
                                                  cudaStream_t st);
template <typename R> cudaError_t launch_adjacency(const StepArgs<R>& a, R radius, R* out, cudaStream_t st);
cudaError_t launch_state_sync(const StepArgs<float>& a, const float* obs_latest, int64_t tiles, cudaStream_t st);
template <typename R> cudaError_t launch_nonfinite(const StepArgs<R>& a, unsigned long long* out, cudaStream_t st);
template <typename R> cudaError_t launch_rollout_pid(const StepArgs<R>& a, int n_steps, const R* waypoints, int n_wp,
                                                     int32_t* wp_counters, R* action, cudaStream_t st);
// gpd_rollout: n_steps control steps of StepArgs::actions ([n_steps][D][A]) in one launch; traj as in include/gpd.h
template <typename R> cudaError_t launch_rollout(const StepArgs<R>& a, int n_steps, void* traj, const LaunchCfg& lc, cudaStream_t st);
// gpd_plan: n_steps control steps of q.n_samples copies of every env (StepArgs::actions [n_steps][E][S][N][A]), handle untouched
template <typename R> cudaError_t launch_plan(const StepArgs<R>& a, const PlanArgs<R>& q, int n_steps, const LaunchCfg& lc,
                                              cudaStream_t st);
// gpd_plan_grad: gpd_plan's returns of a LEAN configuration and their gradient with respect to the actions (q.grad)
template <typename R> cudaError_t launch_plan_grad(const StepArgs<R>& a, const PlanGradArgs<R>& q, int n_steps,
                                                   const LaunchCfg& lc, cudaStream_t st);

}  // namespace gpd
