// gpd_plan.cuh — planning rollouts (gpd_plan): S candidate action schedules per env, each run for K control steps on a copy
// of the env, scored by its discounted return.  The handle is not modified.
//
// Copy (e, s) of drone i is the virtual drone (e*S + s)*N + i.  It starts from the state the next gpd_step of env e would
// start from (integrator state, previous RPM, DSLPID state, step counter, target) and runs K steps of actions[k][e][s] with no
// auto-reset.  The S threads of one env read the same state rows (L1 / L2 broadcasts).  Block decomposition, per-step
// arithmetic and operation order are rollout_kernel's (gpd_rollout.cuh), with the copies in place of the envs: whole copies
// per CTA, so the downwash snapshots and the MultiHover in-order reductions in shared memory (Smem<R>) work unchanged.  So a
// copy is bit-identical in FP64 to a handle of E*S envs holding the repeated state, stepped K times by gpd_step.
// The per-step blocks are stated here rather than shared with rollout_kernel: moving them into __forceinline__ functions
// changes rollout_kernel's register allocation.  Everything a copy carries stays in registers for all K steps; per
// sample-step the kernel reads one action row and optionally writes one reward.
#pragma once

#include "gpd_kernels.cuh"

namespace gpd {

__device__ __forceinline__ float mul_rn(float x, float y) { return __fmul_rn(x, y); }
__device__ __forceinline__ float add_rn(float x, float y) { return __fadd_rn(x, y); }
__device__ __forceinline__ double mul_rn(double x, double y) { return __dmul_rn(x, y); }
__device__ __forceinline__ double add_rn(double x, double y) { return __dadd_rn(x, y); }

// same register budgets as rollout_kernel
template <typename R, int KIND, bool MULTI, bool VEC>
__global__ void __launch_bounds__(MULTI ? 256 : 128, MULTI ? 2 : (sizeof(R) == 4 ? (KIND == GPD_K_LEAN ? 6 : 4) : GPD_F64_SINGLE_MINB))
plan_kernel(const __grid_constant__ StepArgs<R> a, const __grid_constant__ PlanArgs<R> q, int K)
{
    constexpr bool LEAN = KIND == GPD_K_LEAN, HAS_PID = KIND == GPD_K_PID;
    constexpr bool EARLY_CONST = !M<R>::is_double;
    extern __shared__ __align__(16) unsigned char plan_smem[];
    Smem<R> sm{ plan_smem, a.DPB, a.EPB, false, MULTI };
    const int t = threadIdx.x;
    const int nphys = (int)blockDim.x;
    const int bid = (int)blockIdx.x;
    const int64_t vd = (int64_t)bid * a.DPB + t;   // virtual drone (e*S + s)*N + i
    const bool active = t < a.DPB && vd < q.D;
    const int le = MULTI ? t / a.N : t;            // local copy
    const int i = MULTI ? t - le * a.N : 0;        // drone index in env
    const int64_t ve = MULTI ? (int64_t)bid * a.EPB + le : vd;     // copy e*S + s
    const int64_t e = ve / q.n_samples;            // source env
    const int64_t d = e * a.N + i;                 // source drone
    const bool lead = active && i == 0;            // owns the copy's reward, flags and return
    const DevDrone<R>& P = a.drone;

    State<R> s;
    s.px = s.py = s.pz = s.qx = s.qy = s.qz = R(0); s.qw = R(1);
    s.vx = s.vy = s.vz = s.wx = s.wy = s.wz = R(0);
    R st[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) st[k] = R(0);
    R rpm_prev[4] = { R(0), R(0), R(0), R(0) };
    int32_t cnt = 0;
    V4<R> tg = M<R>::make4(R(0), R(0), R(0), R(0));
    auto load_target = [&]() {
        if (q.targets) {
            const R* p = q.targets + d * 3;
            return M<R>::make4(p[0], p[1], p[2], R(0));
        }
        return a.p.target[a.target_per_env ? d : (int64_t)i];
    };
    // the action row of step k (float32, exact in R)
    auto load_act = [&](int k) {
        V4<R> v = M<R>::make4(R(0), R(0), R(0), R(0));
        if constexpr (VEC) {
            const float4 f = __ldg(reinterpret_cast<const float4*>(a.actions) + (int64_t)k * q.D + vd);
            v = M<R>::make4((R)f.x, (R)f.y, (R)f.z, (R)f.w);
        } else {
            const float* ap = reinterpret_cast<const float*>(a.actions) + ((int64_t)k * q.D + vd) * a.A;
            v.x = (R)__ldg(ap);
            if (a.A > 1) v.y = (R)__ldg(ap + 1);
            if (a.A > 2) v.z = (R)__ldg(ap + 2);
            if (a.A > 3) v.w = (R)__ldg(ap + 3);
        }
        return v;
    };
    V4<R> nx = M<R>::make4(R(0), R(0), R(0), R(0));
    if (active) {
        load_state(a.p, d, s);
        if constexpr (HAS_PID) {
#pragma unroll
            for (int k = 0; k < 9; ++k) st[k] = a.p.pid[(int64_t)k * a.D + d];
        }
        if constexpr (!LEAN) {
            if (a.phy & GPD_PHY_DRAG) {
                V4<R> v = a.p.aux_rpm[d];
                rpm_prev[0] = v.x; rpm_prev[1] = v.y; rpm_prev[2] = v.z; rpm_prev[3] = v.w;
            }
        }
        if constexpr (EARLY_CONST) tg = load_target();
        cnt = a.p.counter[e];
        nx = load_act(0);
    }
    // the discounted return, rounded in R operation by operation (include/gpd.h)
    R G = R(0), w = R(1);
    const R gamma = q.gamma;
    int done_k = K;

    R roll = R(0), pitch = R(0), yaw = R(0), avx = R(0), avy = R(0), avz = R(0);
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
        const V4<R> cur = nx;
        if (active && k + 1 < K) nx = load_act(k + 1);       // in flight under this step's physics
        const float act[4] = { (float)cur.x, (float)cur.y, (float)cur.z, (float)cur.w };

        // ---- _preprocessAction -> rpm (BaseRLAviary.py:189-238, VelocityAviary.py:129-170) ----
        double rpm[4] = { 0., 0., 0., 0. };
        if (a.action_type == GPD_ACT_RPM) {
#pragma unroll
            for (int j = 0; j < 4; ++j) rpm[j] = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[j]));
        } else if (a.action_type == GPD_ACT_ONE_D_RPM) {
            const double v = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[0]));
            rpm[0] = rpm[1] = rpm[2] = rpm[3] = v;
        }
        if constexpr (HAS_PID) {
            if (active) {
                R r4[4] = { R(0), R(0), R(0), R(0) };
                pid_action_st(a, s, act, st, r4);
                rpm[0] = r4[0]; rpm[1] = r4[1]; rpm[2] = r4[2]; rpm[3] = r4[3];
            }
        }
        Forcing<R> F;
        make_forcing(P, rpm, F);
        const R rpm_r[4] = { (R)rpm[0], (R)rpm[1], (R)rpm[2], (R)rpm[3] };

        // ---- PYB_STEPS_PER_CTRL substeps (BaseAviary.py:343-372) ----
        avx = avy = avz = R(0);
        R wsum_prev = R(0), wsum_cur = R(0);
        if constexpr (!LEAN) {
            if (a.phy & GPD_PHY_DRAG) { wsum_prev = drag_wsum(rpm_prev); wsum_cur = drag_wsum(rpm_r); }
        }
        int sub0 = 0;
        if constexpr (LEAN && !M<R>::is_double) {
            LeanStep c;
            c.kt2 = (2.f * P.DT_INV_M) * F.Ttot; c.ktmg = P.DT_INV_M * F.T;
            c.cx = P.DT_JINV[0] * F.tx; c.cy = P.DT_JINV[1] * F.ty; c.cz = P.DT_JINV[2] * F.tz;
            c.ex = P.DT_EULER[0]; c.ey = P.DT_EULER[1]; c.ez = P.DT_EULER[2];
            c.h = a.dt * .5f; c.hh = c.h * c.h;
            for (; sub0 < a.S - 1; ++sub0) lean_substep_f32(a.dt, s, c);
        }
        {
            V4<R>* snap = MULTI ? reinterpret_cast<V4<R>*>(sm.snap()) : nullptr;
            for (int sub = sub0; sub < a.S - 1; ++sub)
                step_substep<R, KIND, MULTI>(a, s, F, rpm_r, sub == 0 ? wsum_prev : wsum_cur, false, avx, avy, avz, snap, le, nphys, t, active);
            step_substep<R, KIND, MULTI>(a, s, F, rpm_r, a.S == 1 ? wsum_prev : wsum_cur, true, avx, avy, avz, snap, le, nphys, t, active);
        }

        // ---- reward and flags (HoverAviary.py:68-117, MultiHoverAviary.py:84-130) ----
        quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
        if constexpr (!EARLY_CONST) {
            if (active) tg = load_target();
        }
        R rew = R(0);
        int term = 0, trunc = 0;
        {
            R ex = tg.x - s.px, ey = tg.y - s.py, ez = tg.z - s.pz;
            R dist = M<R>::sqrt(ex * ex + ey * ey + ez * ez);
            R d2 = dist * dist;
            R v = R(2) - d2 * d2;       // HoverAviary.py:78 / MultiHoverAviary.py:87
            R r_i = v > R(0) ? v : R(0);
            const R lim = a.env_kind == GPD_ENV_HOVER ? R(1.5) : R(2.0);       // HoverAviary.py:111 / MultiHoverAviary.py:124
            int tr_i = (M<R>::abs(s.px) > lim || M<R>::abs(s.py) > lim || s.pz > R(2.0) ||
                        M<R>::abs(roll) > R(.4) || M<R>::abs(pitch) > R(.4)) ? 1 : 0;
            if constexpr (MULTI) {      // in-order sums over the copy's drones (MultiHoverAviary.py:86-88,103-105)
                R* red = sm.red();
                int* redi = sm.redi();
                phys_sync(nphys);
                if (t < a.DPB) { red[2 * t] = active ? r_i : R(0); red[2 * t + 1] = active ? dist : R(0); redi[t] = active ? tr_i : 0; }
                phys_sync(nphys);
                if (lead) {
                    R rs = R(0), ds = R(0);
                    int tr = 0;
                    for (int j = 0; j < a.N; ++j) { rs += red[2 * (t + j)]; ds += red[2 * (t + j) + 1]; tr |= redi[t + j]; }
                    rew = rs;
                    term = a.env_kind == GPD_ENV_HOVER ? (red[2 * t + 1] < R(.0001)) : (ds < R(.0001));
                    trunc = tr;
                }
            } else {
                rew = r_i; term = dist < R(.0001); trunc = tr_i;
            }
        }
        if (lead) {
            if (cnt > a.max_counter) trunc = 1;           // HoverAviary.py:114 (counter BEFORE the increment)
            if (q.reward) q.reward[(int64_t)k * q.E + ve] = rew;
            const bool ended = done_k < K;
            if (!ended) G = add_rn(G, mul_rn(w, rew));
            if (!ended && (term | trunc)) done_k = k;
            else if (!ended) w = mul_rn(w, gamma);
        }
        cnt += a.S;                     // BaseAviary.py:382; no auto-reset
        if constexpr (!LEAN) {
#pragma unroll
            for (int j = 0; j < 4; ++j) rpm_prev[j] = rpm_r[j];           // _drag of the next step: last_clipped_action
        }
    }

    if (lead) {
        q.returns[ve] = G;
        if (q.done_step) q.done_step[ve] = done_k;
    }
    if (q.final_kin && active) {        // the kin part gpd_step would write at step K-1
        float4* r = reinterpret_cast<float4*>(q.final_kin) + vd * 3;
        r[0] = make_float4((float)s.px, (float)s.py, (float)s.pz, (float)roll);
        r[1] = make_float4((float)pitch, (float)yaw, (float)s.vx, (float)s.vy);
        r[2] = make_float4((float)s.vz, (float)avx, (float)avy, (float)avz);
    }
}

}  // namespace gpd
