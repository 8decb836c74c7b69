// gpd_rollout.cuh — open-loop rollouts: K control steps of a caller-given action schedule in one launch (gpd_rollout).
//
// Equivalent to K gpd::step_kernel launches on actions[k], each reading the previous one's observation, but nothing of the
// intermediate observations is written: the RL observation of step k is (kin of step k, ring of actions[k-B+1..k]), and the
// ring is a pure function of the schedule and of obs_prev, so it is composed once at the end.  One thread per drone with the
// block decomposition of the step kernel (whole envs per CTA: downwash snapshots and the MultiHover reductions stay in shared
// memory, Smem<R>); integrator state, rates, ang_v, the previous RPM (drag), the step counter, the episode return and the
// DSLPID state stay in registers for all K steps.  Per env-step the kernel moves the action row, reward and flags (and,
// when asked for, the traj / terminal_kin rows): it is bound by arithmetic and latency, not by HBM.
// The per-step arithmetic is gpd::step_kernel's (same device functions, same order of operations): bit-identical to K steps
// in FP64; in FP32 the two may differ in the compiler's FMA contraction.
#pragma once

#include "gpd_kernels.cuh"

namespace gpd {

// registers: FP32 lean <= 80 (6 CTAs of 128 threads), DSLPID / force models <= 128; multi-drone <= 128 (FP64 as gpd::step_kernel:
// C3's 512 CTAs of 128 threads then fit one wave; a CTA runs all K steps, so a partly filled second wave costs K steps);
// FP64 single-drone as gpd::step_kernel
template <typename R, int KIND, bool MULTI, bool VEC>
__global__ void __launch_bounds__(MULTI ? 256 : 128, MULTI ? 2 : (sizeof(R) == 4 ? (KIND == GPD_K_LEAN ? 6 : 4) : GPD_F64_SINGLE_MINB))
rollout_kernel(const __grid_constant__ StepArgs<R> a, int K, void* __restrict__ traj)
{
    constexpr bool LEAN = KIND == GPD_K_LEAN, HAS_PID = KIND == GPD_K_PID;
    constexpr bool EARLY_CONST = !M<R>::is_double;
    extern __shared__ __align__(16) unsigned char rollout_smem[];
    const bool ctrl = a.env_kind == GPD_ENV_CTRL;
    Smem<R> sm{ rollout_smem, a.DPB, a.EPB, false, MULTI };
    const int t = threadIdx.x;
    const int nphys = (int)blockDim.x;
    const int bid = (int)blockIdx.x;
    const int64_t row0 = (int64_t)bid * a.DPB;
    const int64_t d = row0 + t;
    const bool active = t < a.DPB && d < a.D;
    const int le = MULTI ? t / a.N : t;          // local env
    const int i = MULTI ? t - le * a.N : 0;      // drone index in env
    const int64_t e = MULTI ? (int64_t)bid * a.EPB + le : d;
    const bool lead = active && i == 0;          // owns the env's reward, flags and statistics
    const DevDrone<R>& P = a.drone;
    const int64_t D = a.D;

    State<R> s;
    s.px = s.py = s.pz = s.qx = s.qy = s.qz = R(0); s.qw = R(1);
    s.vx = s.vy = s.vz = s.wx = s.wy = s.wz = R(0);
    R st[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) st[k] = R(0);
    R rpm_prev[4] = { R(0), R(0), R(0), R(0) };
    int32_t cnt = 0;
    float ep = 0.f;
    V4<R> tg = M<R>::make4(R(0), R(0), R(0), R(0));
    // the action row of step k: RL actions are float32 (exact in R), Ctrl actions R
    auto load_act = [&](int k) {
        V4<R> v = M<R>::make4(R(0), R(0), R(0), R(0));
        if (ctrl) {
            v = reinterpret_cast<const V4<R>*>(a.actions)[(int64_t)k * D + d];
        } else if constexpr (VEC) {
            const float4 f = __ldg(reinterpret_cast<const float4*>(a.actions) + (int64_t)k * D + d);
            v = M<R>::make4((R)f.x, (R)f.y, (R)f.z, (R)f.w);
        } else {
            const float* ap = reinterpret_cast<const float*>(a.actions) + ((int64_t)k * D + d) * a.A;
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
            for (int k = 0; k < 9; ++k) st[k] = a.p.pid[(int64_t)k * D + d];
        }
        if constexpr (!LEAN) {
            if (a.phy & GPD_PHY_DRAG) {
                V4<R> v = a.p.aux_rpm[d];
                rpm_prev[0] = v.x; rpm_prev[1] = v.y; rpm_prev[2] = v.z; rpm_prev[3] = v.w;
            }
        }
        if constexpr (EARLY_CONST) {
            if (!ctrl) tg = a.p.target[a.target_per_env ? d : (int64_t)i];
        }
        cnt = a.p.counter[e];
        if (a.auto_reset) ep = a.p.ep_ret[e];
        nx = load_act(0);
    }
    // per-thread episode-statistics partials over all K steps (lead threads only), combined into the CTA's slot at the end
    double st_s1 = 0., st_s2 = 0.;
    int st_n = 0, st_len = 0, st_nt = 0, st_mn = 0x7fffffff, st_mx = (int)0x80000000;

    R roll = R(0), pitch = R(0), yaw = R(0), avx = R(0), avy = R(0), avz = R(0);
    R out_rpm[4] = { R(0), R(0), R(0), R(0) };
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
        const V4<R> cur = nx;
        if (active && k + 1 < K) nx = load_act(k + 1);       // in flight under this step's physics
        const float act[4] = { (float)cur.x, (float)cur.y, (float)cur.z, (float)cur.w };

        // ---- _preprocessAction -> rpm (BaseRLAviary.py:189-238, CtrlAviary.py:140, VelocityAviary.py:129-170) ----
        double rpm[4] = { 0., 0., 0., 0. };
        if (a.action_type == GPD_ACT_CTRL_RPM) {
            rpm[0] = clip(cur.x, R(0), P.MAX_RPM); rpm[1] = clip(cur.y, R(0), P.MAX_RPM);
            rpm[2] = clip(cur.z, R(0), P.MAX_RPM); rpm[3] = clip(cur.w, R(0), P.MAX_RPM);
        } else if (a.action_type == GPD_ACT_RPM) {
#pragma unroll
            for (int j = 0; j < 4; ++j) rpm[j] = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[j]));
        } else if (a.action_type == GPD_ACT_ONE_D_RPM) {
            const double v = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[0]));
            rpm[0] = rpm[1] = rpm[2] = rpm[3] = v;
        }
        if constexpr (HAS_PID) {
            if (active) {
                R r4[4] = { R(0), R(0), R(0), R(0) };
                if (a.action_type == GPD_ACT_CTRL_VEL) {             // as gpd::step_kernel, in the action's own precision
                    R n = M<R>::sqrt(cur.x * cur.x + cur.y * cur.y + cur.z * cur.z);
                    R u0 = R(0), u1 = R(0), u2 = R(0);
                    if (n != R(0)) { u0 = cur.x / n; u1 = cur.y / n; u2 = cur.z / n; }
                    const R sp = a.speed_limit * M<R>::abs(cur.w);
                    const R tv[3] = { sp * u0, sp * u1, sp * u2 }, tp[3] = { s.px, s.py, s.pz }, z3[3] = { R(0), R(0), R(0) };
                    R ro, pi, ya, pe[3], ye;
                    quat_to_euler(s.qx, s.qy, s.qz, s.qw, ro, pi, ya);
                    const R trpy[3] = { R(0), R(0), ya };
                    pid_compute(a.pid, a.ctrl_dt, s.px, s.py, s.pz, s.qx, s.qy, s.qz, s.qw, s.vx, s.vy, s.vz, tp, trpy, tv, z3,
                                st, r4, pe, ye);
                } else {
                    pid_action_st(a, s, act, st, r4);
                }
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

        // ---- _updateAndStoreKinematicInformation (BaseAviary.py:374,509-519), reward and flags ----
        quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
        R rew = R(-1);                  // CtrlAviary.py:144-200: dummy reward/flags
        int term = 0, trunc = 0;
        if (!ctrl) {
            if constexpr (!EARLY_CONST) {
                if (active) tg = a.p.target[a.target_per_env ? d : (int64_t)i];
            }
            R ex = tg.x - s.px, ey = tg.y - s.py, ez = tg.z - s.pz;
            R dist = M<R>::sqrt(ex * ex + ey * ey + ez * ez);
            R d2 = dist * dist;
            R v = R(2) - d2 * d2;       // HoverAviary.py:78 / MultiHoverAviary.py:87
            R r_i = v > R(0) ? v : R(0);
            const R lim = a.env_kind == GPD_ENV_HOVER ? R(1.5) : R(2.0);       // HoverAviary.py:111 / MultiHoverAviary.py:124
            int tr_i = (M<R>::abs(s.px) > lim || M<R>::abs(s.py) > lim || s.pz > R(2.0) ||
                        M<R>::abs(roll) > R(.4) || M<R>::abs(pitch) > R(.4)) ? 1 : 0;
            if constexpr (MULTI) {      // in-order sums over the env's drones (MultiHoverAviary.py:86-88,103-105)
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
            if (!ctrl && cnt > a.max_counter) trunc = 1;   // HoverAviary.py:114 (counter BEFORE the increment)
            const int64_t o = (int64_t)k * a.E + e;
            if (a.reward) a.reward[o] = rew;
            if (a.terminated) a.terminated[o] = (uint8_t)term;
            if (a.truncated) a.truncated[o] = (uint8_t)trunc;
        }
        int done = 0;
        if (a.auto_reset) {
            done = term | trunc;
            if constexpr (MULTI) {
                int* envf = sm.envf();
                phys_sync(nphys);
                if (lead) envf[le] = done;
                phys_sync(nphys);
                done = active ? envf[le] : 0;
            }
            if (lead) {                 // Monitor-style episode statistics, as gpd::step_kernel
                const float er = ep + (float)rew;
                if (done) {
                    ++st_n; st_s1 += (double)er; st_s2 += (double)(er * er);
                    st_len += cnt / a.S + 1; st_nt += term;
                    st_mn = min(st_mn, float_to_ordered(er)); st_mx = max(st_mx, float_to_ordered(er));
                }
                ep = done ? 0.f : er;
            }
        }

        float kin[12];
        kin[0] = (float)s.px; kin[1] = (float)s.py; kin[2] = (float)s.pz;
        kin[3] = (float)roll; kin[4] = (float)pitch; kin[5] = (float)yaw;
        kin[6] = (float)s.vx; kin[7] = (float)s.vy; kin[8] = (float)s.vz;
        kin[9] = (float)avx; kin[10] = (float)avy; kin[11] = (float)avz;
        out_rpm[0] = rpm_r[0]; out_rpm[1] = rpm_r[1]; out_rpm[2] = rpm_r[2]; out_rpm[3] = rpm_r[3];
        if (done && active) {
            if (a.terminal_kin && !ctrl) {
                float4* tk = reinterpret_cast<float4*>(a.terminal_kin) + ((int64_t)k * D + d) * 3;
                tk[0] = make_float4(kin[0], kin[1], kin[2], kin[3]);
                tk[1] = make_float4(kin[4], kin[5], kin[6], kin[7]);
                tk[2] = make_float4(kin[8], kin[9], kin[10], kin[11]);
            }
            init_state(a, d, i, s);     // BaseAviary.reset -> _housekeeping (BaseAviary.py:451-491)
            quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
            avx = avy = avz = R(0);
            out_rpm[0] = out_rpm[1] = out_rpm[2] = out_rpm[3] = R(0);       // last_clipped_action zeroed, :468
            kin[0] = (float)s.px; kin[1] = (float)s.py; kin[2] = (float)s.pz;
            kin[3] = (float)roll; kin[4] = (float)pitch; kin[5] = (float)yaw;
#pragma unroll
            for (int j = 6; j < 12; ++j) kin[j] = 0.f;
        }
        cnt = done ? 0 : cnt + a.S;    // BaseAviary.py:382
        if constexpr (!LEAN) {
#pragma unroll
            for (int j = 0; j < 4; ++j) rpm_prev[j] = out_rpm[j];          // _drag of the next step: last_clipped_action
        }
        if (traj && active) {           // what gpd_step writes into the observation row
            if (ctrl) {
                R* r = reinterpret_cast<R*>(traj) + ((int64_t)k * D + d) * 20;
                r[0] = s.px; r[1] = s.py; r[2] = s.pz; r[3] = s.qx; r[4] = s.qy; r[5] = s.qz; r[6] = s.qw;
                r[7] = roll; r[8] = pitch; r[9] = yaw; r[10] = s.vx; r[11] = s.vy; r[12] = s.vz;
                r[13] = avx; r[14] = avy; r[15] = avz; r[16] = out_rpm[0]; r[17] = out_rpm[1]; r[18] = out_rpm[2]; r[19] = out_rpm[3];
            } else {
                float4* r = reinterpret_cast<float4*>(traj) + ((int64_t)k * D + d) * 3;
                r[0] = make_float4(kin[0], kin[1], kin[2], kin[3]);
                r[1] = make_float4(kin[4], kin[5], kin[6], kin[7]);
                r[2] = make_float4(kin[8], kin[9], kin[10], kin[11]);
            }
        }
    }

    // ---- state, counters and the final observation ----
    if (active) {
        store_state(a.p, d, s);
        if constexpr (HAS_PID) {
#pragma unroll
            for (int k = 0; k < 9; ++k) a.p.pid[(int64_t)k * D + d] = st[k];
        }
        if (!(LEAN && a.skip_aux)) {    // lean FP32 KIN sims: both live in the observation row written below (derive_aux)
            a.p.aux_av[d] = M<R>::make4(avx, avy, avz, R(0));
            a.p.aux_rpm[d] = M<R>::make4(out_rpm[0], out_rpm[1], out_rpm[2], out_rpm[3]);
        } else if (d == 0) {
            *a.p.aux_auth = 0;
        }
        if (lead) {
            a.p.counter[e] = cnt;
            if (a.auto_reset) a.p.ep_ret[e] = ep;
        }
        if (ctrl) {                     // CtrlAviary.py:117: obs = state20 rows
            R* r = reinterpret_cast<R*>(a.obs_out) + d * 20;
            r[0] = s.px; r[1] = s.py; r[2] = s.pz; r[3] = s.qx; r[4] = s.qy; r[5] = s.qz; r[6] = s.qw;
            r[7] = roll; r[8] = pitch; r[9] = yaw; r[10] = s.vx; r[11] = s.vy; r[12] = s.vz;
            r[13] = avx; r[14] = avy; r[15] = avz; r[16] = out_rpm[0]; r[17] = out_rpm[1]; r[18] = out_rpm[2]; r[19] = out_rpm[3];
        } else {
            // KIN part of the last step, then the ring (BaseRLAviary.py:187,317-318): slot j (0 = oldest) holds actions[K-B+j]
            // or, for K-B+j < 0, slot j+K of the old ring (zeros without a previous observation).  It survives auto-reset.
            float* row = reinterpret_cast<float*>(a.obs_out) + d * a.W;
            const float* prev = a.obs_prev ? a.obs_prev + d * a.W + 12 : nullptr;
            const float* acts = reinterpret_cast<const float*>(a.actions);
            const int B = a.B, A = a.A;
            if constexpr (VEC) {
                float4* r4 = reinterpret_cast<float4*>(row);
                r4[0] = make_float4((float)s.px, (float)s.py, (float)s.pz, (float)roll);
                r4[1] = make_float4((float)pitch, (float)yaw, (float)s.vx, (float)s.vy);
                r4[2] = make_float4((float)s.vz, (float)avx, (float)avy, (float)avz);
                const float4* prev4 = reinterpret_cast<const float4*>(prev);
                for (int j = 0; j < B; ++j) {
                    const int ks = K - B + j;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ks >= 0) v = __ldg(reinterpret_cast<const float4*>(acts) + (int64_t)ks * D + d);
                    else if (prev4) v = __ldg(prev4 + j + K);
                    r4[3 + j] = v;
                }
            } else {
                const float kin[12] = { (float)s.px, (float)s.py, (float)s.pz, (float)roll, (float)pitch, (float)yaw,
                                        (float)s.vx, (float)s.vy, (float)s.vz, (float)avx, (float)avy, (float)avz };
#pragma unroll
                for (int j = 0; j < 12; ++j) row[j] = kin[j];
                for (int j = 0; j < B; ++j) {
                    const int ks = K - B + j;
                    for (int c = 0; c < A; ++c) {
                        float v = 0.f;
                        if (ks >= 0) v = __ldg(acts + ((int64_t)ks * D + d) * A + c);
                        else if (prev) v = __ldg(prev + (j + K) * A + c);
                        row[12 + j * A + c] = v;
                    }
                }
            }
        }
    }

    if (a.auto_reset) {                 // every warp's partials, reduced once, RED into this CTA's slot
        const unsigned FULL = 0xffffffffu;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            st_s1 += __shfl_xor_sync(FULL, st_s1, off);
            st_s2 += __shfl_xor_sync(FULL, st_s2, off);
        }
        const int n = __reduce_add_sync(FULL, st_n), len = __reduce_add_sync(FULL, st_len), nt = __reduce_add_sync(FULL, st_nt);
        const int mn = __reduce_min_sync(FULL, st_mn), mx = __reduce_max_sync(FULL, st_mx);
        StatSlot* slot = a.p.stat_slots + bid;
        if ((t & 31) == 0 && n > 0) {
            atomicAdd(&slot->s[0], (double)n);
            atomicAdd(&slot->s[1], st_s1);
            atomicAdd(&slot->s[2], (double)len);
            atomicAdd(&slot->s[3], st_s2);
            atomicMin(&slot->mn, mn);
            atomicMax(&slot->mx, mx);
            if (nt > 0) atomicAdd(&slot->s[5], (double)nt);
        }
        if (t == 0) {
            const int64_t envs = MULTI ? min((int64_t)a.EPB, a.E - (int64_t)bid * a.EPB) : min((int64_t)a.DPB, a.D - row0);
            atomicAdd(&slot->s[4], (double)K * (double)envs);
        }
    }
}

}  // namespace gpd
