// gpd_plan_grad.cuh — planning gradients (gpd_plan_grad): gpd_plan's returns of S candidate schedules per env together with
// the gradient of each return with respect to its schedule, by reverse-mode differentiation in the same launch.
//
// Forward: plan_kernel's LEAN forward (gpd_plan.cuh), the same device calls in the same order, so returns and done_step are
// gpd_plan's; each copy drone also stores its state at the start of every control step to the tape.  Backward, per copy
// drone and without block barriers (Physics.DYN couples no drones, and the flags and the end step are constants of the
// derivative): the adjoint (p, q, v, w) runs from k = min(done_step, K-1) down to 0.  At step k it adds the reward's
// position gradient, recomputes the step's substeps from the tape (their (q, w) held in a local array of GPD_PG_CAP
// entries, longer steps in segments recomputed from the checkpoint), back-propagates through them in reverse, and maps the
// accumulated thrust and torque adjoints through make_forcing and the RPM map onto the action row.  The adjoint is formed
// with the full-form derivatives of dyn_substep / integrate_q in both precisions; the lean FP32 regrouping is a forward
// optimisation only.
#pragma once

#include "gpd_plan.cuh"

namespace gpd {

enum { GPD_PG_CAP = 16 };           // substep states held per segment (FP64: 16 x 7 x 8 B of local memory per thread)
enum { GPD_PG_TAPE = 13 };          // Reals per copy drone and control step: p, q, v, w

template <typename R>
struct Adj {
    R px, py, pz, qx, qy, qz, qw, vx, vy, vz, wx, wy, wz;
};

// Adjoint of one DYN substep (dyn_substep without force models, integrate_q's smooth update).  (x, y, z, w) and (p, q, r)
// are the substep's input quaternion and rates, T the total thrust; b holds the adjoint of the substep's output on entry
// and of its input on return; Tb / tb accumulate the thrust and torque adjoints.
template <typename R>
__device__ __forceinline__ void adj_substep(const DevDrone<R>& P, R dt, R T, const R (&tau)[3], R x, R y, R z, R w, R p,
                                            R q, R r, Adj<R>& b, R& Tb, R (&tb)[3])
{
    // the rates after the substep: w' = w + dt J^-1 (tau - w x Jw)  (:852-854,858)
    const R Jx = P.J[0], Jy = P.J[1], Jz = P.J[2];
    const R gx = (Jz - Jy) * q * r, gy = (Jx - Jz) * r * p, gz = (Jy - Jx) * p * q;
    const R p1 = p + dt * P.JINV[0] * (tau[0] - gx), q1 = q + dt * P.JINV[1] * (tau[1] - gy), r1 = r + dt * P.JINV[2] * (tau[2] - gz);

    // q' = Phi(w') q with Phi = cos(theta) I + (sin(theta)/|w'|) Lambda(w'), theta = |w'| dt/2 (:860, :876-889)
    const R h = dt * R(.5);
    const R t = (p1 * p1 + q1 * q1 + r1 * r1) * (h * h);     // theta^2
    R cs, sc, dcs, dsc;                                        // cos, sin(theta)/|w'|, and their derivatives in t
    if (t < R(0.01)) {
        cs = R(1) + t * (R(-1. / 2) + t * (R(1. / 24) + t * (R(-1. / 720) + t * R(1. / 40320))));
        dcs = R(-1. / 2) + t * (R(2. / 24) + t * (R(-3. / 720) + t * R(4. / 40320)));
        sc = h * (R(1) + t * (R(-1. / 6) + t * (R(1. / 120) + t * (R(-1. / 5040) + t * R(1. / 362880)))));
        dsc = h * (R(-1. / 6) + t * (R(2. / 120) + t * (R(-3. / 5040) + t * R(4. / 362880))));
    } else {
        const R th = M<R>::sqrt(t);
        R sn;
        M<R>::sincos(th, &sn, &cs);
        sc = h * sn / th;
        dcs = -sn / (R(2) * th);
        dsc = h * (th * cs - sn) / (R(2) * t * th);
    }
    const R ap = sc * p1, aq = sc * q1, ar = sc * r1;
    const R bx = b.qx, by = b.qy, bz = b.qz, bw = b.qw;
    const R cb = x * bx + y * by + z * bz + w * bw;
    const R apb = w * bx + z * by - y * bz - x * bw;
    const R aqb = -z * bx + w * by + x * bz - y * bw;
    const R arb = y * bx - x * by + w * bz - z * bw;
    b.qx = cs * bx - ar * by + aq * bz - ap * bw;
    b.qy = ar * bx + cs * by - ap * bz - aq * bw;
    b.qz = -aq * bx + ap * by + cs * bz - ar * bw;
    b.qw = ap * bx + aq * by + ar * bz + cs * bw;
    const R kt = R(2) * (h * h) * (dcs * cb + dsc * (apb * p1 + aqb * q1 + arb * r1));
    R wbx = b.wx + sc * apb + kt * p1, wby = b.wy + sc * aqb + kt * q1, wbz = b.wz + sc * arb + kt * r1;

    // p' = p + dt v'; v' = v + dt F / M  (:857,859)
    const R vb0 = b.vx + dt * b.px, vb1 = b.vy + dt * b.py, vb2 = b.vz + dt * b.pz;
    b.vx = vb0; b.vy = vb1; b.vz = vb2;
    const R fs = dt / P.M;
    const R Fx = fs * vb0, Fy = fs * vb1, Fz = fs * vb2;

    // w' = w + dt J^-1 (tau - w x Jw)
    const R ux = dt * P.JINV[0] * wbx, uy = dt * P.JINV[1] * wby, uz = dt * P.JINV[2] * wbz;
    tb[0] += ux; tb[1] += uy; tb[2] += uz;
    b.wx = wbx - (uy * (Jx - Jz) * r + uz * (Jy - Jx) * q);
    b.wy = wby - (ux * (Jz - Jy) * r + uz * (Jy - Jx) * p);
    b.wz = wbz - (ux * (Jz - Jy) * q + uy * (Jx - Jz) * p);

    // F = R(q)[:,2] T - (0, 0, G), R(q) the unnormalised quat_to_mat: s = 2/|q|^2, column 2 = s (xz + wy, yz - wx, -(xx + yy)) + e_z
    const R d = x * x + y * y + z * z + w * w;
    const R s = R(2) / d;
    const R A = x * z + w * y, B = y * z - w * x, C = x * x + y * y;
    Tb += s * (A * Fx + B * Fy - C * Fz) + Fz;
    const R u2 = T * Fx, u5 = T * Fy, u8 = T * Fz;             // adjoints of R02, R12, R22
    const R sb = u2 * A + u5 * B - u8 * C;
    const R s2 = s * s * sb;
    b.qx += s * (u2 * z - u5 * w - R(2) * u8 * x) - s2 * x;
    b.qy += s * (u2 * w + u5 * z - R(2) * u8 * y) - s2 * y;
    b.qz += s * (u2 * x + u5 * y) - s2 * z;
    b.qw += s * (u2 * y - u5 * x) - s2 * w;
}

template <typename R, bool MULTI, bool VEC>
__global__ void __launch_bounds__(MULTI ? 256 : 128)
plan_grad_kernel(const __grid_constant__ StepArgs<R> a, const __grid_constant__ PlanGradArgs<R> q, int K)
{
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
    // _preprocessAction (BaseRLAviary.py:189-238) and the rotor terms of step k
    auto forcing = [&](const V4<R>& cur, double (&rpm)[4], Forcing<R>& F) {
        const float act[4] = { (float)cur.x, (float)cur.y, (float)cur.z, (float)cur.w };
        if (a.action_type == GPD_ACT_RPM) {
#pragma unroll
            for (int j = 0; j < 4; ++j) rpm[j] = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[j]));
        } else {
            const double v = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[0]));
            rpm[0] = rpm[1] = rpm[2] = rpm[3] = v;
        }
        make_forcing(P, rpm, F);
    };
    // the tape: state j of copy drone vd at the start of step k at [(k * 13 + j) * D + vd]
    auto tape_at = [&](int k, int j) -> R& { return q.tape[((int64_t)k * GPD_PG_TAPE + j) * q.D + vd]; };
    V4<R> nx = M<R>::make4(R(0), R(0), R(0), R(0));
    if (active) {
        load_state(a.p, d, s);
        if constexpr (EARLY_CONST) tg = load_target();
        cnt = a.p.counter[e];
        nx = load_act(0);
    }
    // the discounted return, rounded in R operation by operation (include/gpd.h)
    R G = R(0), w = R(1);
    const R gamma = q.gamma;
    int done_k = K;
    const R rpm_zero[4] = { R(0), R(0), R(0), R(0) };

    // ---- forward: plan_kernel's LEAN step, and the step-start states to the tape ----
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
        const V4<R> cur = nx;
        if (active && k + 1 < K) nx = load_act(k + 1);       // in flight under this step's physics
        if (active) {
            const R x13[GPD_PG_TAPE] = { s.px, s.py, s.pz, s.qx, s.qy, s.qz, s.qw, s.vx, s.vy, s.vz, s.wx, s.wy, s.wz };
#pragma unroll
            for (int j = 0; j < GPD_PG_TAPE; ++j) tape_at(k, j) = x13[j];
        }
        double rpm[4];
        Forcing<R> F;
        forcing(cur, rpm, F);

        // ---- PYB_STEPS_PER_CTRL substeps (BaseAviary.py:343-372) ----
        R avx = R(0), avy = R(0), avz = R(0);
        int sub0 = 0;
        if constexpr (!M<R>::is_double) {
            LeanStep c;
            c.kt2 = (2.f * P.DT_INV_M) * F.Ttot; c.ktmg = P.DT_INV_M * F.T;
            c.cx = P.DT_JINV[0] * F.tx; c.cy = P.DT_JINV[1] * F.ty; c.cz = P.DT_JINV[2] * F.tz;
            c.ex = P.DT_EULER[0]; c.ey = P.DT_EULER[1]; c.ez = P.DT_EULER[2];
            c.h = a.dt * .5f; c.hh = c.h * c.h;
            for (; sub0 < a.S - 1; ++sub0) lean_substep_f32(a.dt, s, c);
        }
        for (int sub = sub0; sub < a.S - 1; ++sub)
            step_substep<R, GPD_K_LEAN, MULTI>(a, s, F, rpm_zero, R(0), false, avx, avy, avz, nullptr, le, nphys, t, active);
        step_substep<R, GPD_K_LEAN, MULTI>(a, s, F, rpm_zero, R(0), true, avx, avy, avz, nullptr, le, nphys, t, active);

        // ---- reward and flags (HoverAviary.py:68-117, MultiHoverAviary.py:84-130) ----
        R roll, pitch, yaw;
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
            const bool ended = done_k < K;
            if (!ended) G = add_rn(G, mul_rn(w, rew));
            if (!ended && (term | trunc)) done_k = k;
            else if (!ended) w = mul_rn(w, gamma);
        }
        cnt += a.S;                     // BaseAviary.py:382; no auto-reset
    }

    if (lead) {
        q.returns[ve] = G;
        if (q.done_step) q.done_step[ve] = done_k;
    }
    if constexpr (MULTI) {              // the copy's end step to all its drones
        int* envf = sm.envf();
        phys_sync(nphys);
        if (lead) envf[le] = done_k;
        phys_sync(nphys);
        if (active) done_k = envf[le];
    }
    if (!active) return;

    // ---- backward ----
    const int kend = done_k < K ? done_k : K - 1;
    R* g = q.grad + (int64_t)vd * a.A;
    const int64_t gstride = q.D * a.A;
    for (int k = K - 1; k > kend; --k)
        for (int j = 0; j < a.A; ++j) g[k * gstride + j] = R(0);
    Adj<R> b;
    b.px = b.py = b.pz = b.qx = b.qy = b.qz = b.qw = b.vx = b.vy = b.vz = b.wx = b.wy = b.wz = R(0);
    R qw_[GPD_PG_CAP][7];               // (q, w) at the start of each substep of the current segment
#pragma unroll 1
    for (int k = kend; k >= 0; --k) {
        double rpm[4];
        Forcing<R> F;
        forcing(load_act(k), rpm, F);
        LeanStep c{};
        if constexpr (!M<R>::is_double) {
            c.kt2 = (2.f * P.DT_INV_M) * F.Ttot; c.ktmg = P.DT_INV_M * F.T;
            c.cx = P.DT_JINV[0] * F.tx; c.cy = P.DT_JINV[1] * F.ty; c.cz = P.DT_JINV[2] * F.tz;
            c.ex = P.DT_EULER[0]; c.ey = P.DT_EULER[1]; c.ez = P.DT_EULER[2];
            c.h = a.dt * .5f; c.hh = c.h * c.h;
        }
        // substep sub of step k, as the forward ran it
        auto fwd = [&](State<R>& x, int sub) {
            R avx, avy, avz;
            if constexpr (!M<R>::is_double) {
                if (sub < a.S - 1) { lean_substep_f32(a.dt, x, c); return; }
            }
            step_substep<R, GPD_K_LEAN, MULTI>(a, x, F, rpm_zero, R(0), sub == a.S - 1, avx, avy, avz, nullptr, le, nphys, t, true);
        };
        auto load_x = [&](State<R>& x) {
            x.px = tape_at(k, 0); x.py = tape_at(k, 1); x.pz = tape_at(k, 2);
            x.qx = tape_at(k, 3); x.qy = tape_at(k, 4); x.qz = tape_at(k, 5); x.qw = tape_at(k, 6);
            x.vx = tape_at(k, 7); x.vy = tape_at(k, 8); x.vz = tape_at(k, 9);
            x.wx = tape_at(k, 10); x.wy = tape_at(k, 11); x.wz = tape_at(k, 12);
        };
        const int nseg = (a.S + GPD_PG_CAP - 1) / GPD_PG_CAP;
        R Tb = R(0), tb[3] = { R(0), R(0), R(0) };
        const R tau[3] = { F.tx, F.ty, F.tz };
#pragma unroll 1
        for (int sg = nseg - 1; sg >= 0; --sg) {
            const int s0 = sg * GPD_PG_CAP, s1 = min(a.S, s0 + GPD_PG_CAP);
            State<R> x;
            load_x(x);
#pragma unroll 1
            for (int sub = 0; sub < s0; ++sub) fwd(x, sub);
#pragma unroll 1
            for (int sub = s0; sub < s1; ++sub) {
                R* r = qw_[sub - s0];
                r[0] = x.qx; r[1] = x.qy; r[2] = x.qz; r[3] = x.qw; r[4] = x.wx; r[5] = x.wy; r[6] = x.wz;
                fwd(x, sub);
            }
            if (sg == nseg - 1) {       // the reward of step k: r = v > 0 ? v : 0 with v = 2 - |e|^4, e = target - p
                const R ex = tg.x - x.px, ey = tg.y - x.py, ez = tg.z - x.pz;
                const R dist = M<R>::sqrt(ex * ex + ey * ey + ez * ez);
                const R d2 = dist * dist;
                if (R(2) - d2 * d2 > R(0)) {
                    const R wk = (R)pow((double)gamma, (double)k);
                    const R c4 = wk * R(4) * (ex * ex + ey * ey + ez * ez);
                    b.px += c4 * ex; b.py += c4 * ey; b.pz += c4 * ez;
                }
            }
#pragma unroll 1
            for (int sub = s1 - 1; sub >= s0; --sub) {
                const R* r = qw_[sub - s0];
                adj_substep<R>(P, a.dt, F.Ttot, tau, r[0], r[1], r[2], r[3], r[4], r[5], r[6], b, Tb, tb);
            }
        }
        // make_forcing (:838-851) and the RPM map rpm = HOVER_RPM (1 + 0.05 a) (BaseRLAviary.py:212-229)
        const double Tbd = Tb, txb = tb[0], tyb = tb[1], tzb = tb[2];
        double fb[4];
        if (P.model == GPD_CF2P) {
            fb[0] = Tbd - tyb * P.L_d; fb[1] = Tbd + txb * P.L_d; fb[2] = Tbd + tyb * P.L_d; fb[3] = Tbd - txb * P.L_d;
        } else {
            fb[0] = Tbd + (txb - tyb) * P.ARM_d; fb[1] = Tbd + (txb + tyb) * P.ARM_d;
            fb[2] = Tbd + (-txb + tyb) * P.ARM_d; fb[3] = Tbd + (-txb - tyb) * P.ARM_d;
        }
        const double km = P.model == GPD_RACE ? -P.KM_d : P.KM_d;
        const double da = P.HOVER_RPM_d * (double)0.05f;
        double ab[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double zs = (j & 1) ? tzb : -tzb;
            ab[j] = 2.0 * rpm[j] * (P.KF_d * fb[j] + km * zs) * da;
        }
        R* gk = g + k * gstride;
        if (a.action_type == GPD_ACT_RPM) {
#pragma unroll
            for (int j = 0; j < 4; ++j) gk[j] = (R)ab[j];
        } else {
            gk[0] = (R)(ab[0] + ab[1] + ab[2] + ab[3]);
        }
    }
}

}  // namespace gpd
