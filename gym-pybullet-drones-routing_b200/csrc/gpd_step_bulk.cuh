// gpd_step_bulk.cuh — the fused step kernel of the single-drone RL envs (HoverAviary with any ActionType: the BASELINE
// headline shape and the DSLPID-in-the-loop shape C5), with the observation tile moved by bulk asynchronous copies.
//
// Why a second data path (measured, profiles/stream_microbench.cu, 65,536 envs, 8 rotating sets, PDL): a plain streaming
// kernel moves this launch's bytes in 7.0 us; the step's own 14 address streams accessed per thread take 12.2 us; the same
// streams moved only by cp.async.bulk take 7.1 us.  The per-thread / TMA-box mix of gpd::step_kernel sits at 9.3 us.
//
// One tile = T = DPB envs, T threads per CTA, no DMA warp.  Thread 0 claims the tile (per-tile step sequencing, see
// gpd_kernels.cuh) and issues, on ONE mbarrier,
//     the observation tile   T rows x W floats, CONTIGUOUS in global memory, read from obs_prev at +A floats: in shared
//                            memory row r then holds [old kin[4..11] | old ring slots 1..B-1 | 16 stray bytes], i.e. the
//                            shifted ring already sits where the new row wants it (BaseRLAviary.py:187,317-318).  The
//                            chained-state variant (bulk_chain_variant) reads whole rows into shared memory 16 bytes in
//                            front of the tile instead: the same layout, the stray bytes being row r+1's old kin[0..3], so
//                            every row's whole old kin is in shared memory
//     (bulk_direct < 2)      the state tiles sP, sQ, sV (16/32 B per env); (bulk_direct == 0) sWz, step counter, episode
//                            return and the action tile too — by default (bulk_direct = 2) every thread fetches those itself
//                            and only the observation tile occupies shared memory (BulkSmem)
// A CTA runs one tile, or two one after the other through the same buffer in launches chained behind another handle
// (step_kernel_bulk below).
// Actions narrower than a float4 (ActionType.PID: A = 3, ONE_D_*: A = 1; rows still 16-byte granular): a bulk copy cannot
// shift by 12 bytes, so the tile is loaded UNSHIFTED and every thread slides its own row by A floats inside shared memory
// (aligned float4 reads, a register funnel, aligned float4 writes, in place and conflict-free: consecutive rows start 21 or
// 6 sixteen-byte units apart) — instead of one 32-lane warp funnelling the whole tile to global memory, which was the
// limiter of gpd::step_kernel on these shapes (C5: 11 % of the stall samples on its stores, 11 % on the barrier behind it).
// Every thread then integrates its drone exactly as gpd::step_kernel does (same device functions, same order of
// operations: bit-identical in FP64; in FP32 the two kernels may differ in the compiler's FMA contraction, which is why a
// handle never switches kernels between steps), patches its row (12 kin floats in front, this step's action in the newest
// slot) and writes its state / reward / flags (to global memory, or back into shared memory when staged); after one barrier
// thread 0 stores what is staged with bulk copies (the observation tile as ONE contiguous store: 18 KB per 64 envs).  Reading the full old rows costs 48 B per env more than
// the shifted slots alone (the DRAM atom is 64 B: 32 of them were being fetched anyway); in exchange every byte moves in
// long contiguous bursts.
#pragma once

#include "gpd_kernels.cuh"

namespace gpd {

__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 :: "l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// out = the float4 that starts A floats into (lo, hi)
template <int A>
__device__ __forceinline__ float4 funnel4(const float4& lo, const float4& hi)
{
    if (A == 1) return make_float4(lo.y, lo.z, lo.w, hi.x);
    if (A == 2) return make_float4(lo.z, lo.w, hi.x, hi.y);
    return make_float4(lo.w, hi.x, hi.y, hi.z);
}
// one row of the tile, in place: ring slots move up by A floats, the newest slot receives this step's action
template <int A>
__device__ __forceinline__ void slide_row(float4* r, int W4, const float* act)
{
    float4 lo = r[3];
#pragma unroll 4
    for (int k = 3; k < W4 - 1; ++k) {
        const float4 hi = r[k + 1];
        r[k] = funnel4<A>(lo, hi);
        lo = hi;
    }
    r[W4 - 1] = funnel4<A>(lo, make_float4(act[0], act[1], act[2], 0.f));
}

// shared-memory carve-up of one tile (every region starts 16-byte aligned because T % 16 == 0): `front` bytes (16 in the
// chained-state variant: row 0's old kin[0..3] when A == 4; 0 otherwise), then the observation tile.  `direct` (StepArgs::
// bulk_direct) says what does NOT go through shared memory — shared memory per env is what bounds the number of tiles
// in flight per SM, and with it the launch's throughput (tiles in flight / lifetime of a tile):
//     0  everything staged: 370 B per env (FP32, W = 72)                            9 tiles of 64 envs per SM
//     1  the small per-env arrays (action, rates.z, reward, counter, episode return, flags: 34 B) are read and written
//        by the drone's own thread: 336 B per env                                   10 tiles per SM
//     2  the state vectors sP / sQ / sV too: 288 B per env (the observation tile)    11 tiles per SM
template <typename R>
struct BulkSmem {
    unsigned char* base;
    int T, W, direct, front;
    __device__ float* obs() const { return reinterpret_cast<float*>(base + front); }
    __device__ V4<R>* sP() const { return reinterpret_cast<V4<R>*>(base + front + (size_t)T * W * 4); }
    __device__ V4<R>* sQ() const { return sP() + T; }
    __device__ V4<R>* sV() const { return sQ() + T; }
    __device__ unsigned char* after_state() const { return reinterpret_cast<unsigned char*>(sP() + (direct >= 2 ? 0 : 3 * T)); }
    // direct == 0 only:
    __device__ float4* act() const { return reinterpret_cast<float4*>(after_state()); }
    __device__ R* sWz() const { return reinterpret_cast<R*>(act() + T); }
    __device__ R* rew() const { return sWz() + T; }
    __device__ int32_t* cnt() const { return reinterpret_cast<int32_t*>(rew() + T); }
    __device__ float* ep() const { return reinterpret_cast<float*>(cnt() + T); }
    __device__ uint8_t* term() const { return reinterpret_cast<uint8_t*>(ep() + T); }
    __device__ uint8_t* trunc() const { return term() + T; }
    __device__ float* stat_f() const { return reinterpret_cast<float*>(direct ? after_state() : trunc() + T); }
    __device__ int* stat_i() const { return reinterpret_cast<int*>(stat_f() + 4 * 8); }      // up to 8 warps
    // multi-drone envs (direct == 2 only): per-drone reward terms and flags for the in-order per-env sums, one done flag per env
    __device__ R* red() const { return reinterpret_cast<R*>(stat_i() + 4 * 8); }             // [2 T]
    __device__ int* redi() const { return reinterpret_cast<int*>(red() + 2 * T); }           // [T]
    __device__ int* envf() const { return redi() + T; }                                      // [T / N]
};

// what a thread fetches itself before it waits for the tile (direct >= 1): issued right after the tile's dependency is
// resolved, so the latency runs under the bulk loads
template <typename R>
struct BulkPre {
    float4 act;
    R wz;
    int32_t cnt;
    float ep;
    V4<R> p4, q4, v4;       // direct == 2 (a tile in chained state: rates.x / rates.y from sR, xyz from the old kin in shared memory)
};

// The one kernel variant that takes StepArgs::state_in_obs (lean FP32 single-drone sims, direct == 2): it reads position and
// velocity of a tile in chained state from the old kin in shared memory and rates / episode return from sR (36 B of state per
// env-step each way instead of 60), writes sQ, sR and the counter only, and leaves the tile in chained state.
template <typename R, int KIND, bool MULTI>
__host__ __device__ constexpr bool bulk_chain_variant() { return KIND == GPD_K_LEAN && !MULTI && !M<R>::is_double; }

// One thread's share of a tile: state / action / counters from shared memory, the arithmetic of gpd::step_kernel, results
// back into the tile (plus the few per-drone extras that live only in global memory).  `sub` = timeline slot or -1.
template <typename R, int KIND, bool MULTI>
__device__ __forceinline__ void bulk_tile_physics(const StepArgs<R>& a, const BulkSmem<R>& sm, const BulkPre<R>& pre, int t,
                                                  int64_t row0, int rows, int tl)
{
    constexpr bool LEAN = KIND == GPD_K_LEAN, HAS_PID = KIND == GPD_K_PID;
    const bool chained = bulk_chain_variant<R, KIND, MULTI>() && a.state_in_obs;
    const DevDrone<R>& P = a.drone;
    const int64_t d = row0 + t;             // drone; tiles hold whole envs (T and row0 are multiples of N)
    const int le = MULTI ? t / a.N : t;     // env within the tile
    const int i = MULTI ? t - le * a.N : 0; // drone within its env
    const int64_t e = MULTI ? row0 / a.N + le : d;
    const bool active = t < rows;
    const bool full = rows == sm.T;
    // what does not come through shared memory: per-index constants and the optional per-drone extras
    V4<R> tg = M<R>::make4(R(0), R(0), R(0), R(0)), ip0 = tg, iq0 = tg;
    R rpm_prev[4] = { R(0), R(0), R(0), R(0) };
    const bool pre_init = a.auto_reset && !a.init_per_env;
    constexpr bool EARLY_CONST = !M<R>::is_double;      // FP64: fetched in the epilogue (register budget, see gpd::step_kernel)
    if (active) {
        if constexpr (EARLY_CONST) {
            tg = a.p.target[a.target_per_env ? d : (int64_t)i];
            if (pre_init) { ip0 = a.p.init_pos[i]; iq0 = a.p.init_quat[i]; }
        }
        if constexpr (!LEAN) {
            if (a.phy & GPD_PHY_DRAG) {
                V4<R> v = a.p.aux_rpm[d];
                rpm_prev[0] = v.x; rpm_prev[1] = v.y; rpm_prev[2] = v.z; rpm_prev[3] = v.w;
            }
        }
    }
    State<R> s;
    s.px = s.py = s.pz = s.qx = s.qy = s.qz = R(0); s.qw = R(1);
    s.vx = s.vy = s.vz = s.wx = s.wy = s.wz = R(0);
    float act[4] = { 0.f, 0.f, 0.f, 0.f };
    int32_t cnt = 0;
    float ep_ret0 = 0.f;
    const int direct = sm.direct;
    if (active) {
        const V4<R> p4 = direct >= 2 ? pre.p4 : sm.sP()[t], q4 = direct >= 2 ? pre.q4 : sm.sQ()[t], v4 = direct >= 2 ? pre.v4 : sm.sV()[t];
        s.px = p4.x; s.py = p4.y; s.pz = p4.z; s.wx = p4.w;
        s.qx = q4.x; s.qy = q4.y; s.qz = q4.z; s.qw = q4.w;
        s.vx = v4.x; s.vy = v4.y; s.vz = v4.z; s.wy = v4.w;
        s.wz = direct ? pre.wz : sm.sWz()[t];
        const float4 av = direct ? pre.act : sm.act()[t];
        act[0] = av.x; act[1] = av.y; act[2] = av.z; act[3] = av.w;
        cnt = direct ? pre.cnt : sm.cnt()[t];
        if (a.auto_reset) ep_ret0 = direct ? pre.ep : sm.ep()[t];
    }

    // ---- _preprocessAction -> rpm (BaseRLAviary.py:189-238) ----
    double rpm[4] = { 0., 0., 0., 0. };
    if (a.action_type == GPD_ACT_RPM) {
#pragma unroll
        for (int k = 0; k < 4; ++k) rpm[k] = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[k]));   // :192, float32 inner ops
    } else if (a.action_type == GPD_ACT_ONE_D_RPM) {
        const double v = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[0]));                       // :225
        rpm[0] = rpm[1] = rpm[2] = rpm[3] = v;
    }
    if constexpr (HAS_PID) {
        if ((a.action_type == GPD_ACT_VEL || a.action_type == GPD_ACT_PID || a.action_type == GPD_ACT_ONE_D_PID) && active) {
            R r4[4];
            pid_action(a, d, s, act, r4);
            rpm[0] = r4[0]; rpm[1] = r4[1]; rpm[2] = r4[2]; rpm[3] = r4[3];
        }
    }
    Forcing<R> F;
    make_forcing(P, rpm, F);
    const R rpm_r[4] = { (R)rpm[0], (R)rpm[1], (R)rpm[2], (R)rpm[3] };

    // ---- PYB_STEPS_PER_CTRL substeps (BaseAviary.py:343-372), state in registers ----
    R avx = R(0), avy = R(0), avz = R(0);
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
    for (int sub = sub0; sub < a.S - 1; ++sub)          // same device function as gpd::step_kernel (last substep peeled)
        step_substep<R, KIND, false>(a, s, F, rpm_r, sub == 0 ? wsum_prev : wsum_cur, false, avx, avy, avz, nullptr, 0, 0, t, active);
    step_substep<R, KIND, false>(a, s, F, rpm_r, a.S == 1 ? wsum_prev : wsum_cur, true, avx, avy, avz, nullptr, 0, 0, t, active);
    if (a.timeline && tl >= 0 && t == 0 && s.px == s.px) a.timeline[(int64_t)tl * 8 + 3] = gtime();

    // ---- _updateAndStoreKinematicInformation (BaseAviary.py:374,509-519) + outputs ----
    R roll, pitch, yaw;
    quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
    R rew;
    int term, trunc;
    if constexpr (!EARLY_CONST) {
        if (active) tg = a.p.target[a.target_per_env ? d : (int64_t)i];
    }
    {
        R ex = tg.x - s.px, ey = tg.y - s.py, ez = tg.z - s.pz;
        R dist = M<R>::sqrt(ex * ex + ey * ey + ez * ez);
        R d2 = dist * dist;
        R v = R(2) - d2 * d2;               // HoverAviary.py:78 / MultiHoverAviary.py:87
        const R r_i = v > R(0) ? v : R(0);
        const R lim = a.env_kind == GPD_ENV_HOVER ? R(1.5) : R(2.0);
        const int tr_i = (M<R>::abs(s.px) > lim || M<R>::abs(s.py) > lim || s.pz > R(2.0) ||
                          M<R>::abs(roll) > R(.4) || M<R>::abs(pitch) > R(.4)) ? 1 : 0;
        if constexpr (MULTI) {              // in-order sums over the env's drones (MultiHoverAviary.py:86-88,103-105), as gpd::step_kernel
            R* red = sm.red();
            int* redi = sm.redi();
            if (t < sm.T) { red[2 * t] = active ? r_i : R(0); red[2 * t + 1] = active ? dist : R(0); redi[t] = active ? tr_i : 0; }
            __syncthreads();
            rew = R(0); term = 0; trunc = 0;
            if (active && i == 0) {
                R rs = R(0), ds = R(0);
                int tr = 0;
                for (int j = 0; j < a.N; ++j) { rs += red[2 * (t + j)]; ds += red[2 * (t + j) + 1]; tr |= redi[t + j]; }
                rew = rs;
                term = a.env_kind == GPD_ENV_HOVER ? (red[2 * t + 1] < R(.0001)) : (ds < R(.0001));
                trunc = tr;
            }
        } else {
            rew = r_i; trunc = tr_i; term = dist < R(.0001);
        }
    }
    if (i == 0 && cnt > a.max_counter) trunc = 1;     // HoverAviary.py:114 (counter BEFORE the increment)
    int done = a.auto_reset ? (term | trunc) : 0;
    if constexpr (MULTI) {
        if (a.auto_reset) {                 // the env's flag to all of its drones
            int* envf = sm.envf();
            if (active && i == 0) envf[le] = done;
            __syncthreads();
            done = active ? envf[le] : 0;
        }
    }
    const bool lead = active && i == 0;     // the thread that owns the env's reward, flags, counter and episode statistics

    float kin[12];
    kin[0] = (float)s.px; kin[1] = (float)s.py; kin[2] = (float)s.pz;
    kin[3] = (float)roll; kin[4] = (float)pitch; kin[5] = (float)yaw;
    kin[6] = (float)s.vx; kin[7] = (float)s.vy; kin[8] = (float)s.vz;
    kin[9] = (float)avx; kin[10] = (float)avy; kin[11] = (float)avz;
    R out_rpm[4] = { rpm_r[0], rpm_r[1], rpm_r[2], rpm_r[3] };

    float ep_new = 0.f;
    if (a.auto_reset) {                     // Monitor-style episode statistics, as in gpd::step_kernel
        float er = ep_ret0 + (float)rew;
        int el = cnt / a.S + 1;
        const bool fin = lead && done;
        const unsigned m = __ballot_sync(0xffffffffu, fin);
        float s1 = 0.f, s2 = 0.f;
        int nl = 0, nt = 0, mn = 0x7fffffff, mx = (int)0x80000000;
        if (m) {
            s1 = fin ? er : 0.f; s2 = fin ? er * er : 0.f;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                s1 += __shfl_xor_sync(0xffffffffu, s1, off);
                s2 += __shfl_xor_sync(0xffffffffu, s2, off);
            }
            nl = __reduce_add_sync(0xffffffffu, fin ? el : 0);
            nt = __popc(__ballot_sync(0xffffffffu, fin && term));
            mn = __reduce_min_sync(0xffffffffu, fin ? float_to_ordered(er) : 0x7fffffff);
            mx = __reduce_max_sync(0xffffffffu, fin ? float_to_ordered(er) : (int)0x80000000);
        }
        if ((t & 31) == 0) {
            float* sf = sm.stat_f() + 4 * (t >> 5);
            int* si = sm.stat_i() + 4 * (t >> 5);
            sf[0] = s1; sf[1] = s2; sf[2] = (float)nt;
            si[0] = __popc(m); si[1] = nl; si[2] = mn; si[3] = mx;
        }
        ep_new = fin ? 0.f : er;
    }
    if (a.auto_reset && active && done) {
        if (a.terminal_kin) {
            float4* tk = reinterpret_cast<float4*>(a.terminal_kin) + d * 3;
            tk[0] = make_float4(kin[0], kin[1], kin[2], kin[3]);
            tk[1] = make_float4(kin[4], kin[5], kin[6], kin[7]);
            tk[2] = make_float4(kin[8], kin[9], kin[10], kin[11]);
        }
        if (pre_init) {                     // BaseAviary.reset -> _housekeeping (BaseAviary.py:451-491)
            if constexpr (!EARLY_CONST) { ip0 = a.p.init_pos[i]; iq0 = a.p.init_quat[i]; }
            s.px = ip0.x; s.py = ip0.y; s.pz = ip0.z;
            s.qx = iq0.x; s.qy = iq0.y; s.qz = iq0.z; s.qw = iq0.w;
            s.vx = s.vy = s.vz = R(0);
            s.wx = s.wy = s.wz = R(0);
        } else {
            init_state(a, d, i, s);
        }
        quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
        avx = avy = avz = R(0);
        out_rpm[0] = out_rpm[1] = out_rpm[2] = out_rpm[3] = R(0);
        kin[0] = (float)s.px; kin[1] = (float)s.py; kin[2] = (float)s.pz;
        kin[3] = (float)roll; kin[4] = (float)pitch; kin[5] = (float)yaw;
#pragma unroll
        for (int k = 6; k < 12; ++k) kin[k] = 0.f;
    }

    // ---- everything back into the tile ----
    if (active) {
        if (chained) {                      // position and velocity travel in the observation row written below
            a.p.sQ[d] = M<R>::make4(s.qx, s.qy, s.qz, s.qw);
            a.sR[d] = M<R>::make4(s.wx, s.wy, s.wz, (R)ep_new);
        } else if (direct >= 2) {
            a.p.sP[d] = M<R>::make4(s.px, s.py, s.pz, s.wx);
            a.p.sQ[d] = M<R>::make4(s.qx, s.qy, s.qz, s.qw);
            a.p.sV[d] = M<R>::make4(s.vx, s.vy, s.vz, s.wy);
        } else {
            sm.sP()[t] = M<R>::make4(s.px, s.py, s.pz, s.wx);
            sm.sQ()[t] = M<R>::make4(s.qx, s.qy, s.qz, s.qw);
            sm.sV()[t] = M<R>::make4(s.vx, s.vy, s.vz, s.wy);
        }
        const int32_t cnt_new = done ? 0 : cnt + a.S;                   // BaseAviary.py:382
        if (direct) {
            if (!chained) a.p.sWz[d] = s.wz;
            if (lead) {
                a.p.counter[e] = cnt_new;
                if (a.auto_reset && !chained) a.p.ep_ret[e] = ep_new;
            }
        } else {
            sm.sWz()[t] = s.wz;
            sm.cnt()[t] = cnt_new;
            if (a.auto_reset) sm.ep()[t] = ep_new;
        }
        float4* r = reinterpret_cast<float4*>(sm.obs() + (size_t)t * a.W);
        if (a.A == 4) r[(a.W >> 2) - 1] = make_float4(act[0], act[1], act[2], act[3]);   // newest ring slot, BaseRLAviary.py:187
        else if (a.A == 3) slide_row<3>(r, a.W >> 2, act);              // the tile was loaded unshifted: slide the ring here
        else if (a.A == 2) slide_row<2>(r, a.W >> 2, act);
        else slide_row<1>(r, a.W >> 2, act);
        r[0] = make_float4(kin[0], kin[1], kin[2], kin[3]);             // BaseRLAviary.py:310-316
        r[1] = make_float4(kin[4], kin[5], kin[6], kin[7]);
        r[2] = make_float4(kin[8], kin[9], kin[10], kin[11]);
        if (full && !direct && !a.out_plain) {
            sm.rew()[t] = rew; sm.term()[t] = (uint8_t)term; sm.trunc()[t] = (uint8_t)trunc;
        } else if (lead) {                  // direct mode, caller arrays that are not 16-byte aligned (e.g. rows of a [T][E] uint8 trajectory
                                            // buffer), or the ragged last tile (sizes are no multiples of 16 bytes): plain stores
            if (a.reward) a.reward[e] = rew;
            if (a.terminated) a.terminated[e] = (uint8_t)term;
            if (a.truncated) a.truncated[e] = (uint8_t)trunc;
        }
        if (!(LEAN && a.skip_aux)) {
            a.p.aux_av[d] = M<R>::make4(avx, avy, avz, R(0));
            a.p.aux_rpm[d] = M<R>::make4(out_rpm[0], out_rpm[1], out_rpm[2], out_rpm[3]);
        } else if (d == 0) {
            *a.p.aux_auth = 0;
        }
        if (a.kin_t) {                      // host mirror: feature-major copy of the kin part
#pragma unroll
            for (int k = 0; k < 12; ++k) a.kin_t[(int64_t)k * a.kin_ld + d] = kin[k];
        }
    }
}

// thread 0 of the physics group: combine the warps' statistics partials of one tile, RED into the tile's slot
template <typename R>
__device__ __forceinline__ void bulk_tile_stats(const StepArgs<R>& a, const BulkSmem<R>& sm, int64_t tile, int rows)
{
    const int T = sm.T;
    {
        if (a.auto_reset) {
            StatSlot* slot = a.p.stat_slots + tile;
            int n = 0, len = 0, mn = 0x7fffffff, mx = (int)0x80000000;
            float sr = 0.f, sr2 = 0.f, stt = 0.f;
            for (int w = 0; w < ((T + 31) >> 5); ++w) {
                const float* sf = sm.stat_f() + 4 * w;
                const int* si = sm.stat_i() + 4 * w;
                n += si[0]; len += si[1]; mn = min(mn, si[2]); mx = max(mx, si[3]);
                sr += sf[0]; sr2 += sf[1]; stt += sf[2];
            }
            if (n > 0) {
                atomicAdd(&slot->s[0], (double)n);
                atomicAdd(&slot->s[1], (double)sr);
                atomicAdd(&slot->s[2], (double)len);
                atomicAdd(&slot->s[3], (double)sr2);
                atomicMin(&slot->mn, mn);
                atomicMax(&slot->mx, mx);
                if (stt > 0.f) atomicAdd(&slot->s[5], (double)stt);
            }
            atomicAdd(&slot->s[4], (double)rows);
        }
    }
}

template <typename R, int KIND, bool MULTI>
// registers: FP32 lean 64 (8 CTAs of 128 threads), DSLPID 80 (72 spilled once the tile loop was added), force models 80; FP64 128 — shared memory (26-53 KB per tile)
// caps the FP64 variants at 512 threads per SM anyway, so they get the registers that would otherwise spill
__global__ void __launch_bounds__(128, sizeof(R) == 4 ? (KIND == GPD_K_LEAN ? 8 : (KIND == GPD_K_PID ? 6 : 5)) : 4)
step_kernel_bulk(const __grid_constant__ StepArgs<R> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t bar;
    const int t = threadIdx.x;
    const int T = a.DPB;
    const int direct = a.bulk_direct;
    constexpr bool CHAIN = bulk_chain_variant<R, KIND, MULTI>();
    BulkSmem<R> sm{ smem_raw, T, a.W, direct, CHAIN ? 16 : 0 };
    // Tiles of this CTA: one by default.  A chained launch (gpd_set_step_chaining) gives every CTA up to `tpc` tiles, strided by
    // the grid so that at any moment the CTAs cover a contiguous range: the tiles run one after the other through the SAME
    // shared-memory buffer, all claims are issued up front in one round trip, and a tile is published while the NEXT tile's
    // loads are in flight: its store drain and its release fence no longer hold the buffer idle (a buffer is busy from load
    // issue to store read, not from claim to publish), and a dependent step still sees each tile as soon as it is complete.
    const int tpc = a.tpc > 0 ? a.tpc : 1;
    const int tile_end = a.tile_end;        // first tile NOT covered by this launch
    const int tile0 = (int)blockIdx.x + a.cta0;

    if (a.timeline && t == 0) a.timeline[(int64_t)tile0 * 8 + 0] = gtime();
    if (t == 0) mbar_init(&bar, 1);
    unsigned long long claimed[GPD_BULK_MAX_TPC];
    if (a.tile_dep) {
        if (t == 0) {
            unsigned pend_any = 0;
#pragma unroll
            for (int it = 0; it < GPD_BULK_MAX_TPC; ++it) {
                claimed[it] = 0;
                const int tile = tile0 + it * (int)gridDim.x;
                if (it < tpc && tile < tile_end) claimed[it] = tile_claim(a.tile_seq + (int64_t)tile * 4);
            }
#pragma unroll
            for (int it = 0; it < GPD_BULK_MAX_TPC; ++it) pend_any |= (unsigned)claimed[it];     // every claim is performed
            if (pend_any) tile_wait(a.tile_seq + (int64_t)tile0 * 4, claimed[0]);               // the first tile's predecessors
        }
        __syncthreads();
        if (a.pdl_trigger_early) pdl_launch_dependents();
    } else {
        if (a.pdl_trigger_early) pdl_launch_dependents();
        __syncthreads();
        pdl_wait();
    }
    if (a.timeline && t == 0) a.timeline[(int64_t)tile0 * 8 + 1] = gtime();

#pragma unroll 1
    for (int it = 0; it < tpc; ++it) {
        const int bid = tile0 + it * (int)gridDim.x;
        if (bid >= tile_end) break;             // uniform over the CTA
        const int64_t row0 = (int64_t)bid * T;
        const int rows = (int)min((int64_t)T, a.D - row0);
        const bool full = rows == T;
        if (it > 0) {
            if (t == 0) {
                asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");      // the previous tile's stores have read the buffer
                if (a.tile_dep) {
#pragma unroll
                    for (int k = 1; k < GPD_BULK_MAX_TPC; ++k)
                        if (k == it && (unsigned)claimed[k]) tile_wait(a.tile_seq + (int64_t)bid * 4, claimed[k]);
                }
                if (a.timeline) { a.timeline[(int64_t)bid * 8 + 0] = gtime(); a.timeline[(int64_t)bid * 8 + 1] = gtime(); }
            }
            __syncthreads();                    // buffer free, this tile's previous step visible
        }

        // ---- loads: everything this tile needs, in flight at once ----
        if (t == 0) {
            fence_proxy_async_global();         // generic-proxy writes of the tile's previous step (ragged tails) -> bulk reads
            const uint32_t v4b = (uint32_t)sizeof(V4<R>);
            // A == 4: already shifted, i.e. read at +A floats (the last tile of the buffer must not read past its end: its final
            // row loses the 16 stray bytes) or, in the chained-state variant, whole rows landing 16 bytes in front of the tile.
            // A < 4: whole rows, unshifted (slide_row)
            const uint32_t shift = a.A == 4 && !CHAIN ? 4u : 0u;
            const uint32_t ob = a.obs_prev ? (uint32_t)rows * a.W * 4 - ((shift && row0 + rows >= a.D) ? 16u : 0u) : 0u;
            const uint32_t st = (uint32_t)rows * v4b, sc = (uint32_t)T * (uint32_t)sizeof(R), i4 = (uint32_t)T * 4u;
            const uint32_t total = ob + (direct >= 2 ? 0u : 3 * st) + (direct ? 0u : (uint32_t)rows * 16u + sc + i4 + (a.auto_reset ? i4 : 0u));
            mbar_expect_tx(&bar, total);
            if (ob) bulk_g2s(CHAIN && a.A == 4 ? sm.obs() - 4 : sm.obs(), a.obs_prev + row0 * a.W + shift, ob, &bar);
            if (direct < 2) {
                bulk_g2s(sm.sP(), a.p.sP + row0, st, &bar);
                bulk_g2s(sm.sQ(), a.p.sQ + row0, st, &bar);
                bulk_g2s(sm.sV(), a.p.sV + row0, st, &bar);
            }
            if (!direct) {
                bulk_g2s(sm.act(), reinterpret_cast<const float4*>(a.actions) + row0, (uint32_t)rows * 16u, &bar);
                bulk_g2s(sm.sWz(), a.p.sWz + row0, sc, &bar);              // library arrays are padded to whole tiles
                bulk_g2s(sm.cnt(), a.p.counter + row0, i4, &bar);
                if (a.auto_reset) bulk_g2s(sm.ep(), a.p.ep_ret + row0, i4, &bar);
            }
        }
        BulkPre<R> pre;
        pre.act = make_float4(0.f, 0.f, 0.f, 0.f); pre.wz = R(0); pre.cnt = 0; pre.ep = 0.f;
        pre.p4 = pre.q4 = pre.v4 = M<R>::make4(R(0), R(0), R(0), R(0));
        // this tile's state lives in the observation chain (set by its previous step, cleared by launch_state_sync; the
        // claim above acquired it together with the tile).  A step without obs_prev is preceded by a sync on the host.
        const bool from_obs = CHAIN && a.state_in_obs && a.obs_prev &&
                              a.tile_seq[(int64_t)bid * 4 + 1] != 0ull;
        if (direct && t < rows) {               // the thread's own small inputs: in flight under the bulk loads
            const int64_t d = row0 + t;
            if (a.A == 4) {
                pre.act = __ldg(reinterpret_cast<const float4*>(a.actions) + d);
            } else {
                const float* ap = reinterpret_cast<const float*>(a.actions) + d * a.A;
                pre.act.x = __ldg(ap);
                if (a.A > 1) pre.act.y = __ldg(ap + 1);
                if (a.A > 2) pre.act.z = __ldg(ap + 2);
            }
            if (!from_obs) pre.wz = a.p.sWz[d];
            const int64_t e = MULTI ? d / a.N : d;      // every drone of an env reads the env's counter / return (one address per env)
            pre.cnt = a.p.counter[e];
            if (from_obs) {
                const V4<R> r4 = a.sR[d];
                pre.q4 = a.p.sQ[d];
                pre.p4.w = r4.x; pre.v4.w = r4.y; pre.wz = r4.z; pre.ep = (float)r4.w;
            } else {
                if (a.auto_reset) pre.ep = a.p.ep_ret[e];
                if (direct >= 2) { pre.p4 = a.p.sP[d]; pre.q4 = a.p.sQ[d]; pre.v4 = a.p.sV[d]; }
            }
        }
        if (!a.obs_prev && t < rows) {          // no previous observation: all-zero ring (BaseRLAviary.py:153-154)
            float* r = sm.obs() + (size_t)t * a.W;
            for (int k = 12; k < a.W; ++k) r[k] = 0.f;
        }
        if (it > 0 && t == 0 && a.tile_dep) {   // the previous tile: its stores drain and its release fence runs under THIS tile's loads
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            const int prev = bid - (int)gridDim.x;
            tile_publish(a.tile_seq + (int64_t)prev * 4);
            if (a.timeline) a.timeline[(int64_t)prev * 8 + 7] = gtime();
        }
        mbar_wait(&bar, (uint32_t)(it & 1));
        if (a.timeline && t == 0) a.timeline[(int64_t)bid * 8 + 2] = gtime();
        if (from_obs) {
            if (t < rows) {                     // the old row starts 16 bytes in front of the new one when A == 4 (kin[0..3] at
                                                // the end of row t-1's slot), at it otherwise
                const float* k = sm.obs() + (size_t)t * a.W - (a.A == 4 ? 4 : 0);
                pre.p4.x = k[0]; pre.p4.y = k[1]; pre.p4.z = k[2];
                pre.v4.x = k[6]; pre.v4.y = k[7]; pre.v4.z = k[8];
            }
            if (a.A == 4) __syncthreads();      // row t-1's newest ring slot overwrites row t's old kin[0..3]
        }

        bulk_tile_physics<R, KIND, MULTI>(a, sm, pre, t, row0, rows, bid);
        fence_proxy_async_smem();               // this thread's shared-memory writes -> the bulk stores below
        __syncthreads();
        if (a.timeline && t == 0) a.timeline[(int64_t)bid * 8 + 4] = gtime();

        if (t == 0) {
            const uint32_t v4b = (uint32_t)sizeof(V4<R>);
            const uint32_t st = (uint32_t)rows * v4b, sc = (uint32_t)T * (uint32_t)sizeof(R), i4 = (uint32_t)T * 4u;
            bulk_s2g(reinterpret_cast<float*>(a.obs_out) + row0 * a.W, sm.obs(), (uint32_t)rows * a.W * 4);
            if (direct < 2) {
                bulk_s2g(a.p.sP + row0, sm.sP(), st);
                bulk_s2g(a.p.sQ + row0, sm.sQ(), st);
                bulk_s2g(a.p.sV + row0, sm.sV(), st);
            }
            if (!direct) {
                bulk_s2g(a.p.sWz + row0, sm.sWz(), sc);
                bulk_s2g(a.p.counter + row0, sm.cnt(), i4);
                if (a.auto_reset) bulk_s2g(a.p.ep_ret + row0, sm.ep(), i4);
            }
            if (full && !direct && !a.out_plain) {
                if (a.reward) bulk_s2g(a.reward + row0, sm.rew(), sc);
                if (a.terminated) bulk_s2g(a.terminated + row0, sm.term(), (uint32_t)T);
                if (a.truncated) bulk_s2g(a.truncated + row0, sm.trunc(), (uint32_t)T);
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            bulk_tile_stats<R>(a, sm, bid, MULTI ? rows / a.N : rows);
            // published with the tile: its next step reads position and velocity from this observation
            if (CHAIN && a.state_in_obs && !from_obs) a.tile_seq[(int64_t)bid * 4 + 1] = 1ull;
        }
    }

    if (t == 0) {
        if (a.tile_dep) {
            // Measured (profiles/r02/sweep_b6..b8.jsonl, unsafe experiments): waiting for the stores costs nothing; the claim
            // (ATOMG + L1 invalidate) ~0.5 us and the release fence below (MEMBAR.ALL.GPU) ~0.6 us of an 8.6 us one-tile step.  A
            // relaxed publish alone is not a release pattern: the next step of a tile could then read stale state.
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");     // the CTA's last tile is in global memory: publish it
            int last = tile0;
#pragma unroll 1
            for (int it = 1; it < tpc; ++it)
                if (tile0 + it * (int)gridDim.x < tile_end) last = tile0 + it * (int)gridDim.x;
            tile_publish(a.tile_seq + (int64_t)last * 4);
            if (a.timeline) a.timeline[(int64_t)last * 8 + 7] = gtime();
        } else {
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            if (a.timeline) a.timeline[(int64_t)tile0 * 8 + 7] = gtime();
        }
    }
    if (!a.pdl_trigger_early) pdl_launch_dependents();
    if (a.tile_dep) pdl_wait();             // keep stream order transitive (see gpd::step_kernel)
}


}  // namespace gpd
