// gpd_kernels.cuh — the fused step kernel and its helpers, templated on the compute type.
// Included by gpd_f32.cu (float, FMA on) and gpd_f64.cu (double, -fmad=false).
//
// One thread per drone; a block owns EPB whole envs (DPB = EPB*N consecutive drones), so the
// per-env reductions (MultiHover reward/termination, downwash) stay inside shared memory.
// The 13-float integrator state lives in registers across the whole PYB_STEPS_PER_CTRL loop.
// The RL observation IS the action ring (BaseRLAviary.py:317-318): its history part is a one-slot-shifted copy of the
// previous observation, moved by TMA tensor copies issued by a dedicated DMA warp (A = 4), by a TMA load plus a
// shared-memory funnel shift (A = 1..3 with 16-byte rows) or by a register copy (other shapes); each drone's own thread
// writes the 48-byte kinematic part and the newest ring slot.  The Ctrl observation (state20 rows) is staged in shared
// memory and written as one contiguous tile.
#pragma once

#include "gpd_math.cuh"

namespace gpd {

template <typename R> using V4 = typename Vec4<R>::type;

__device__ __forceinline__ float4 ldg_stream(const float4* p)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// Programmatic dependent launch (PDL): a step kernel launched with programmaticStreamSerialization may start while the
// previous kernel of the stream drains; pdl_wait() blocks until that kernel has completed and its writes are visible,
// so only the CTA launch, the constant-bank parameter fetch and the shared-memory set-up overlap. No-ops otherwise.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Per-CTA step sequencing (tile_dep): CTA i of step k+1 depends only on CTA i of step k (same rows, same DPB), so instead
// of the whole-grid griddepcontrol.wait it waits for its own tile's previous step.  The step kernel is launched with
// programmatic stream serialization and releases its dependents as soon as every CTA has CLAIMED its tile; a dependent
// grid therefore starts only after every CTA of every earlier step kernel of the stream has started (and claimed), which
// orders the claims and excludes deadlock: a spinning CTA only ever waits for a CTA that is already resident.
//
// One 64-bit word per tile, ONE L2 round trip at each end of a CTA's life:
//     high 32 bits = steps claimed so far (wraps harmlessly: it falls off the top of the word)
//     low  32 bits = steps claimed and not yet published (0 or 1 outside a transition, never more than the grids in flight)
// claim   = atom.acquire.add (1 << 32) + 1: the old word tells this CTA its sequence number and, in the common case
//           (pending == 0), that its predecessor has published — the acquire side makes the predecessor's tile visible;
// publish = red.release.add -1 (borrows nothing: pending >= 1 while this CTA is alive).
// A CTA that found predecessors pending polls until pending - 1 - (claims made after its own) == 0.
// claim: returns the old word (several claims may be in flight at once: nothing waits here)
__device__ __forceinline__ unsigned long long tile_claim(unsigned long long* w)
{
    unsigned long long old;
    // acquire only: a claiming CTA has written nothing yet (an acq_rel atomic would put MEMBAR.ALL.GPU + ERRBAR in front, ~1 us)
    asm volatile("atom.acquire.gpu.global.add.u64 %0, [%1], %2;" : "=l"(old) : "l"(w), "l"(0x100000001ull) : "memory");
    return old;
}
// wait until every step claimed before `old`'s claim has published
__device__ __forceinline__ void tile_wait(unsigned long long* w, unsigned long long old)
{
    if ((uint32_t)old == 0u) return;
    const uint32_t mine = (uint32_t)(old >> 32);
    for (;;) {
        unsigned long long cur;
        asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(cur) : "l"(w) : "memory");
        const uint32_t later = (uint32_t)(cur >> 32) - mine - 1u;      // claims made after this one
        if ((uint32_t)cur - 1u - later == 0u) break;
        __nanosleep(32);
    }
}
__device__ __forceinline__ void tile_claim_and_wait(unsigned long long* w) { tile_wait(w, tile_claim(w)); }
__device__ __forceinline__ void tile_publish(unsigned long long* w)
{
    asm volatile("red.release.gpu.global.add.u64 [%0], %1;" :: "l"(w), "l"(0xffffffffffffffffull) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_global() { asm volatile("fence.proxy.async.global;" ::: "memory"); }

__device__ __forceinline__ unsigned long long gtime()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Physics-only barrier (named barrier 1): the DMA/copy warp of the block never joins it.
__device__ __forceinline__ void phys_sync(int nthreads) { asm volatile("bar.sync 1, %0;" :: "r"(nthreads) : "memory"); }

// ---- TMA (cp.async.bulk.tensor) helpers: the action history of a block tile is one 2-D box [rows][(B-1)*16 bytes] ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok = 0;
    while (!ok)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 :: "r"(smem_u32(smem_dst)), "l"(tm), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, int c0, int c1, const void* smem_src)
{
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                 :: "l"(tm), "r"(c0), "r"(c1), "r"(smem_u32(smem_src)) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// the bulk store's global writes are complete (not only its shared-memory reads): needed before this CTA publishes its tile
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- shared-memory layout -------------------------------------------------------------
//   tile  : RL envs with A == 4: TMA box of the action history, DPB x (B-1) float4 (a.tma_bytes)
//   stage : Ctrl env R[DPB*20] (state20 rows)
//   MULTI : snap R[DPB*4] (x,y,z,-), red R[DPB*2], redi int[DPB], envf int[EPB*2]
//   stats : per physics warp float[4] + int[4] (plain stores, combined by thread 0 after the block barrier)
template <typename R>
struct Smem {
    unsigned char* base;     // dynamic shared memory + the TMA history tile (tma_bytes, 128-byte multiple) that precedes everything
    int DPB, EPB;
    bool ctrl, multi;
    __device__ float* stage_f() const { return reinterpret_cast<float*>(base); }
    __device__ R* stage_r() const { return reinterpret_cast<R*>(base); }
    __device__ size_t stage_bytes() const { return ctrl ? size_t(DPB) * 20 * sizeof(R) : 0; }
    __device__ R* snap() const { return reinterpret_cast<R*>(base + ((stage_bytes() + 15) & ~size_t(15))); }
    __device__ R* red() const { return snap() + (multi ? size_t(DPB) * 4 : 0); }
    __device__ int* redi() const { return reinterpret_cast<int*>(red() + (multi ? size_t(DPB) * 2 : 0)); }
    __device__ int* envf() const { return redi() + (multi ? DPB : 0); }
    __device__ float* stat_f() const { return reinterpret_cast<float*>(envf() + (multi ? 2 * EPB : 0)); }
    __device__ int* stat_i() const { return reinterpret_cast<int*>(stat_f() + 4 * 9); }     // up to 9 physics warps
};

__device__ __forceinline__ int float_to_ordered(float f)
{
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_to_float(int i)
{
    return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff);
}

// History write-out for A = 1..3 when the rows are still 16-byte granular (e.g. ActionType.PID at 48 Hz, W = 84): the whole
// old ring of the tile was TMA-loaded into shared memory (tile[row][A*B floats]); every aligned output float4 is funnelled
// from two aligned shared-memory float4s (shift by A floats), the last A floats of a row come from this step's action.
template <int A>
__device__ __forceinline__ void write_shifted_from_smem(const float4* __restrict__ tile, float* __restrict__ out,
                                                        const float* __restrict__ act, int64_t row0, int rows, int W, int B,
                                                        int ct, int CT)
{
    const int W4 = W >> 2, H4 = (A * B) >> 2, keep = A * (B - 1);
    const int ktail = keep >> 2;                      // first float4 of a row that holds a float of the new slot
    const float* actb = act + row0 * A;
    float4* out4 = reinterpret_cast<float4*>(out) + row0 * W4 + 3;
    // (row, k) advance by CT float4s per iteration without a division in the loop
    int row = ct / H4, k = ct - row * H4;
    const int dq = CT / H4, dr = CT - dq * H4;
    while (row < rows) {
        const float4* src = tile + row * H4 + k;
        const float4 lo = src[0];
        const float4 hi = (k + 1 < H4) ? src[1] : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 v;
        if (A == 1) v = make_float4(lo.y, lo.z, lo.w, hi.x);
        else if (A == 2) v = make_float4(lo.z, lo.w, hi.x, hi.y);
        else v = make_float4(lo.w, hi.x, hi.y, hi.z);
        if (k >= ktail) {
            const int c = 4 * k;
            const float* ar = actb + row * A;
            if (c + 0 >= keep) v.x = __ldg(ar + (c + 0 - keep));
            if (c + 1 >= keep) v.y = __ldg(ar + (c + 1 - keep));
            if (c + 2 >= keep) v.z = __ldg(ar + (c + 2 - keep));
            if (c + 3 >= keep) v.w = __ldg(ar + (c + 3 - keep));
        }
        out4[row * W4 + k] = v;
        k += dr; row += dq;
        if (k >= H4) { k -= H4; ++row; }
    }
}

// History part of the observation tile: out[row][12 + c] = prev[row][12 + c + A] (c < A*(B-1)),
// newest entry = this step's action (BaseRLAviary.py:187, deque(maxlen=B)).  shift = false for reset (ring survives).
// Executed by CT "copier" threads (index ct): either the whole block or, warp-specialised, its upper half.
// Element k of the tile maps to (row, c) = (k / Hc, k % Hc); a thread visits k = ct, ct+CT, ... so (row, c) advances
// by a fixed (CT / Hc, CT % Hc) with carry — no per-element division.
template <bool VEC>
__device__ __forceinline__ void copy_history(const float* __restrict__ prev, float* __restrict__ out,
                                             const float* __restrict__ act, int64_t row0, int rows, int W, int A, int B,
                                             bool shift, int ct, int CT)
{
    constexpr int U = 4;     // independent loads in flight per thread before the first store (memory-level parallelism)
    if constexpr (VEC) {     // A == 4: rows are whole float4s, the shift is one float4
        // 8 lanes walk one row (8 x 16 B = one 128-byte segment per pass over the columns); index math is one IMAD.
        const int W4 = W >> 2;
        const float4* prev4 = prev ? reinterpret_cast<const float4*>(prev) + row0 * W4 + 3 : nullptr;   // tile base
        const float4* act4 = reinterpret_cast<const float4*>(act) + row0;
        float4* out4 = reinterpret_cast<float4*>(out) + row0 * W4 + 3;
        const int lane_c = ct & 7, r0 = ct >> 3, RS = CT >> 3;      // CT is a multiple of 32
        const int src_shift = shift ? 1 : 0;
        for (int c = lane_c; c < B; c += 8) {
            const bool newest = shift && c == B - 1;
            for (int rb = r0; rb < rows; rb += RS * U) {
                float4 v[U];
#pragma unroll
                for (int j = 0; j < U; ++j) {
                    const int row = rb + j * RS;
                    v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (row < rows) {
                        if (newest) v[j] = __ldg(act4 + row);
                        else if (prev4) v[j] = ldg_stream(prev4 + row * W4 + c + src_shift);
                    }
                }
#pragma unroll
                for (int j = 0; j < U; ++j) {
                    const int row = rb + j * RS;
                    if (row < rows) out4[row * W4 + c] = v[j];
                }
            }
        }
    } else {
        const int H = A * B, keep = A * (B - 1);
        const float* prevb = prev ? prev + row0 * (int64_t)W + 12 : nullptr;
        const float* actb = act + row0 * A;
        float* outb = out + row0 * (int64_t)W + 12;
        const int total = rows * H;
        const int qs = CT / H, rs = CT - qs * H;
        int row = ct / H, c = ct - row * H;
        const int src_shift = shift ? A : 0;
        for (int base = ct; base < total; base += U * CT) {
            float v[U];
            int off[U];
#pragma unroll
            for (int j = 0; j < U; ++j) {
                off[j] = row * W + c;
                const bool ok = base + j * CT < total;
                v[j] = 0.f;
                if (ok) {
                    if (shift && c >= keep) v[j] = __ldg(actb + row * A + (c - keep));
                    else if (prevb) v[j] = __ldg(prevb + off[j] + src_shift);
                }
                c += rs; row += qs;
                if (c >= H) { c -= H; row += 1; }
            }
#pragma unroll
            for (int j = 0; j < U; ++j)
                if (base + j * CT < total) outb[off[j]] = v[j];
        }
    }
}

template <typename R>
__device__ __forceinline__ void load_state(const SimPtrs<R>& p, int64_t d, State<R>& s)
{
    V4<R> a = p.sP[d], q = p.sQ[d], v = p.sV[d];
    s.px = a.x; s.py = a.y; s.pz = a.z; s.wx = a.w;
    s.qx = q.x; s.qy = q.y; s.qz = q.z; s.qw = q.w;
    s.vx = v.x; s.vy = v.y; s.vz = v.z; s.wy = v.w;
    s.wz = p.sWz[d];
}

template <typename R>
__device__ __forceinline__ void store_state(const SimPtrs<R>& p, int64_t d, const State<R>& s)
{
    p.sP[d] = M<R>::make4(s.px, s.py, s.pz, s.wx);
    p.sQ[d] = M<R>::make4(s.qx, s.qy, s.qz, s.qw);
    p.sV[d] = M<R>::make4(s.vx, s.vy, s.vz, s.wy);
    p.sWz[d] = s.wz;
}

// Lean FP32 KIN sims: ang_v and last_clipped_action re-derived from an observation row (float32 kin[9..11]; newest ring
// slot through the action map of BaseRLAviary.py:192,225 — bit-identical to what the step computed; zero right after a
// reset, i.e. while the env's step counter is 0, BaseAviary.py:468).
template <typename R>
__device__ __forceinline__ void derive_aux(const StepArgs<R>& a, const float* __restrict__ obs, int64_t d, int64_t e,
                                           R av[3], R rpm[4])
{
    const float* row = obs + d * a.W;
    av[0] = (R)row[9]; av[1] = (R)row[10]; av[2] = (R)row[11];
    rpm[0] = rpm[1] = rpm[2] = rpm[3] = R(0);
    if (a.p.counter[e] != 0) {
        const float* act = row + a.W - a.A;
        if (a.action_type == GPD_ACT_RPM) {
#pragma unroll
            for (int k = 0; k < 4; ++k) rpm[k] = (R)(a.drone.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[k])));
        } else if (a.action_type == GPD_ACT_ONE_D_RPM) {
            rpm[0] = rpm[1] = rpm[2] = rpm[3] = (R)(a.drone.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[0])));
        }
    }
}

template <typename R>
__device__ __forceinline__ void init_state(const StepArgs<R>& a, int64_t d, int i, State<R>& s)
{
    int64_t k = a.init_per_env ? d : (int64_t)i;
    V4<R> ip = a.p.init_pos[k], iq = a.p.init_quat[k];
    s.px = ip.x; s.py = ip.y; s.pz = ip.z;
    s.qx = iq.x; s.qy = iq.y; s.qz = iq.z; s.qw = iq.w;
    s.vx = s.vy = s.vz = R(0);
    s.wx = s.wy = s.wz = R(0);
}

// _preprocessAction for the PID-family action types (BaseRLAviary.py:193-235), on the DSLPID state st[9] held by the caller.
template <typename R>
__device__ __forceinline__ void pid_action_st(const StepArgs<R>& a, const State<R>& s, const float* act, R (&st)[9], R rpm[4])
{
    R tp[3], trpy[3] = { R(0), R(0), R(0) }, tv[3] = { R(0), R(0), R(0) }, tr[3] = { R(0), R(0), R(0) }, pe[3], ye;
    if (a.action_type == GPD_ACT_PID) {
        // BaseAviary._calculateNextStep (BaseAviary.py:1105-1147), step_size = 1
        R dx = R(act[0]) - s.px, dy = R(act[1]) - s.py, dz = R(act[2]) - s.pz;
        R dist = M<R>::sqrt(dx * dx + dy * dy + dz * dz);
        if (dist <= R(1)) { tp[0] = R(act[0]); tp[1] = R(act[1]); tp[2] = R(act[2]); }
        else { tp[0] = s.px + dx / dist * R(1); tp[1] = s.py + dy / dist * R(1); tp[2] = s.pz + dz / dist * R(1); }
    } else if (a.action_type == GPD_ACT_VEL) {
        // BaseRLAviary.py:208-223; the unit vector and the speed are float32 expressions in the reference
        // np.linalg.norm(float32[3]) = sqrt(sdot(x, x)): float32 products, OpenBLAS accumulates the scalar tail in double and
        // rounds the sum to float32, then a float32 sqrt (checked bit for bit against numpy on 200,000 random vectors)
        const double sq = (double)__fmul_rn(act[0], act[0]) + (double)__fmul_rn(act[1], act[1]) + (double)__fmul_rn(act[2], act[2]);
        float n = __fsqrt_rn((float)sq);
        float u0 = 0.f, u1 = 0.f, u2 = 0.f;
        if (n != 0.f) { u0 = __fdiv_rn(act[0], n); u1 = __fdiv_rn(act[1], n); u2 = __fdiv_rn(act[2], n); }
        float sp = __fmul_rn((float)a.speed_limit, fabsf(act[3]));
        tv[0] = R(__fmul_rn(sp, u0)); tv[1] = R(__fmul_rn(sp, u1)); tv[2] = R(__fmul_rn(sp, u2));
        tp[0] = s.px; tp[1] = s.py; tp[2] = s.pz;
        R roll, pitch, yaw;
        quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
        trpy[2] = yaw;
    } else {  // GPD_ACT_ONE_D_PID, BaseRLAviary.py:226-235
        tp[0] = s.px + R(0.1) * R(0); tp[1] = s.py + R(0.1) * R(0); tp[2] = s.pz + R(0.1) * R(act[0]);
    }
    pid_compute(a.pid, a.ctrl_dt, s.px, s.py, s.pz, s.qx, s.qy, s.qz, s.qw, s.vx, s.vy, s.vz, tp, trpy, tv, tr, st, rpm, pe, ye);
}

// the same, with the DSLPID state of drone d read from and written back to a.p.pid
template <typename R>
__device__ __forceinline__ void pid_action(const StepArgs<R>& a, int64_t d, const State<R>& s, const float* act, R rpm[4])
{
    R st[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) st[k] = a.p.pid[(int64_t)k * a.D + d];
    pid_action_st(a, s, act, st, rpm);
#pragma unroll
    for (int k = 0; k < 9; ++k) a.p.pid[(int64_t)k * a.D + d] = st[k];
}

// One substep of the ctrl step's loop (BaseAviary.py:343-372): rotation matrix, the optional force models, _dynamics.
// `last` is a literal at both call sites (the final substep is peeled off the loop): only there ang_v = R_old·w_new
// (BaseAviary.py:870) is observable, so in the looped substeps the rotation matrix dies before _integrateQ — 18 registers
// less across the FP64 loop — and the three outputs are not carried through it.
//   snap / le / nphys / t / active : MULTI only (downwash against the substep-start snapshot in shared memory)
template <typename R, int KIND, bool MULTI>
__device__ __forceinline__ void step_substep(const StepArgs<R>& a, State<R>& s, const Forcing<R>& F, const R (&rpm_r)[4],
                                             R wsum, bool last, R& avx, R& avy, R& avz,
                                             V4<R>* snap, int le, int nphys, int t, bool active)
{
    const DevDrone<R>& P = a.drone;
    R m[9];
    const R omz = quat_to_mat(s.qx, s.qy, s.qz, s.qw, m);    // :836 (shared with the force models)
    if constexpr (KIND == GPD_K_LEAN) {
        dyn_substep<R>(P, a.dt, s, m, omz, F, nullptr, nullptr, last, avx, avy, avz);
    } else {
        R gnd[4], fb[3] = { R(0), R(0), R(0) };
        const R* pg = nullptr;
        const R* pb = nullptr;
        if (a.phy & GPD_PHY_GND) {
            // The gate |roll|,|pitch| < pi/2 of the rpy snapshot (BaseAviary.py:346-347,518,742) needs only the signs of
            // the atan2/asin arguments: |atan2(y,x)| < pi/2 <=> x > 0 (or x = y = 0); Bullet's gimbal branch
            // (|s| >= 0.99999) returns pitch = +-pi/2 and fails the gate, otherwise |asin(s)| < pi/2.  Exact in both
            // precisions except where atan2 ROUNDS to pi/2: for x > 0 the correctly rounded double atan2(y, x) = pi/2 - x/|y|
            // equals double(pi/2) once x/|y| <= (pi/2 - double(pi/2)) + 2^-53 = 1.7225e-16 (roll = +-pi/2 exactly, x a
            // rounding residue), and the reference's gate is then false; FP64 tests that bound.  Three libm calls per
            // substep saved.
            const R sarg = R(-2) * (s.qx * s.qz - s.qw * s.qy);
            const R rx = s.qw * s.qw - s.qx * s.qx - s.qy * s.qy + s.qz * s.qz, ry = R(2) * (s.qy * s.qz + s.qw * s.qx);
            const bool gimbal = sarg <= R(-0.99999) || sarg >= R(0.99999);
            const bool upright = M<R>::is_double ? (rx > R(0) && M<R>::abs(ry) * R(1.7225464241988331e-16) < rx) : rx > R(0);
            const R roll = gimbal ? R(0) : ((upright || (rx == R(0) && ry == R(0))) ? R(0) : R(GPD_PI));
            const R pitch = gimbal ? R(GPD_PI) : R(0);
            if (ground_effect(P, rpm_r, s.pz, m, roll, pitch, gnd)) pg = gnd;
        }
        if (a.phy & GPD_PHY_DRAG) {                          // :359,366: rpm = last_clipped_action
            R db[3];
            drag_body_w(P, wsum, m, s.vx, s.vy, s.vz, db);
            fb[0] += db[0]; fb[1] += db[1]; fb[2] += db[2];
            pb = fb;
        }
        if constexpr (MULTI) {
            if (a.phy & GPD_PHY_DW) {                        // :362,367 against the substep-start snapshot
                // FP32: x and y enter the snapshot pre-scaled (downwash_pair<R, true>): one multiply less in each of the N pairs
                constexpr bool SC = !M<R>::is_double;
                const R sx = SC ? s.px * R(GPD_DW_XY_SCALE) : s.px, sy = SC ? s.py * R(GPD_DW_XY_SCALE) : s.py;
                phys_sync(nphys);
                if (t < a.DPB) snap[t] = M<R>::make4(sx, sy, s.pz, R(0));   // (x, y, z, -): one 16/32-byte read per pair
                phys_sync(nphys);
                R dw = R(0);
                const V4<R>* env = snap + le * a.N;
                if (active) {
#pragma unroll 4
                    for (int j = 0; j < a.N; ++j) {
                        const V4<R> o = env[j];
                        dw += downwash_pair<R, SC>(P, sx, sy, s.pz, o.x, o.y, o.z);
                    }
                }
                fb[2] += dw;
                pb = fb;
            }
        }
        dyn_substep<R>(P, a.dt, s, m, omz, F, pg, pb, last, avx, avy, avz);
    }
}

// ============================================================================================
// The fused step kernel: BaseAviary.step (BaseAviary.py:259-383).
//   KIND  : which optional code the variant carries (each keeps its own register budget)
//             GPD_K_LEAN   plain Physics.DYN with an RPM-type action (no controller, no force models)
//             GPD_K_FORCES RPM-type action with ground effect / drag / downwash
//             GPD_K_PID    DSLPID in the loop (PID / VEL / ONE_D_PID / CTRL_VEL actions), force models optional
//   MULTI : N > 1 (per-env reductions / downwash need block-level exchange)
//   VEC   : A == 4 (observation rows are float4-granular)
// ============================================================================================
template <typename R, int KIND, bool MULTI, bool VEC>
// FP64: occupancy beats spill-free code.  Multi-drone: 128 registers (two 256-thread CTAs per SM) instead of 168 is 1.2-1.4x
// faster (C3, C4) and no longer spills since the last substep is peeled and the epilogue constants are fetched late;
// single-drone (the shapes the bulk kernel does not take): 96 registers (four 160-thread CTAs) with 70-380 bytes of spills
// stay 0-32 % faster than the spill-free 128-register build (GPD_F64_SINGLE_MINB=3; profiles/r02/f64_single_register_cap.jsonl:
// CtrlAviary x1 8.07 vs 9.13 us, ONE_D_RPM at 30 Hz 17.3 vs 22.9 us, PID at 30 Hz 41.4 vs 48.5 us); 80 registers lose again.
#ifndef GPD_F64_SINGLE_MINB
#define GPD_F64_SINGLE_MINB 4
#endif
__global__ void __launch_bounds__(MULTI ? (sizeof(R) == 8 ? 256 : 288) : 160, MULTI ? (sizeof(R) == 8 ? 2 : 1) : (sizeof(R) == 4 ? (KIND == GPD_K_LEAN ? 6 : (KIND == GPD_K_PID ? 5 : 4)) : GPD_F64_SINGLE_MINB))
step_kernel(const __grid_constant__ StepArgs<R> a, const __grid_constant__ CUtensorMap tm_prev,
            const __grid_constant__ CUtensorMap tm_out, const __grid_constant__ CUtensorMap tm_edge)
{
    constexpr bool LEAN = KIND == GPD_K_LEAN, HAS_PID = KIND == GPD_K_PID;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ uint64_t tma_bar;
    const bool ctrl = a.env_kind == GPD_ENV_CTRL;
    Smem<R> sm{ smem_raw + a.tma_bytes, a.DPB, a.EPB, ctrl, MULTI };
    const int t = threadIdx.x;
    const int bid = (int)blockIdx.x + a.cta0;     // a.cta0 is 0 (StepArgs)
    const int64_t row0 = (int64_t)bid * a.DPB;
    const int64_t d = row0 + t;
    const bool active = t < a.DPB && d < a.D;
    const int rows = (int)min((int64_t)a.DPB, a.D - row0);
    const int le = MULTI ? t / a.N : t;          // local env
    const int i = MULTI ? t - le * a.N : 0;      // drone index in env
    const int64_t e = MULTI ? (int64_t)bid * a.EPB + le : d;
    const DevDrone<R>& P = a.drone;
    // Warp specialisation (RL envs): the last `copy_threads` threads of the block (one warp) move the action history of
    // the tile — as two TMA tensor copies issued by one lane when the rows are float4-granular — while the other warps
    // integrate the physics.  The two roles never wait for each other except at the final block barrier.
    const int nphys = (int)blockDim.x - a.copy_threads;
    const bool spec = a.copy_threads > 0;
    const bool run_physics = t < nphys;

    if (a.timeline && t == 0) a.timeline[(int64_t)bid * 8 + 0] = gtime();      // 0: CTA start (params fetched)
    const bool tma_copy = spec && a.use_tma;
    const bool edge_smem = tma_copy && VEC && a.tma_edge;       // physics threads read the two edge slots from shared memory
    if (tma_copy && t == nphys) mbar_init(&tma_bar, 1);
    if (a.tile_dep) {
        if (t == 0) tile_claim_and_wait(a.tile_seq + (int64_t)bid * 4);
        __syncthreads();                // the claim is performed: dependents may start; the tile's previous step is visible
        if (a.pdl_trigger_early) pdl_launch_dependents();
    } else {
        if (a.pdl_trigger_early) pdl_launch_dependents();
        if (edge_smem) __syncthreads(); // the physics threads will wait on the mbarrier the DMA lane just initialised
        pdl_wait();                     // everything above touched only parameters and shared memory
    }
    if (a.timeline && t == 0) a.timeline[(int64_t)bid * 8 + 1] = gtime();      // 1: previous step of this tile complete

    if (!ctrl && !tma_copy)             // no TMA for this row shape (A = 3 or 1) or no previous observation: every thread
        copy_history<VEC>(a.obs_prev, reinterpret_cast<float*>(a.obs_out), reinterpret_cast<const float*>(a.actions),
                          row0, rows, a.W, a.A, a.B, true, t, (int)blockDim.x);   // of the block shares the register copy
    if (spec && !run_physics) {
        if (tma_copy && !VEC) {         // A = 1..3: TMA load of the whole old ring, shifted write-out by the 32 lanes
            if (t == nphys) {
                if (a.tile_dep) fence_proxy_async_global();
                mbar_expect_tx(&tma_bar, (uint32_t)a.tma_bytes_box);
                tma_load_2d(smem_raw, &tm_prev, 12, (int)row0, &tma_bar);
            }
            __syncwarp();
            mbar_wait(&tma_bar, 0);
            const float4* tile = reinterpret_cast<const float4*>(smem_raw);
            float* o = reinterpret_cast<float*>(a.obs_out);
            const float* ac = reinterpret_cast<const float*>(a.actions);
            if (a.A == 3) write_shifted_from_smem<3>(tile, o, ac, row0, rows, a.W, a.B, t - nphys, a.copy_threads);
            else if (a.A == 2) write_shifted_from_smem<2>(tile, o, ac, row0, rows, a.W, a.B, t - nphys, a.copy_threads);
            else write_shifted_from_smem<1>(tile, o, ac, row0, rows, a.W, a.B, t - nphys, a.copy_threads);
        } else if (tma_copy) {
            if (t == nphys) {           // one lane drives the TMA engine: global -> shared -> global, shifted by one slot
                // box = ring slots [edge, B-1-edge) of the new obs = slots [edge+1, B-edge) of the old one.  edge = 1 when the
                // rows are 32-byte aligned: the two sectors shared with the kin part / the newest slot are then written
                // whole by the drone's own thread (no partial-sector L2 fills from DRAM); the two old slots it needs
                // (1 and B-1) arrive through two more, 16-byte-wide TMA boxes on the same mbarrier.
                if (a.tile_dep) fence_proxy_async_global();     // generic-proxy writes of the tile's previous step -> TMA reads
                mbar_expect_tx(&tma_bar, (uint32_t)(a.tma_bytes_box + (a.tma_edge ? 2 * a.DPB * 16 : 0)));
                if (a.tma_edge) {
                    tma_load_2d(smem_raw + a.tma_bytes - 2 * a.tma_edge_bytes, &tm_edge, 16, (int)row0, &tma_bar);
                    tma_load_2d(smem_raw + a.tma_bytes - a.tma_edge_bytes, &tm_edge, a.W - 4, (int)row0, &tma_bar);
                }
                tma_load_2d(smem_raw, &tm_prev, 12 + 4 * (a.tma_edge + 1), (int)row0, &tma_bar);
                mbar_wait(&tma_bar, 0);
                if (a.timeline) a.timeline[(int64_t)bid * 8 + 5] = gtime();    // 5: history tile landed in smem
                tma_store_2d(&tm_out, 12 + 4 * a.tma_edge, (int)row0, smem_raw);
                if (a.timeline) a.timeline[(int64_t)bid * 8 + 6] = gtime();    // 6: TMA store has read smem
                if (a.tile_dep) tma_store_wait_all();
            }
        }
    }

    if (run_physics) {
    // ---- state and action loads first (their latency overlaps the history copy below) ----
    State<R> s;
    s.px = s.py = s.pz = s.qx = s.qy = s.qz = R(0); s.qw = R(1);
    s.vx = s.vy = s.vz = s.wx = s.wy = s.wz = R(0);
    double rpm[4] = { 0., 0., 0., 0. };
    float act[4] = { 0.f, 0.f, 0.f, 0.f };
    R rpm_prev[4] = { R(0), R(0), R(0), R(0) };
    int32_t cnt = 0;
    float ep_ret0 = 0.f;
    float4 edge_lo = make_float4(0.f, 0.f, 0.f, 0.f), edge_hi = edge_lo;     // old ring slots 1 and B-1 (see the DMA warp)
    V4<R> tg = M<R>::make4(R(0), R(0), R(0), R(0)), ip0 = tg, iq0 = tg;
    const bool pre_init = a.auto_reset && !a.init_per_env;      // shared initial pose: fetch it now, off the epilogue's critical path
    // FP64 (parity mode): these 24 doubles would sit in registers across the substep loop; they are fetched in the epilogue
    // instead (per-index constants: L1/L2 hits), which is what keeps the FP64 variants inside their register budgets
    constexpr bool EARLY_CONST = !M<R>::is_double;
    if (active) {
        load_state(a.p, d, s);
        if constexpr (EARLY_CONST) {
            if (!ctrl) tg = a.p.target[a.target_per_env ? d : (int64_t)i];
            if (pre_init) { ip0 = a.p.init_pos[i]; iq0 = a.p.init_quat[i]; }
        }
        if (i == 0) {                   // per-env bookkeeping: loaded here so its DRAM latency hides behind the physics
            cnt = a.p.counter[e];
            if (a.auto_reset) ep_ret0 = a.p.ep_ret[e];
        }

        if (a.action_type == GPD_ACT_CTRL_RPM) {                 // CtrlAviary.py:140
            V4<R> v = reinterpret_cast<const V4<R>*>(a.actions)[d];
            rpm[0] = clip(v.x, R(0), P.MAX_RPM); rpm[1] = clip(v.y, R(0), P.MAX_RPM);
            rpm[2] = clip(v.z, R(0), P.MAX_RPM); rpm[3] = clip(v.w, R(0), P.MAX_RPM);
        } else if (a.action_type == GPD_ACT_CTRL_VEL) {
            if constexpr (HAS_PID) {                             // VelocityAviary.py:129-170, in the action's own precision
                V4<R> v = reinterpret_cast<const V4<R>*>(a.actions)[d];
                R n = M<R>::sqrt(v.x * v.x + v.y * v.y + v.z * v.z);
                R u0 = R(0), u1 = R(0), u2 = R(0);
                if (n != R(0)) { u0 = v.x / n; u1 = v.y / n; u2 = v.z / n; }
                const R sp = a.speed_limit * M<R>::abs(v.w);
                const R tv[3] = { sp * u0, sp * u1, sp * u2 }, tp[3] = { s.px, s.py, s.pz }, z3[3] = { R(0), R(0), R(0) };
                R roll, pitch, yaw, st[9], r4[4], pe[3], ye;
                quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
                const R trpy[3] = { R(0), R(0), yaw };
#pragma unroll
                for (int k = 0; k < 9; ++k) st[k] = a.p.pid[(int64_t)k * a.D + d];
                pid_compute(a.pid, a.ctrl_dt, s.px, s.py, s.pz, s.qx, s.qy, s.qz, s.qw, s.vx, s.vy, s.vz, tp, trpy, tv, z3,
                            st, r4, pe, ye);
#pragma unroll
                for (int k = 0; k < 9; ++k) a.p.pid[(int64_t)k * a.D + d] = st[k];
                rpm[0] = r4[0]; rpm[1] = r4[1]; rpm[2] = r4[2]; rpm[3] = r4[3];
            }
        } else {
            const float* ap = reinterpret_cast<const float*>(a.actions) + d * a.A;
            if constexpr (VEC) {
                float4 v = __ldg(reinterpret_cast<const float4*>(ap));
                act[0] = v.x; act[1] = v.y; act[2] = v.z; act[3] = v.w;
            } else {
                for (int k = 0; k < a.A; ++k) act[k] = __ldg(ap + k);
            }
        }
        if constexpr (!LEAN) {
            if (a.phy & GPD_PHY_DRAG) {
                V4<R> v = a.p.aux_rpm[d];
                rpm_prev[0] = v.x; rpm_prev[1] = v.y; rpm_prev[2] = v.z; rpm_prev[3] = v.w;
            }
        }
    }

    // ---- _preprocessAction -> rpm (BaseRLAviary.py:189-238) ----
    if (a.action_type == GPD_ACT_RPM) {
#pragma unroll
        for (int k = 0; k < 4; ++k) rpm[k] = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[k]));   // :192, float32 inner ops
    } else if (a.action_type == GPD_ACT_ONE_D_RPM) {
        double v = P.HOVER_RPM_d * (double)__fadd_rn(1.0f, __fmul_rn(0.05f, act[0]));                             // :225
        rpm[0] = rpm[1] = rpm[2] = rpm[3] = v;
    }
    if constexpr (HAS_PID) {
        if (a.action_type == GPD_ACT_PID || a.action_type == GPD_ACT_VEL || a.action_type == GPD_ACT_ONE_D_PID) {
            if (active) {
                R r4[4];
                pid_action(a, d, s, act, r4);
                rpm[0] = r4[0]; rpm[1] = r4[1]; rpm[2] = r4[2]; rpm[3] = r4[3];
            }
        }
    }
    Forcing<R> F;
    make_forcing(P, rpm, F);
    const R rpm_r[4] = { (R)rpm[0], (R)rpm[1], (R)rpm[2], (R)rpm[3] };
    if (a.timeline && t == 0 && F.T == F.T) a.timeline[(int64_t)bid * 8 + 2] = gtime();   // 2: state + action arrived

    // ---- PYB_STEPS_PER_CTRL substeps (BaseAviary.py:343-372), state in registers ----
    R avx = R(0), avy = R(0), avz = R(0);
    R wsum_prev = R(0), wsum_cur = R(0);            // _drag's sum of rotor speeds (:773): constant over the substeps
    if constexpr (!LEAN) {
        if (a.phy & GPD_PHY_DRAG) { wsum_prev = drag_wsum(rpm_prev); wsum_cur = drag_wsum(rpm_r); }
    }
    int sub0 = 0;
    if constexpr (LEAN && !M<R>::is_double) {       // all but the last substep: nothing but the state is needed
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

    if (a.timeline && t == 0 && s.px == s.px) a.timeline[(int64_t)bid * 8 + 3] = gtime(); // 3: substeps done
    // ---- _updateAndStoreKinematicInformation (BaseAviary.py:374,509-519) + outputs ----
    R roll, pitch, yaw;
    quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);

    R rew = R(-1);                      // CtrlAviary.py:144-200: dummy reward/flags
    int term = 0, trunc = 0;
    if constexpr (!EARLY_CONST) {
        if (active && !ctrl) tg = a.p.target[a.target_per_env ? d : (int64_t)i];
    }
    if (!ctrl) {
        R ex = tg.x - s.px, ey = tg.y - s.py, ez = tg.z - s.pz;
        R dist = M<R>::sqrt(ex * ex + ey * ey + ez * ez);
        R d2 = dist * dist;
        R v = R(2) - d2 * d2;           // HoverAviary.py:78 / MultiHoverAviary.py:87
        R r_i = v > R(0) ? v : R(0);
        const R lim = a.env_kind == GPD_ENV_HOVER ? R(1.5) : R(2.0);       // HoverAviary.py:111 / MultiHoverAviary.py:124
        int tr_i = (M<R>::abs(s.px) > lim || M<R>::abs(s.py) > lim || s.pz > R(2.0) ||
                    M<R>::abs(roll) > R(.4) || M<R>::abs(pitch) > R(.4)) ? 1 : 0;
        if constexpr (MULTI) {
            R* red = sm.red();
            int* redi = sm.redi();
            phys_sync(nphys);
            if (t < a.DPB) { red[2 * t] = active ? r_i : R(0); red[2 * t + 1] = active ? dist : R(0); redi[t] = active ? tr_i : 0; }
            phys_sync(nphys);
            if (active && i == 0) {     // in-order sums over the env's drones (MultiHoverAviary.py:86-88,103-105)
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
    if (active && i == 0) {
        if (!ctrl && cnt > a.max_counter) trunc = 1;   // HoverAviary.py:114 (counter BEFORE the increment); threshold from the host
        if (a.reward) a.reward[e] = rew;
        if (a.terminated) a.terminated[e] = (uint8_t)term;
        if (a.truncated) a.truncated[e] = (uint8_t)trunc;
    }
    int done = 0;
    if (a.auto_reset) {
        done = term | trunc;
        if constexpr (MULTI) {
            int* envf = sm.envf();
            phys_sync(nphys);
            if (active && i == 0) envf[le] = done;
            phys_sync(nphys);
            done = active ? envf[le] : 0;
        }
    }

    float kin[12];
    kin[0] = (float)s.px; kin[1] = (float)s.py; kin[2] = (float)s.pz;
    kin[3] = (float)roll; kin[4] = (float)pitch; kin[5] = (float)yaw;
    kin[6] = (float)s.vx; kin[7] = (float)s.vy; kin[8] = (float)s.vz;
    kin[9] = (float)avx; kin[10] = (float)avy; kin[11] = (float)avz;
    R out_rpm[4] = { rpm_r[0], rpm_r[1], rpm_r[2], rpm_r[3] };

    if (a.auto_reset) {                 // Monitor-style episode statistics (examples/learn.py:53-57 wraps the env in Monitor)
        const bool lead = active && i == 0;
        float er = ep_ret0 + (float)rew;
        int el = cnt / a.S + 1;         // episode length in ctrl steps: the counter restarts with the episode
        const bool fin = lead && done;
        const unsigned m = __ballot_sync(0xffffffffu, fin);
        float s1 = 0.f, s2 = 0.f;
        int nl = 0, nt = 0, mn = 0x7fffffff, mx = (int)0x80000000;
        if (m) {                        // reduce the finished episodes of this warp
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
        if ((t & 31) == 0) {            // every physics warp owns a slot: plain stores, no atomics, no initialisation pass
            float* sf = sm.stat_f() + 4 * (t >> 5);
            int* si = sm.stat_i() + 4 * (t >> 5);
            sf[0] = s1; sf[1] = s2; sf[2] = (float)nt;
            si[0] = __popc(m); si[1] = nl; si[2] = mn; si[3] = mx;
        }
        if (lead) a.p.ep_ret[e] = fin ? 0.f : er;
    }
    if (a.auto_reset && active) {
        if (done) {
            if (a.terminal_kin && !ctrl) {
                float4* tk = reinterpret_cast<float4*>(a.terminal_kin) + d * 3;
                tk[0] = make_float4(kin[0], kin[1], kin[2], kin[3]);
                tk[1] = make_float4(kin[4], kin[5], kin[6], kin[7]);
                tk[2] = make_float4(kin[8], kin[9], kin[10], kin[11]);
            }
            if (pre_init) {             // BaseAviary.reset -> _housekeeping (BaseAviary.py:451-491)
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
            out_rpm[0] = out_rpm[1] = out_rpm[2] = out_rpm[3] = R(0);       // last_clipped_action zeroed, :468
            kin[0] = (float)s.px; kin[1] = (float)s.py; kin[2] = (float)s.pz;
            kin[3] = (float)roll; kin[4] = (float)pitch; kin[5] = (float)yaw;
#pragma unroll
            for (int k = 6; k < 12; ++k) kin[k] = 0.f;
        }
    }
    if (active) {
        if (i == 0) a.p.counter[e] = (a.auto_reset && done) ? 0 : cnt + a.S;   // BaseAviary.py:382
        store_state(a.p, d, s);
        if (!(LEAN && a.skip_aux)) {    // lean FP32 KIN sims: both live in the observation row written below (derive_aux)
            a.p.aux_av[d] = M<R>::make4(avx, avy, avz, R(0));
            a.p.aux_rpm[d] = M<R>::make4(out_rpm[0], out_rpm[1], out_rpm[2], out_rpm[3]);
        } else if (d == 0) {
            *a.p.aux_auth = 0;
        }
    }

    if (a.kin_t && active && !ctrl) {   // host mirror (gpd_step_mirror): feature-major copy of the kin part, coalesced per feature
#pragma unroll
        for (int k = 0; k < 12; ++k) a.kin_t[(int64_t)k * a.kin_ld + d] = kin[k];
    }

    // ---- stage this drone's observation row in shared memory ----
    if (t < a.DPB) {
        if (ctrl) {                     // CtrlAviary.py:117: obs = state20 rows
            R* r = sm.stage_r() + 20 * t;
            r[0] = s.px; r[1] = s.py; r[2] = s.pz; r[3] = s.qx; r[4] = s.qy; r[5] = s.qz; r[6] = s.qw;
            r[7] = roll; r[8] = pitch; r[9] = yaw; r[10] = s.vx; r[11] = s.vy; r[12] = s.vz;
            r[13] = avx; r[14] = avy; r[15] = avz; r[16] = out_rpm[0]; r[17] = out_rpm[1]; r[18] = out_rpm[2]; r[19] = out_rpm[3];
        } else if (active) {
            // KIN observation, BaseRLAviary.py:310-316: 12 float32 at the head of this drone's row.  48 contiguous
            // bytes per thread; L2 merges them with the history part written by the copy warps.
            if constexpr (VEC) {
                float4* r = reinterpret_cast<float4*>(reinterpret_cast<float*>(a.obs_out) + d * a.W);
                r[0] = make_float4(kin[0], kin[1], kin[2], kin[3]);
                r[1] = make_float4(kin[4], kin[5], kin[6], kin[7]);
                r[2] = make_float4(kin[8], kin[9], kin[10], kin[11]);
                const int W4 = a.W >> 2;
                r[W4 - 1] = make_float4(act[0], act[1], act[2], act[3]);           // newest ring slot, BaseRLAviary.py:187
                if (edge_smem) {        // complete the two sectors shared with the TMA part from the edge boxes
                    mbar_wait(&tma_bar, 0);
                    const float4* elo = reinterpret_cast<const float4*>(smem_raw + a.tma_bytes - 2 * a.tma_edge_bytes);
                    const float4* ehi = reinterpret_cast<const float4*>(smem_raw + a.tma_bytes - a.tma_edge_bytes);
                    edge_lo = elo[t]; edge_hi = ehi[t];
                    r[3] = edge_lo; r[W4 - 2] = edge_hi;
                }
            } else {
                float* r = reinterpret_cast<float*>(a.obs_out) + d * a.W;
#pragma unroll
                for (int k = 0; k < 12; ++k) r[k] = kin[k];
            }
        }
    }
    }   // run_physics

    if (!a.pdl_trigger_early) pdl_launch_dependents();   // this CTA has issued all its loads and (physics warps) stores
    if (a.timeline && t == 0) a.timeline[(int64_t)bid * 8 + 4] = gtime();      // 4: physics thread 0 stored everything
    // ---- Ctrl observation tile: coalesced write of the staged state20 rows (contiguous in global memory) ----
    if (ctrl || a.auto_reset || a.tile_dep) __syncthreads();
    if (a.timeline && t == 0) a.timeline[(int64_t)bid * 8 + 7] = gtime();      // 7: block barrier passed
    if (ctrl) {
        const R* st = sm.stage_r();
        R* out = reinterpret_cast<R*>(a.obs_out) + row0 * 20;
        for (int idx = t; idx < rows * 20; idx += blockDim.x) out[idx] = st[idx];
    }

    if (a.auto_reset && t == 0) {       // combine the warps' partials, then RED (no return value, no wait) into this CTA's slot
        StatSlot* slot = a.p.stat_slots + bid;
        int n = 0, len = 0, mn = 0x7fffffff, mx = (int)0x80000000;
        float sr = 0.f, sr2 = 0.f, st = 0.f;
        for (int w = 0; w < (nphys >> 5); ++w) {
            const float* sf = sm.stat_f() + 4 * w;
            const int* si = sm.stat_i() + 4 * w;
            n += si[0]; len += si[1]; mn = min(mn, si[2]); mx = max(mx, si[3]);
            sr += sf[0]; sr2 += sf[1]; st += sf[2];
        }
        if (n > 0) {
            atomicAdd(&slot->s[0], (double)n);
            atomicAdd(&slot->s[1], (double)sr);
            atomicAdd(&slot->s[2], (double)len);
            atomicAdd(&slot->s[3], (double)sr2);
            atomicMin(&slot->mn, mn);
            atomicMax(&slot->mx, mx);
            if (st > 0.f) atomicAdd(&slot->s[5], (double)st);
        }
        atomicAdd(&slot->s[4], (double)(MULTI ? min((int64_t)a.EPB, a.E - (int64_t)bid * a.EPB) : rows));
    }
    if (a.tile_dep) {
        if (ctrl) __syncthreads();      // the tile write-out above is part of what the next step of this tile reads
        // every global write of this CTA happened before the barrier(s) above: publish the tile (release, gpu scope)
        if (t == 0) tile_publish(a.tile_seq + (int64_t)bid * 4);
        // keep stream order transitive: this grid does not complete before the grids it was allowed to overtake
        pdl_wait();
    }
}

// ============================================================================================
// reset: BaseAviary.reset (BaseAviary.py:220-255) for the masked envs + observation of every env.
// ============================================================================================
template <typename R, bool VEC>
__global__ void __launch_bounds__(288)
reset_kernel(const __grid_constant__ StepArgs<R> a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const bool ctrl = a.env_kind == GPD_ENV_CTRL;
    Smem<R> sm{ smem_raw + a.tma_bytes, a.DPB, a.EPB, ctrl, false };
    const int t = threadIdx.x;
    const int64_t row0 = (int64_t)blockIdx.x * a.DPB;
    const int64_t d = row0 + t;
    const bool active = t < a.DPB && d < a.D;
    const int rows = (int)min((int64_t)a.DPB, a.D - row0);
    const int le = t / a.N, i = t - le * a.N;
    const int64_t e = (int64_t)blockIdx.x * a.EPB + le;

    if (!ctrl && a.obs_out)
        copy_history<VEC>(a.obs_prev, reinterpret_cast<float*>(a.obs_out), nullptr, row0, rows, a.W, a.A, a.B, false, t, (int)blockDim.x);

    State<R> s;
    s.px = s.py = s.pz = s.qx = s.qy = s.qz = R(0); s.qw = R(1);
    s.vx = s.vy = s.vz = s.wx = s.wy = s.wz = R(0);
    R avx = R(0), avy = R(0), avz = R(0);
    R rpm[4] = { R(0), R(0), R(0), R(0) };
    if (active) {
        bool doit = a.reset_mask == nullptr || a.reset_mask[e] != 0;
        if (doit) {
            init_state(a, d, i, s);
            store_state(a.p, d, s);
            a.p.aux_av[d] = M<R>::make4(R(0), R(0), R(0), R(0));
            a.p.aux_rpm[d] = M<R>::make4(R(0), R(0), R(0), R(0));
            if (i == 0) {
                a.p.counter[e] = 0;
                if (a.p.ep_ret) a.p.ep_ret[e] = 0.f;
            }
            if (d == 0 && a.reset_mask == nullptr) *a.p.aux_auth = 1;     // everything was reset: the (zero) arrays are exact
        } else {
            load_state(a.p, d, s);
            if (a.skip_aux && a.obs_prev && *a.p.aux_auth == 0) {
                R av3[3];
                derive_aux(a, a.obs_prev, d, e, av3, rpm);
                avx = av3[0]; avy = av3[1]; avz = av3[2];
            } else {
                V4<R> av = a.p.aux_av[d], rp = a.p.aux_rpm[d];
                avx = av.x; avy = av.y; avz = av.z;
                rpm[0] = rp.x; rpm[1] = rp.y; rpm[2] = rp.z; rpm[3] = rp.w;
            }
        }
    }
    if (!a.obs_out) return;
    R roll, pitch, yaw;
    quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
    if (ctrl) {
        R* st = sm.stage_r();
        if (t < a.DPB) {
            R* r = st + 20 * t;
            r[0] = s.px; r[1] = s.py; r[2] = s.pz; r[3] = s.qx; r[4] = s.qy; r[5] = s.qz; r[6] = s.qw;
            r[7] = roll; r[8] = pitch; r[9] = yaw; r[10] = s.vx; r[11] = s.vy; r[12] = s.vz;
            r[13] = avx; r[14] = avy; r[15] = avz; r[16] = rpm[0]; r[17] = rpm[1]; r[18] = rpm[2]; r[19] = rpm[3];
        }
        __syncthreads();
        R* out = reinterpret_cast<R*>(a.obs_out) + row0 * 20;
        for (int idx = t; idx < rows * 20; idx += blockDim.x) out[idx] = st[idx];
    } else if (active) {                // KIN part of the row, BaseRLAviary.py:310-316 (the ring part was copied above)
        const float kin[12] = { (float)s.px, (float)s.py, (float)s.pz, (float)roll, (float)pitch, (float)yaw,
                                (float)s.vx, (float)s.vy, (float)s.vz, (float)avx, (float)avy, (float)avz };
        float* r = reinterpret_cast<float*>(a.obs_out) + d * a.W;
        if constexpr (VEC) {
            float4* r4 = reinterpret_cast<float4*>(r);
            r4[0] = make_float4(kin[0], kin[1], kin[2], kin[3]);
            r4[1] = make_float4(kin[4], kin[5], kin[6], kin[7]);
            r4[2] = make_float4(kin[8], kin[9], kin[10], kin[11]);
        } else {
#pragma unroll
            for (int k = 0; k < 12; ++k) r[k] = kin[k];
        }
    }
}

// ---- state export / import (BaseAviary._getDroneStateVector, BaseAviary.py:541-561) ----
template <typename R>
__global__ void get_state_kernel(const StepArgs<R> a, const float* __restrict__ obs_latest, R* __restrict__ state20,
                                 R* __restrict__ rpy_rates, R* __restrict__ pid_state, int32_t* __restrict__ counter)
{
    int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d < a.E && counter) counter[d] = a.p.counter[d];
    if (d >= a.D) return;
    State<R> s;
    load_state(a.p, d, s);
    if (state20) {
        R roll, pitch, yaw;
        quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
        V4<R> av, rp;
        if (a.skip_aux && obs_latest && *a.p.aux_auth == 0) {
            R av3[3], r4[4];
            derive_aux(a, obs_latest, d, d / a.N, av3, r4);
            av = M<R>::make4(av3[0], av3[1], av3[2], R(0)); rp = M<R>::make4(r4[0], r4[1], r4[2], r4[3]);
        } else {
            av = a.p.aux_av[d]; rp = a.p.aux_rpm[d];
        }
        R* r = state20 + d * 20;
        r[0] = s.px; r[1] = s.py; r[2] = s.pz; r[3] = s.qx; r[4] = s.qy; r[5] = s.qz; r[6] = s.qw;
        r[7] = roll; r[8] = pitch; r[9] = yaw; r[10] = s.vx; r[11] = s.vy; r[12] = s.vz;
        r[13] = av.x; r[14] = av.y; r[15] = av.z; r[16] = rp.x; r[17] = rp.y; r[18] = rp.z; r[19] = rp.w;
    }
    if (rpy_rates) { rpy_rates[d * 3] = s.wx; rpy_rates[d * 3 + 1] = s.wy; rpy_rates[d * 3 + 2] = s.wz; }
    if (pid_state && a.p.pid)
        for (int k = 0; k < 9; ++k) pid_state[d * 9 + k] = a.p.pid[(int64_t)k * a.D + d];
}

template <typename R>
__global__ void set_state_kernel(const StepArgs<R> a, const R* __restrict__ state20, const R* __restrict__ rpy_rates,
                                 const R* __restrict__ pid_state, const int32_t* __restrict__ counter)
{
    int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d < a.E && counter) a.p.counter[d] = counter[d];
    if (d >= a.D) return;
    State<R> s;
    load_state(a.p, d, s);
    if (state20) {
        const R* r = state20 + d * 20;
        s.px = r[0]; s.py = r[1]; s.pz = r[2]; s.qx = r[3]; s.qy = r[4]; s.qz = r[5]; s.qw = r[6];
        s.vx = r[10]; s.vy = r[11]; s.vz = r[12];
        a.p.aux_av[d] = M<R>::make4(r[13], r[14], r[15], R(0));
        a.p.aux_rpm[d] = M<R>::make4(r[16], r[17], r[18], r[19]);
        if (d == 0) *a.p.aux_auth = 1;      // every drone's ang_v / last_clipped_action was just written
    }
    if (rpy_rates) { s.wx = rpy_rates[d * 3]; s.wy = rpy_rates[d * 3 + 1]; s.wz = rpy_rates[d * 3 + 2]; }
    store_state(a.p, d, s);
    if (pid_state && a.p.pid)
        for (int k = 0; k < 9; ++k) a.p.pid[(int64_t)k * a.D + d] = pid_state[d * 9 + k];
}

// ---- failure detection: count drones with a non-finite integrator state ----
template <typename R>
__global__ void nonfinite_kernel(const StepArgs<R> a, unsigned long long* __restrict__ out)
{
    int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool bad = false;
    if (d < a.D) {
        State<R> s;
        load_state(a.p, d, s);
        const R v[13] = { s.px, s.py, s.pz, s.qx, s.qy, s.qz, s.qw, s.vx, s.vy, s.vz, s.wx, s.wy, s.wz };
#pragma unroll
        for (int k = 0; k < 13; ++k) bad |= !isfinite(v[k]);
    }
    const unsigned m = __ballot_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(out, (unsigned long long)__popc(m));
}

// ---- batched DSLPIDControl.computeControl (control/DSLPIDControl.py:82-145) ----
template <typename R>
__global__ void pid_kernel(const DevPid<R> c, int64_t n, R dt, const R* __restrict__ cur_pos, const R* __restrict__ cur_quat,
                           const R* __restrict__ cur_vel, const R* __restrict__ target_pos, const R* __restrict__ target_rpy,
                           const R* __restrict__ target_vel, const R* __restrict__ target_rates, R* __restrict__ pid_state,
                           R* __restrict__ rpm_out, R* __restrict__ pos_e_out, R* __restrict__ yaw_e_out)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    R tp[3], trpy[3] = { 0, 0, 0 }, tv[3] = { 0, 0, 0 }, tr[3] = { 0, 0, 0 }, st[9], rpm[4], pe[3], ye;
    for (int j = 0; j < 3; ++j) {
        tp[j] = target_pos[k * 3 + j];
        if (target_rpy) trpy[j] = target_rpy[k * 3 + j];
        if (target_vel) tv[j] = target_vel[k * 3 + j];
        if (target_rates) tr[j] = target_rates[k * 3 + j];
    }
    for (int j = 0; j < 9; ++j) st[j] = pid_state[k * 9 + j];
    pid_compute(c, dt, cur_pos[k * 3], cur_pos[k * 3 + 1], cur_pos[k * 3 + 2], cur_quat[k * 4], cur_quat[k * 4 + 1],
                cur_quat[k * 4 + 2], cur_quat[k * 4 + 3], cur_vel[k * 3], cur_vel[k * 3 + 1], cur_vel[k * 3 + 2],
                tp, trpy, tv, tr, st, rpm, pe, ye);
    for (int j = 0; j < 9; ++j) pid_state[k * 9 + j] = st[j];
    for (int j = 0; j < 4; ++j) rpm_out[k * 4 + j] = rpm[j];
    if (pos_e_out) for (int j = 0; j < 3; ++j) pos_e_out[k * 3 + j] = pe[j];
    if (yaw_e_out) yaw_e_out[k] = ye;
}

// ---- force-model unit-test kernels (BaseAviary.py:715-811) ----
template <typename R>
__global__ void ground_effect_kernel(const DevDrone<R> P, int64_t n, const R* __restrict__ rpm, const R* __restrict__ pos,
                                     const R* __restrict__ quat, R* __restrict__ out, uint8_t* __restrict__ applied)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    R m[9], roll, pitch, yaw, g[4];
    const R* q = quat + k * 4;
    quat_to_mat(q[0], q[1], q[2], q[3], m);
    quat_to_euler(q[0], q[1], q[2], q[3], roll, pitch, yaw);
    R r4[4] = { rpm[k * 4], rpm[k * 4 + 1], rpm[k * 4 + 2], rpm[k * 4 + 3] };
    bool ok = ground_effect(P, r4, pos[k * 3 + 2], m, roll, pitch, g);
    for (int j = 0; j < 4; ++j) out[k * 4 + j] = g[j];
    if (applied) applied[k] = ok ? 1 : 0;
}

template <typename R>
__global__ void drag_kernel(const DevDrone<R> P, int64_t n, const R* __restrict__ rpm, const R* __restrict__ quat,
                            const R* __restrict__ vel, R* __restrict__ out)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    R m[9], o[3];
    const R* q = quat + k * 4;
    quat_to_mat(q[0], q[1], q[2], q[3], m);
    R r4[4] = { rpm[k * 4], rpm[k * 4 + 1], rpm[k * 4 + 2], rpm[k * 4 + 3] };
    drag_body(P, r4, m, vel[k * 3], vel[k * 3 + 1], vel[k * 3 + 2], o);
    for (int j = 0; j < 3; ++j) out[k * 3 + j] = o[j];
}

template <typename R>
__global__ void downwash_kernel(const DevDrone<R> P, int64_t E, int N, const R* __restrict__ pos, R* __restrict__ out)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= E * N) return;
    int64_t e = k / N;
    const R* env = pos + e * N * 3;
    const R* me = pos + k * 3;
    R dw = R(0);
    for (int j = 0; j < N; ++j) dw += downwash_pair(P, me[0], me[1], me[2], env[3 * j], env[3 * j + 1], env[3 * j + 2]);
    out[k] = dw;
}

// ============================================================================================
// examples/pid.py:127-147 as one launch: n_steps x { step(action); action = DSLPID(obs, waypoint) }.
// Ctrl env, one thread per drone, state + controller state in registers for the whole rollout.
// ============================================================================================
template <typename R>
__global__ void __launch_bounds__(128)
rollout_pid_kernel(const __grid_constant__ StepArgs<R> a, int n_steps, const R* __restrict__ waypoints, int n_wp,
                   int32_t* __restrict__ wp_counters, R* __restrict__ action)
{
    const int64_t d = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= a.D) return;
    const int i = (int)(d % a.N);
    const int64_t e = d / a.N;
    const DevDrone<R>& P = a.drone;
    State<R> s;
    load_state(a.p, d, s);
    R st[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) st[k] = a.p.pid[(int64_t)k * a.D + d];
    V4<R> av4 = reinterpret_cast<V4<R>*>(action)[d];
    R act[4] = { av4.x, av4.y, av4.z, av4.w };
    V4<R> rp = a.p.aux_rpm[d];
    R rpm_prev[4] = { rp.x, rp.y, rp.z, rp.w };
    int wp = wp_counters[d];
    const int64_t ik = a.init_per_env ? d : (int64_t)i;
    V4<R> ip = a.p.init_pos[ik], iq = a.p.init_quat[ik];
    R ir, ipt, iy;
    quat_to_euler(iq.x, iq.y, iq.z, iq.w, ir, ipt, iy);
    const R trpy[3] = { ir, ipt, iy }, zero3[3] = { R(0), R(0), R(0) };
    R avx = a.p.aux_av[d].x, avy = a.p.aux_av[d].y, avz = a.p.aux_av[d].z;
    R rpm_r[4] = { rpm_prev[0], rpm_prev[1], rpm_prev[2], rpm_prev[3] };
    for (int it = 0; it < n_steps; ++it) {
        double rpm[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) { rpm_r[k] = clip(act[k], R(0), P.MAX_RPM); rpm[k] = rpm_r[k]; }   // CtrlAviary.py:140
        Forcing<R> F;
        make_forcing(P, rpm, F);
        for (int sub = 0; sub < a.S; ++sub) {
            R m[9];
            const R omz = quat_to_mat(s.qx, s.qy, s.qz, s.qw, m);
            R gnd[4], fb[3] = { R(0), R(0), R(0) };
            const R* pg = nullptr;
            const R* pb = nullptr;
            if (a.phy & GPD_PHY_GND) {
                R roll, pitch, yaw;
                quat_to_euler(s.qx, s.qy, s.qz, s.qw, roll, pitch, yaw);
                if (ground_effect(P, rpm_r, s.pz, m, roll, pitch, gnd)) pg = gnd;
            }
            if (a.phy & GPD_PHY_DRAG) {
                drag_body(P, sub == 0 ? rpm_prev : rpm_r, m, s.vx, s.vy, s.vz, fb);
                pb = fb;
            }
            dyn_substep<R>(P, a.dt, s, m, omz, F, pg, pb, true, avx, avy, avz);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) rpm_prev[k] = rpm_r[k];
        // examples/pid.py:142-147 computeControlFromState(state=obs[j], target_pos=[wp.xy, INIT z], target_rpy=INIT_RPYS[j])
        const R tp[3] = { waypoints[3 * wp], waypoints[3 * wp + 1], ip.z };
        R pe[3], ye;
        pid_compute(a.pid, a.ctrl_dt, s.px, s.py, s.pz, s.qx, s.qy, s.qz, s.qw, s.vx, s.vy, s.vz, tp, trpy, zero3, zero3,
                    st, act, pe, ye);
        wp = wp < n_wp - 1 ? wp + 1 : 0;                                                   // examples/pid.py:151
    }
    store_state(a.p, d, s);
    a.p.aux_av[d] = M<R>::make4(avx, avy, avz, R(0));
    a.p.aux_rpm[d] = M<R>::make4(rpm_r[0], rpm_r[1], rpm_r[2], rpm_r[3]);
#pragma unroll
    for (int k = 0; k < 9; ++k) a.p.pid[(int64_t)k * a.D + d] = st[k];
    reinterpret_cast<V4<R>*>(action)[d] = M<R>::make4(act[0], act[1], act[2], act[3]);
    wp_counters[d] = wp;
    if (i == 0) a.p.counter[e] += a.S * n_steps;
}


// ============================================================================================
// BaseAviary._getAdjacencyMatrix (BaseAviary.py:658-675): adj[e][i][j] = 1 on the diagonal and where
// ||pos_i - pos_j|| < NEIGHBOURHOOD_RADIUS (np.linalg.norm of a float64 3-vector = sqrt of the in-order sum of squares;
// pos_i - pos_j with i < j as in the reference loop, mirrored), else 0.  Same per-env position tile in shared memory
// as the downwash snapshot of the step kernel; a CTA owns whole envs, its threads sweep the N x N outputs contiguously.
// ============================================================================================
template <typename R>
__global__ void __launch_bounds__(256)
adjacency_kernel(const typename Vec4<R>::type* __restrict__ sP, int64_t E, int N, int EPC, R radius, R* __restrict__ out)
{
    extern __shared__ __align__(16) unsigned char adj_smem[];
    V4<R>* pos = reinterpret_cast<V4<R>*>(adj_smem);
    const int64_t e0 = (int64_t)blockIdx.x * EPC;
    const int envs = (int)min((int64_t)EPC, E - e0);
    for (int k = threadIdx.x; k < envs * N; k += blockDim.x) pos[k] = sP[e0 * N + k];
    __syncthreads();
    const int NN = N * N;
    R* o = out + e0 * NN;
    for (int idx = threadIdx.x; idx < envs * NN; idx += blockDim.x) {
        const int le = idx / NN, r = idx - le * NN, i = r / N, j = r - i * N;
        R v = R(1);
        if (i != j) {
            const V4<R> a = pos[le * N + min(i, j)], b = pos[le * N + max(i, j)];
            const R dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z;
            v = M<R>::sqrt(dx * dx + dy * dy + dz * dz) < radius ? R(1) : R(0);
        }
        o[idx] = v;
    }
}

}  // namespace gpd
