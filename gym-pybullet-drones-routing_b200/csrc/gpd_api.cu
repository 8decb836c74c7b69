// gpd_api.cu — the C ABI of libgpd_b200 (include/gpd.h): handle management, argument checking,
// dispatch on precision.  No compute happens on the host: without a CUDA device every entry point
// that would compute returns GPD_ERR_NO_DEVICE (there is no CPU fallback).
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <mutex>
#include <new>
#include <unordered_map>
#include <vector>

#include <dlfcn.h>
#include <nccl.h>          // types only: the library is bound at run time (dlopen), never linked
#include <xmmintrin.h>

#include "gpd_internal.h"

namespace gpd {
cudaError_t launch_stats(const StatSlot* slots, int64_t nslots, double* out8, int clear, StatSlot* slots_mut, cudaStream_t st);
cudaError_t launch_stats_combine(const double* gathered, int nranks, double* out8, cudaStream_t st);
cudaError_t launch_transpose_cols(const float* obs, int64_t D, int W, int j0, int j1, float* out, int64_t ld, cudaStream_t st);
}

using namespace gpd;

static thread_local char g_err[512] = "";

typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_tiled_fn get_encode_fn()
{
    static encode_tiled_fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (encode_tiled_fn)p;
    }
    return fn;
}

static int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail(_e == cudaErrorNoDevice || _e == cudaErrorInsufficientDriver ? GPD_ERR_NO_DEVICE : GPD_ERR_CUDA, \
                        "%s failed: %s", #call, cudaGetErrorString(_e));                           \
    } while (0)

// Host mirror of the RL observation (gpd_step_mirror): the observation window of every drone lives in a feature-major log in
// pinned host memory, log[row][col]: row = observation feature, col = drone.  The window of step t is rows [row, row + W):
// 12 kin rows then the A*B ring rows, oldest -> newest.  A step slides the window by A rows: the device sends only what it
// computed (12 kin rows, reward, flags); the newest action is written by the host from its own copy; nothing is echoed.
struct Mirror {
    float* log = nullptr;
    int64_t rows = 0, ld = 0, col0 = 0;
    int64_t row = 0;                // first row of the current window
    bool valid = false;             // the window matches the device observation `synced_obs` as of sequence `synced_seq`
    uint64_t synced_seq = 0;
    const void* synced_obs = nullptr;
    float* d_kin_t = nullptr;       // device [12][D]
    float* d_log = nullptr;         // device alias of the pinned log (cudaHostGetDevicePointer), or nullptr
    int zero_copy = 1;              // the step kernel reads the actions from and writes kin / reward / flags to pinned host memory itself
    float* d_full_t = nullptr;      // device [W][D], refresh scratch (lazy)
    bool pending = false;           // a begin without its end
    const void* pending_obs = nullptr;
    const float* pending_actions = nullptr;
};

struct TmapEntry { CUtensorMap tm; uint64_t tick; };

struct gpd_sim {
    gpd_config cfg;
    int A, B, W, S;
    int64_t D;
    LaunchCfg lc;
    int dpb = 0;
    int copy_threads = 0;
    int tile_dep = 1;                 // per-CTA step sequencing (decided in gpd_create from the number of waves)
    int chaining = 0;                 // gpd_set_step_chaining: the caller vouches for its step inputs (see gpd.h)
    bool bulk_ok = false;             // single-drone RL env with 4-wide actions: the bulk-copy data path (gpd_step_bulk.cuh)
    LaunchCfg lc_bulk{};
    int bulk_direct = 0;              // BulkSmem::direct
    int bulk_tpc = 1;                 // tiles per CTA of chained bulk launches
    int64_t d_pad = 0;                // per-env scalar arrays are allocated for whole tiles (grid * DPB entries)
    const void* last_obs = nullptr;   // the observation buffer most recently written by gpd_step / gpd_reset (device)
    uint64_t obs_seq = 0;             // bumped whenever the device observation chain advances (or is replaced by the caller)
    std::vector<void*> allocs;
    StepArgs<float> a32;
    StepArgs<double> a64;
    std::vector<double> target_host;
    // host-buffer paths (gpd_step_host / gpd_step_mirror): device staging, allocated lazily and all-or-nothing
    void* h_act = nullptr;            // actions
    void* h_obs[2] = { nullptr, nullptr };   // internal observation ping-pong: [obs | reward | terminated | truncated] each
    float* h_tkin = nullptr;
    uint8_t* h_mask = nullptr;        // persistent reset mask
    int h_cur = 0;
    bool h_has_prev = false;
    double* stats_out = nullptr;
    double* stats_gather = nullptr;   // [nranks][8] for the in-library NCCL all-gather
    int stats_gather_ranks = 0;
    void* init_bufs[2] = { nullptr, nullptr };   // current initial-pose arrays (replaced by gpd_set_init_poses)
    void* target_buf = nullptr;
    Mirror mir;
    // TMA: one tensor map per observation buffer the caller has passed (2-D [D rows][W floats], box [DPB][(B-1)*4])
    bool tma_ok = false;
    int tma_bytes = 0, tma_bytes_box = 0, tma_edge = 0;
    std::unordered_map<const void*, TmapEntry> tmaps, tmaps_edge;
    uint64_t tmap_tick = 0;
    int tma_edge_bytes = 0;
};

// Tensor maps are cached per observation buffer (trajectory-chained rollouts use one buffer per step, rollout.py); the
// least recently used entry is evicted beyond GPD_TMAP_CACHE entries.  Returned by value: no pointer into the table escapes.
enum { GPD_TMAP_CACHE = 1024 };
static bool get_tmap(gpd_sim* s, const void* base, bool edge, CUtensorMap* out)
{
    auto& cache = edge ? s->tmaps_edge : s->tmaps;
    auto it = cache.find(base);
    if (it != cache.end()) { it->second.tick = ++s->tmap_tick; *out = it->second.tm; return true; }
    encode_tiled_fn enc = get_encode_fn();
    if (!enc || ((uintptr_t)base & 15)) return false;
    if (cache.size() >= GPD_TMAP_CACHE) {
        auto victim = cache.begin();
        for (auto jt = cache.begin(); jt != cache.end(); ++jt)
            if (jt->second.tick < victim->second.tick) victim = jt;
        cache.erase(victim);
    }
    CUtensorMap tm;
    cuuint64_t gdim[2] = { (cuuint64_t)s->W, (cuuint64_t)s->D };
    cuuint64_t gstr[1] = { (cuuint64_t)s->W * 4 };
    // A = 4: the shifted slots only; A < 4: the whole ring (the shift happens in shared memory)
    cuuint32_t box[2] = { (cuuint32_t)(edge ? 4 : (s->A == 4 ? (s->B - 1 - 2 * s->tma_edge) * 4 : s->A * s->B)), (cuuint32_t)s->dpb };
    cuuint32_t estr[2] = { 1, 1 };
    CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return false;
    cache.emplace(base, TmapEntry{ tm, ++s->tmap_tick });
    *out = tm;
    return true;
}

// cudaSetDevice only when the calling thread's current device differs (the step path is called ~1e5 times per second)
static cudaError_t use_device(int dev)
{
    int cur = -1;
    cudaError_t e = cudaGetDevice(&cur);
    if (e != cudaSuccess) return e;
    return cur == dev ? cudaSuccess : cudaSetDevice(dev);
}

// Chained stepping (gpd_set_step_chaining): a step kernel is launched programmatically only behind ANOTHER step kernel of
// this library on the same stream (of any handle: independent env sets stepped in rotation chain too).  The library tracks
// per (device, stream) whether its last launch there was a step kernel; every other launch it makes (reset, set/get state,
// statistics, ...) breaks the chain, so the step that follows is fully ordered behind it.  Work enqueued by others is the
// caller's side of the contract.
struct ChainTable {
    struct Entry { bool last_was_step; unsigned long long capture; const void* sim; };   // capture = id of the stream capture the launch
                                                                                         // belonged to (0: none); sim = its handle
    std::mutex mu;
    std::unordered_map<unsigned long long, Entry> tab;
    static unsigned long long key(int dev, cudaStream_t st) { return ((unsigned long long)(uintptr_t)st << 6) ^ (unsigned long long)dev; }
    bool get(int dev, cudaStream_t st, unsigned long long capture, const void** last_sim = nullptr)
    {
        std::lock_guard<std::mutex> l(mu);
        auto it = tab.find(key(dev, st));
        if (last_sim) *last_sim = it != tab.end() ? it->second.sim : nullptr;
        return it != tab.end() && it->second.last_was_step && it->second.capture == capture;
    }
    void set(int dev, cudaStream_t st, bool v, unsigned long long capture, const void* sim = nullptr)
    {
        std::lock_guard<std::mutex> l(mu);
        if (tab.size() > 4096) tab.clear();      // stream handles come and go; forgetting one only costs one unchained launch
        tab[key(dev, st)] = Entry{ v, capture, sim };
    }
    void clear() { std::lock_guard<std::mutex> l(mu); tab.clear(); }
};
// A step captured into a CUDA graph chains only behind a step of the SAME capture (a stream handle is reused across captures
// and eager work; a graph's first kernel must not claim a predecessor it does not have).
static unsigned long long capture_id(cudaStream_t st)
{
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    unsigned long long id = 0;
    if (cudaStreamGetCaptureInfo(st, &status, &id) != cudaSuccess) { cudaGetLastError(); return 0; }
    return status == cudaStreamCaptureStatusActive ? id : 0;
}
static ChainTable g_chain;
// a launch on `st` that is not a step kernel; calls without a stream of their own (synchronous uploads) break every chain
static inline void unchain(gpd_sim* s, void* stream = nullptr, bool all = false)
{
    if (!s) return;
    if (all) g_chain.clear();
    else g_chain.set(s->cfg.device, (cudaStream_t)stream, false, 0);
}

// Chained-state handles (SimPtrs): writes the state of every tile in chained state back into sP / sV / sWz / ep_ret, reading
// position and velocity from the latest observation, and marks those tiles as held in the arrays.  Every entry point that
// reads or writes the state other than the bulk step calls it first, on its own stream.  A step launched behind it must not
// be chained (it would not wait for it): callers on the step path unchain the stream.
static int sync_state(gpd_sim* s, void* stream)
{
    if (!s->a32.state_in_obs) return GPD_OK;
    CU(launch_state_sync(s->a32, (const float*)s->last_obs, s->lc.grid, (cudaStream_t)stream));
    return GPD_OK;
}

static int action_width(int act)
{
    switch (act) {
    case GPD_ACT_RPM: case GPD_ACT_VEL: case GPD_ACT_CTRL_RPM: case GPD_ACT_CTRL_VEL: return 4;
    case GPD_ACT_PID: return 3;
    case GPD_ACT_ONE_D_RPM: case GPD_ACT_ONE_D_PID: return 1;
    default: return -1;
    }
}

template <typename R>
static void fill_drone(const gpd_drone_params& p, DevDrone<R>& d)
{
    d.model = p.model;
    d.M = (R)p.M; d.L = (R)p.L; d.ARM = (R)(p.L / std::sqrt(2.0));
    d.INV_M = (R)(1.0 / p.M);
    d.KF = (R)p.KF; d.KM = (R)p.KM;
    for (int k = 0; k < 3; ++k) { d.J[k] = (R)p.J[k]; d.JINV[k] = (R)p.J_INV[k]; d.DRAG[k] = (R)p.DRAG_COEFF[k]; }
    d.GRAVITY = (R)p.GRAVITY; d.MAX_RPM = (R)p.MAX_RPM;
    d.GND_EFF_COEFF = (R)p.GND_EFF_COEFF; d.PROP_RADIUS = (R)p.PROP_RADIUS; d.GND_EFF_H_CLIP = (R)p.GND_EFF_H_CLIP;
    for (int i = 0; i < 4; ++i) for (int k = 0; k < 3; ++k) d.ROTOR[i][k] = (R)p.ROTOR_XYZ[i][k];
    d.DW1 = (R)p.DW_COEFF_1; d.DW2 = (R)p.DW_COEFF_2; d.DW3 = (R)p.DW_COEFF_3;
    d.DW1_NEG_PR2_16 = (R)(-p.DW_COEFF_1 * (p.PROP_RADIUS * 0.25) * (p.PROP_RADIUS * 0.25));
    d.KF_d = p.KF; d.KM_d = p.KM; d.GRAVITY_d = p.GRAVITY; d.L_d = p.L; d.ARM_d = p.L / std::sqrt(2.0);
    d.HOVER_RPM_d = p.HOVER_RPM; d.MAX_RPM_d = p.MAX_RPM;
    d.DT_INV_M = (R)0; d.DT_JINV[0] = d.DT_JINV[1] = d.DT_JINV[2] = (R)0;
    d.DT_EULER[0] = d.DT_EULER[1] = d.DT_EULER[2] = (R)0;
}

template <typename R>
static void fill_pid(const gpd_pid_params& p, DevPid<R>& c)
{
    for (int k = 0; k < 3; ++k) {
        c.P_FOR[k] = (R)p.P_FOR[k]; c.I_FOR[k] = (R)p.I_FOR[k]; c.D_FOR[k] = (R)p.D_FOR[k];
        c.P_TOR[k] = (R)p.P_TOR[k]; c.I_TOR[k] = (R)p.I_TOR[k]; c.D_TOR[k] = (R)p.D_TOR[k];
    }
    c.PWM2RPM_SCALE = (R)p.PWM2RPM_SCALE; c.PWM2RPM_CONST = (R)p.PWM2RPM_CONST;
    c.MIN_PWM = (R)p.MIN_PWM; c.MAX_PWM = (R)p.MAX_PWM;
    for (int i = 0; i < 4; ++i) for (int k = 0; k < 3; ++k) c.MIXER[i][k] = (R)p.MIXER[i][k];
    c.GRAVITY = (R)p.GRAVITY; c.KF4 = (R)(4 * p.KF);
}

static size_t smem_bytes(bool f64, bool ctrl, bool multi, int DPB, int EPB)
{
    size_t rs = f64 ? 8 : 4;
    size_t stage = ctrl ? (size_t)DPB * 20 * rs : 0;
    size_t b = (stage + 15) & ~size_t(15);
    if (multi) b += (size_t)DPB * 4 * rs + (size_t)DPB * 2 * rs + (size_t)DPB * 4 + (size_t)EPB * 2 * 4;
    b += 9 * 32;        // per-physics-warp statistics slots (float[4] + int[4] each)
    return (b + 15) & ~size_t(15);
}

template <typename T>
static int dev_alloc(gpd_sim* s, T** p, size_t count, bool zero = true)
{
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T) ? count * sizeof(T) : 16);
    if (e != cudaSuccess) return fail(GPD_ERR_ALLOC, "cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    if (zero) {
        e = cudaMemset(q, 0, count * sizeof(T) ? count * sizeof(T) : 16);
        if (e != cudaSuccess) return fail(GPD_ERR_CUDA, "cudaMemset failed: %s", cudaGetErrorString(e));
    }
    s->allocs.push_back(q);
    *p = (T*)q;
    return GPD_OK;
}

// closed forms used to build the initial poses on the host (BaseAviary.py:488: p.getQuaternionFromEuler)
static void host_quat_from_euler(const double rpy[3], double q[4])
{
    double hr = rpy[0] * 0.5, hp = rpy[1] * 0.5, hy = rpy[2] * 0.5;
    double cy = std::cos(hy), sy = std::sin(hy), cp = std::cos(hp), sp = std::sin(hp), cr = std::cos(hr), sr = std::sin(hr);
    double x = sr * cp * cy - cr * sp * sy, y = cr * sp * cy + sr * cp * sy;
    double z = cr * cp * sy - sr * sp * cy, w = cr * cp * cy + sr * sp * sy;
    double n = std::sqrt(x * x + y * y + z * z + w * w);
    q[0] = x / n; q[1] = y / n; q[2] = z / n; q[3] = w / n;
}

template <typename R>
static int upload_init(gpd_sim* s, StepArgs<R>& a, const double* xyz, const double* rpy, int per_env)
{
    using V = typename Vec4<R>::type;
    int64_t n = per_env ? s->D : s->cfg.num_drones;
    std::vector<V> hp((size_t)n), hq((size_t)n);
    for (int64_t k = 0; k < n; ++k) {
        double q[4];
        host_quat_from_euler(rpy + 3 * k, q);
        hp[k].x = (R)xyz[3 * k]; hp[k].y = (R)xyz[3 * k + 1]; hp[k].z = (R)xyz[3 * k + 2]; hp[k].w = (R)0;
        hq[k].x = (R)q[0]; hq[k].y = (R)q[1]; hq[k].z = (R)q[2]; hq[k].w = (R)q[3];
    }
    // the previous arrays may still be read by kernels in flight on any stream: drain the device, then replace them
    V* dp = nullptr; V* dq = nullptr;
    cudaError_t e = cudaMalloc((void**)&dp, sizeof(V) * n);
    if (e == cudaSuccess) e = cudaMalloc((void**)&dq, sizeof(V) * n);
    if (e == cudaSuccess) e = cudaMemcpy(dp, hp.data(), sizeof(V) * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dq, hq.data(), sizeof(V) * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(dp); cudaFree(dq);
        return fail(GPD_ERR_ALLOC, "initial-pose upload failed: %s", cudaGetErrorString(e));
    }
    cudaFree(s->init_bufs[0]); cudaFree(s->init_bufs[1]);
    s->init_bufs[0] = dp; s->init_bufs[1] = dq;
    a.p.init_pos = dp; a.p.init_quat = dq; a.init_per_env = per_env ? 1 : 0;
    return GPD_OK;
}

// HoverAviary.TARGET_POS (HoverAviary.py:51) / MultiHoverAviary.TARGET_POS = INIT_XYZS + [0,0,1/(i+1)] (MultiHoverAviary.py:71):
// [N][3] shared by every env, or [E][N][3] when the envs start from their own poses.
template <typename R>
static int upload_targets(gpd_sim* s, StepArgs<R>& a, const double* t, int per_env)
{
    using V = typename Vec4<R>::type;
    int64_t n = per_env ? s->D : s->cfg.num_drones;
    std::vector<V> ht((size_t)n);
    for (int64_t k = 0; k < n; ++k) { ht[k].x = (R)t[3 * k]; ht[k].y = (R)t[3 * k + 1]; ht[k].z = (R)t[3 * k + 2]; ht[k].w = (R)0; }
    V* dt_ = nullptr;
    cudaError_t e = cudaMalloc((void**)&dt_, sizeof(V) * n);
    if (e == cudaSuccess) e = cudaMemcpy(dt_, ht.data(), sizeof(V) * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { cudaFree(dt_); return fail(GPD_ERR_ALLOC, "target upload failed: %s", cudaGetErrorString(e)); }
    cudaFree(s->target_buf);
    s->target_buf = dt_;
    a.p.target = dt_; a.target_per_env = per_env ? 1 : 0;
    return GPD_OK;
}

template <typename R>
static int build_args(gpd_sim* s, StepArgs<R>& a)
{
    using V = typename Vec4<R>::type;
    const gpd_config& c = s->cfg;
    memset((void*)&a, 0, sizeof a);
    a.D = s->D; a.E = c.num_envs; a.N = c.num_drones; a.S = s->S; a.A = s->A; a.B = s->B; a.W = s->W;
    a.env_kind = c.env_kind; a.action_type = c.action_type; a.phy = c.physics_flags; a.auto_reset = c.auto_reset;
    a.dt = (R)(1.0 / c.pyb_freq); a.ctrl_dt = (R)(1.0 / c.ctrl_freq); a.speed_limit = (R)c.speed_limit;
    a.pyb_freq = (double)c.pyb_freq; a.episode_len = c.episode_len_sec;
    {   // `step_counter/PYB_FREQ > EPISODE_LEN_SEC` in Python float arithmetic (HoverAviary.py:114) as an integer test
        double guess = std::floor(c.episode_len_sec * c.pyb_freq);
        long long k = guess > 2e9 ? 2000000000LL : (guess < 0 ? 0 : (long long)guess);
        while (k > 0 && (double)k / (double)c.pyb_freq > c.episode_len_sec) --k;
        while (k < 2000000000LL && (double)(k + 1) / (double)c.pyb_freq <= c.episode_len_sec) ++k;
        a.max_counter = (int32_t)k;
    }
    fill_drone(c.drone, a.drone);
    a.drone.DT_INV_M = (R)((1.0 / c.pyb_freq) / c.drone.M);
    for (int k = 0; k < 3; ++k) a.drone.DT_JINV[k] = (R)((1.0 / c.pyb_freq) * c.drone.J_INV[k]);
    for (int k = 0; k < 3; ++k)
        a.drone.DT_EULER[k] = (R)((1.0 / c.pyb_freq) * c.drone.J_INV[k] * (c.drone.J[(k + 2) % 3] - c.drone.J[(k + 1) % 3]));
    fill_pid(c.pid, a.pid);
    int rc;
    V *sP, *sQ, *sV, *av, *rp; R* wz;
    if ((rc = dev_alloc(s, &sP, (size_t)s->D))) return rc;
    if ((rc = dev_alloc(s, &sQ, (size_t)s->D))) return rc;
    if ((rc = dev_alloc(s, &sV, (size_t)s->D))) return rc;
    if ((rc = dev_alloc(s, &wz, (size_t)s->d_pad))) return rc;       // whole tiles: the bulk path copies T entries per CTA
    if ((rc = dev_alloc(s, &av, (size_t)s->D))) return rc;
    if ((rc = dev_alloc(s, &rp, (size_t)s->D))) return rc;
    a.p.sP = sP; a.p.sQ = sQ; a.p.sV = sV; a.p.sWz = wz; a.p.aux_av = av; a.p.aux_rpm = rp;
    int32_t* auth;
    if ((rc = dev_alloc(s, &auth, (size_t)1))) return rc;
    a.p.aux_auth = auth;
    const bool pidfam = c.action_type == GPD_ACT_PID || c.action_type == GPD_ACT_VEL || c.action_type == GPD_ACT_ONE_D_PID;
    R* pid = nullptr;
    if ((rc = dev_alloc(s, &pid, (size_t)s->D * 9))) return rc;      // also used by gpd_rollout_pid
    (void)pidfam;
    a.p.pid = pid;
    int32_t* cnt;
    if ((rc = dev_alloc(s, &cnt, (size_t)(s->d_pad > c.num_envs ? s->d_pad : c.num_envs)))) return rc;
    a.p.counter = cnt;
    if (c.auto_reset) {
        float* er; StatSlot* slots;
        if ((rc = dev_alloc(s, &er, (size_t)(s->d_pad > c.num_envs ? s->d_pad : c.num_envs)))) return rc;
        if ((rc = dev_alloc(s, &slots, (size_t)s->lc.grid))) return rc;
        std::vector<StatSlot> init((size_t)s->lc.grid);
        for (auto& q : init) { for (double& v : q.s) v = 0.0; q.mn = 0x7fffffff; q.mx = (int32_t)0x80000000; }
        CU(cudaMemcpy(slots, init.data(), init.size() * sizeof(StatSlot), cudaMemcpyHostToDevice));
        a.p.ep_ret = er; a.p.stat_slots = slots;
    }
    if ((rc = upload_targets(s, a, s->target_host.data(), 0))) return rc;
    {   // per-CTA step sequencing (see tile_claim_and_wait in gpd_kernels.cuh): one 64-bit word per CTA at a 32-byte stride
        unsigned long long* seq = nullptr;
        if ((rc = dev_alloc(s, &seq, (size_t)s->lc.grid * 4))) return rc;
        a.tile_seq = seq;
        a.tile_dep = s->tile_dep;
    }
    a.DPB = s->dpb;
    a.copy_threads = s->copy_threads;
    a.tma_bytes = s->tma_bytes;
    a.tma_bytes_box = s->tma_bytes_box;
    a.tma_edge = s->tma_edge;
    {
        const char* ev = getenv("GPD_PDL_EARLY");
        a.pdl_trigger_early = ev ? atoi(ev) : ((a.tile_dep || s->lc.grid <= 296) ? 1 : 0);
        // lean FP32 KIN sims keep ang_v / last_clipped_action only in the observation row (32 B per drone-step less to write)
        const bool rpm_act = c.action_type == GPD_ACT_RPM || c.action_type == GPD_ACT_ONE_D_RPM;
        ev = getenv("GPD_AUX_ALWAYS");
        a.skip_aux = (sizeof(R) == 4 && rpm_act && c.physics_flags == 0 && c.env_kind != GPD_ENV_CTRL && !(ev && atoi(ev))) ? 1 : 0;
        // of those, single-drone sims on the bulk kernel chain position and velocity through the observation (SimPtrs): 48 B
        // per env-step less state traffic
        ev = getenv("GPD_STATE_IN_OBS");
        a.state_in_obs = (a.skip_aux && c.num_drones == 1 && s->bulk_ok && s->bulk_direct == 2 && !(ev && atoi(ev) == 0)) ? 1 : 0;
    }
    if (a.state_in_obs) {
        V* sr;
        if ((rc = dev_alloc(s, &sr, (size_t)s->D))) return rc;
        a.sR = sr;
        s->lc_bulk.smem += 16;      // row 0's old kin[0..3] in front of the tile (BulkSmem)
    }
    a.tma_edge_bytes = s->tma_edge_bytes;
    a.bulk_direct = s->bulk_direct;
    a.use_tma = 0;
    a.EPB = a.DPB / c.num_drones;
    // default initial poses, BaseAviary.py:194-207
    std::vector<double> xyz((size_t)c.num_drones * 3), rpy((size_t)c.num_drones * 3, 0.0);
    for (int k = 0; k < c.num_drones; ++k) {
        xyz[3 * k] = k * 4 * c.drone.L; xyz[3 * k + 1] = k * 4 * c.drone.L;
        xyz[3 * k + 2] = c.drone.COLLISION_H / 2 - c.drone.COLLISION_Z_OFFSET + .1;
    }
    return upload_init(s, a, xyz.data(), rpy.data(), 0);
}

// gpd_plan: the copies of every env as PlanArgs, the handle's own StepArgs for everything else
template <typename R>
static cudaError_t plan_launch(const gpd_sim* s, const StepArgs<R>& src, int n_steps, int n_samples, const void* actions,
                               const void* targets, double gamma, void* returns, int32_t* done_step, void* reward,
                               void* final_kin, const LaunchCfg& lc, cudaStream_t st)
{
    StepArgs<R> a = src;
    a.actions = actions;
    PlanArgs<R> q{};
    q.E = s->cfg.num_envs * (int64_t)n_samples;
    q.D = q.E * s->cfg.num_drones;
    q.n_samples = n_samples;
    q.gamma = (R)gamma;
    q.targets = (const R*)targets;
    q.returns = (R*)returns;
    q.done_step = done_step;
    q.reward = (R*)reward;
    q.final_kin = (float*)final_kin;
    return launch_plan<R>(a, q, n_steps, lc, st);
}

// gpd_plan_grad: gpd_plan's copies with the gradient and the tape
template <typename R>
static cudaError_t plan_grad_launch(const gpd_sim* s, const StepArgs<R>& src, int n_steps, int n_samples, const void* actions,
                                    const void* targets, double gamma, void* returns, int32_t* done_step, void* grad,
                                    void* tape, const LaunchCfg& lc, cudaStream_t st)
{
    StepArgs<R> a = src;
    a.actions = actions;
    PlanGradArgs<R> q{};
    q.E = s->cfg.num_envs * (int64_t)n_samples;
    q.D = q.E * s->cfg.num_drones;
    q.n_samples = n_samples;
    q.gamma = (R)gamma;
    q.targets = (const R*)targets;
    q.returns = (R*)returns;
    q.done_step = done_step;
    q.grad = (R*)grad;
    q.tape = (R*)tape;
    return launch_plan_grad<R>(a, q, n_steps, lc, st);
}

// the tape of gpd_plan_grad: 13 Reals per copy drone and control step
static int64_t plan_grad_tape_bytes(const gpd_sim* s, int32_t n_steps, int32_t n_samples)
{
    const int64_t D = s->cfg.num_envs * (int64_t)n_samples * s->cfg.num_drones;
    const int64_t rs = s->cfg.precision == GPD_F64 ? 8 : 4;
    if (D > INT64_MAX / 13 / rs / n_steps) return -1;
    return (int64_t)n_steps * 13 * D * rs;
}

extern "C" {

int gpd_version(void) { return GPD_VERSION; }
const char* gpd_last_error(void) { return g_err; }

int gpd_device_count(void)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return fail(GPD_ERR_NO_DEVICE, "cudaGetDeviceCount failed: %s (no CPU fallback exists)", cudaGetErrorString(e));
    return n;
}

int gpd_create(const gpd_config* cfg, gpd_sim** out)
{
    if (!cfg || !out) return fail(GPD_ERR_INVALID, "gpd_create: null argument");
    *out = nullptr;
    if (cfg->num_envs < 1) return fail(GPD_ERR_INVALID, "num_envs must be >= 1");
    if (cfg->num_drones < 1 || cfg->num_drones > GPD_MAX_DRONES_PER_ENV)
        return fail(GPD_ERR_INVALID, "num_drones must be in [1, %d]", GPD_MAX_DRONES_PER_ENV);
    if (cfg->pyb_freq < 1 || cfg->ctrl_freq < 1 || cfg->pyb_freq % cfg->ctrl_freq != 0)
        return fail(GPD_ERR_INVALID, "pyb_freq is not divisible by ctrl_freq");          // BaseAviary.py:79-80
    if (cfg->precision != GPD_F32 && cfg->precision != GPD_F64) return fail(GPD_ERR_INVALID, "bad precision");
    int A = action_width(cfg->action_type);
    if (A < 0) return fail(GPD_ERR_INVALID, "bad action_type");
    const bool ctrl = cfg->env_kind == GPD_ENV_CTRL;
    if (ctrl != (cfg->action_type == GPD_ACT_CTRL_RPM || cfg->action_type == GPD_ACT_CTRL_VEL))
        return fail(GPD_ERR_INVALID, "GPD_ACT_CTRL_RPM / GPD_ACT_CTRL_VEL go with GPD_ENV_CTRL and only with it");
    if (cfg->env_kind == GPD_ENV_HOVER && cfg->num_drones != 1) return fail(GPD_ERR_INVALID, "HoverAviary is single-drone");
    if (cfg->env_kind < GPD_ENV_CTRL || cfg->env_kind > GPD_ENV_MULTIHOVER) return fail(GPD_ERR_INVALID, "bad env_kind");
    if (!ctrl && !cfg->target_pos) return fail(GPD_ERR_INVALID, "target_pos is required for the RL envs");
    const bool pidfam = cfg->action_type == GPD_ACT_PID || cfg->action_type == GPD_ACT_VEL || cfg->action_type == GPD_ACT_ONE_D_PID ||
                        cfg->action_type == GPD_ACT_CTRL_VEL;
    if (pidfam && cfg->drone.model == GPD_RACE)
        return fail(GPD_ERR_INVALID, "no controller is available for the specified drone_model");   // BaseRLAviary.py:77-78
    if ((cfg->physics_flags & ~(GPD_PHY_GND | GPD_PHY_DRAG | GPD_PHY_DW)) != 0) return fail(GPD_ERR_INVALID, "bad physics_flags");
    if (cfg->threads_per_block != 0 && (cfg->threads_per_block % 32 != 0 || cfg->threads_per_block > 256 || cfg->threads_per_block < 32))
        return fail(GPD_ERR_INVALID, "threads_per_block must be a multiple of 32 in [32, 256]");
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(GPD_ERR_NO_DEVICE, "CUDA device %d not available (%d visible)", cfg->device, ndev);
    CU(cudaSetDevice(cfg->device));

    gpd_sim* s = new (std::nothrow) gpd_sim();
    if (!s) return fail(GPD_ERR_ALLOC, "out of host memory");
    s->cfg = *cfg;
    s->A = A;
    s->B = ctrl ? 0 : cfg->ctrl_freq / 2;                                               // BaseRLAviary.py:66
    s->W = ctrl ? 20 : 12 + A * s->B;
    s->S = cfg->pyb_freq / cfg->ctrl_freq;                                              // BaseAviary.py:81
    s->D = cfg->num_envs * (int64_t)cfg->num_drones;
    s->target_host.assign((size_t)cfg->num_drones * 3, 0.0);
    if (cfg->target_pos) memcpy(s->target_host.data(), cfg->target_pos, sizeof(double) * cfg->num_drones * 3);
    s->cfg.target_pos = nullptr;
    // Thread layout: P physics threads (one per drone, whole envs per block) + one DMA/copy warp for the RL envs.
    const int N = cfg->num_drones;
    const bool tma_shape = !ctrl && s->W % 4 == 0 && s->B >= 2 && get_encode_fn() != nullptr &&
                           (A == 4 ? (s->B - 1) * 4 <= 256 : ((A * s->B) % 4 == 0 && A * s->B <= 256));
    bool tma_on = tma_shape;
    int edge_req = -1;                                    // -1: automatic
    {
        const char* ev = getenv("GPD_TMA");
        if (ev && atoi(ev) == 0) tma_on = false;
        ev = getenv("GPD_TMA_EDGE");
        if (ev) edge_req = atoi(ev) ? 1 : 0;
    }
    struct Layout { int P, DPB, EPB, threads, copy, tma, tma_edge, tma_bytes_box, tma_edge_bytes, tma_bytes; int64_t grid; size_t smem; };
    int smem_optin = 227 * 1024;
    cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cfg->device);
    auto make_layout = [&](int P, bool allow_tma = true) {
        Layout L{};
        if (N == 1 && P > 128) P = 128;                   // register budget of the single-drone kernels
        L.DPB = P >= N ? (P / N) * N : N;
        L.P = (L.DPB + 31) / 32 * 32;
        L.EPB = L.DPB / N;
        // the FP64 multi-drone kernels are built for at most 256 threads (128 registers, two CTAs per SM): envs of more than
        // 224 drones run without the DMA warp there (the whole block shares the history copy)
        L.copy = (ctrl || (cfg->precision == GPD_F64 && N > 1 && L.P + 32 > 256)) ? 0 : 32;
        L.threads = L.P + L.copy;
        L.grid = (cfg->num_envs + L.EPB - 1) / L.EPB;
        const bool tma = allow_tma && tma_on && L.DPB <= 256 && L.copy > 0;
        L.tma = tma ? 1 : 0;
        // whole-sector split of the row between the drone's thread and TMA (the two old slots the thread needs arrive
        // through two extra 16-byte-wide TMA boxes): no read-modify-write of half-written sectors in ECC HBM.  Measured
        // +10 % at >= 1 M drones, +4 % at 131,072, +2 % at 65,536, -3 % at <= 32,768 (latency-bound: the physics threads
        // then wait on the mbarrier and one more block barrier)
        const bool edge_ok = tma && A == 4 && (s->W / 4) % 2 == 0 && s->B >= 4;
        L.tma_edge = edge_ok && (edge_req < 0 ? s->D >= 65536 : edge_req == 1) ? 1 : 0;
        L.tma_bytes_box = !tma ? 0 : (A == 4 ? L.DPB * (s->B - 1 - 2 * L.tma_edge) * 16 : L.DPB * A * s->B * 4);
        L.tma_edge_bytes = L.tma_edge ? (L.DPB * 16 + 127) / 128 * 128 : 0;
        L.tma_bytes = (L.tma_bytes_box + 127) / 128 * 128 + 2 * L.tma_edge_bytes;
        L.smem = (size_t)L.tma_bytes + smem_bytes(cfg->precision == GPD_F64, ctrl, N > 1, L.DPB, L.EPB);
        return L;
    };
    // defaults (measured, profiles/README.md): 64 physics threads for the lean FP32 single-drone kernel (64 registers: more,
    // smaller CTAs balance better over 148 SMs) and for A < 4, 128 for the other single-drone kernels; multi-drone envs
    // 224 (+ the DMA warp = 256), 64 with downwash
    const bool f64 = cfg->precision == GPD_F64;
    const bool rpm_like = cfg->action_type == GPD_ACT_RPM || cfg->action_type == GPD_ACT_ONE_D_RPM || cfg->action_type == GPD_ACT_CTRL_RPM;
    const bool lean = rpm_like && cfg->physics_flags == 0;
    int P0 = 64;
    if (N == 1) P0 = (A == 4 && (f64 || !lean)) ? 128 : 64;      // A < 4: the 32 funnel-copy lanes limit the tile to 64 rows
    else P0 = (cfg->physics_flags & GPD_PHY_DW) ? 64 : 224;     // downwash: two block barriers per substep favour small CTAs
                                                                // (512 envs x 64 drones: 17.4 us at 64 threads, 24.1 at 128)
    // multi-drone RL envs without downwash run the bulk kernel (tiles of at most 128 drones, whole envs): that fixes the tile
    // size, the wave search below is for gpd::step_kernel
    bool multi_bulk = false;
    {
        const char* bv = getenv("GPD_BULK");
        multi_bulk = N > 1 && N <= 128 && !ctrl && !(cfg->physics_flags & GPD_PHY_DW) && (12 + A * (cfg->ctrl_freq / 2)) % 4 == 0 &&
                     (bv ? atoi(bv) != 0 : (12 + A * (cfg->ctrl_freq / 2)) * 4 <= 512);
        if (multi_bulk) P0 = 128;
    }
    // lean FP32 sims on the bulk kernel: 128-env tiles in the range where launches are sequenced per tile and still give every SM
    // two CTAs of two tiles each (profiles/r02/sweep_b14/b16.jsonl, two tiles per CTA: 65,536 envs 7.74 us with 128-env tiles,
    // 8.12 us with 64; 16,384 envs 3.42 vs 3.28 us; 262,144 envs equal; 524,288 envs 68.4 vs 65.5 us, 1 M envs 124.6 vs 121.9 us)
    if (N == 1 && A == 4 && !f64 && lean && !ctrl && s->D >= 4 * 148 * 64 && s->D <= 262144) P0 = 128;
    Layout L = make_layout(cfg->threads_per_block ? cfg->threads_per_block : P0);
    // a history tile beyond the shared-memory limit (e.g. 256 drones per env with a 60-slot ring): register-copy path instead
    if (L.smem > (size_t)smem_optin) L = make_layout(cfg->threads_per_block ? cfg->threads_per_block : P0, false);
    if (!cfg->threads_per_block && !multi_bulk) {
        // Wave quantisation: a launch of 1..4 waves pays for its partly filled last wave (MultiHover x2 FP32 at 32,768
        // envs: 512 CTAs on 444 slots = 28.5 us, 293 CTAs on 296 slots = 19.5 us).  Take the block size with the fewest
        // waves; the default wins ties.
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
        auto waves = [&](const Layout& l, double& fill) {
            const int b = cfg->precision == GPD_F64
                ? step_blocks_per_sm<double>(cfg->action_type, cfg->physics_flags, N, A, s->W, cfg->env_kind, l.threads, l.smem)
                : step_blocks_per_sm<float>(cfg->action_type, cfg->physics_flags, N, A, s->W, cfg->env_kind, l.threads, l.smem);
            if (b <= 0) { fill = 0; return (int64_t)1 << 40; }
            const int64_t slots = (int64_t)b * sms, w = (l.grid + slots - 1) / slots;
            fill = (double)l.grid / (double)(w * slots);
            return w;
        };
        double fill0 = 0;
        const int64_t w0 = waves(L, fill0);
        if (w0 > 1 && w0 <= 4) {
            int64_t wb = w0;
            for (int P = 64; P <= (N == 1 ? 128 : 256); P += 32) {      // 32-thread CTAs always lose (measured)
                if (P < N) continue;
                Layout c = make_layout(P);
                if (c.smem > (size_t)smem_optin) continue;
                double f = 0;
                const int64_t w = waves(c, f);
                if (getenv("GPD_DEBUG_LAYOUT"))
                    fprintf(stderr, "[gpd]   candidate P=%d threads=%d smem=%zu grid=%lld waves=%lld fill=%.2f\n", c.P, c.threads, c.smem,
                            (long long)c.grid, (long long)w, f);
                if (w < wb) { wb = w; L = c; }
            }
        }
        if (getenv("GPD_DEBUG_LAYOUT"))
            fprintf(stderr, "[gpd] layout: %d physics threads, grid %lld, %lld wave(s) (default: %lld), smem %zu\n", L.P,
                    (long long)L.grid, (long long)waves(L, fill0), (long long)w0, L.smem);
    }
    const int DPB = L.DPB, EPB = L.EPB;
    s->copy_threads = L.copy;
    s->lc.threads = L.threads;
    s->dpb = DPB;
    s->lc.grid = L.grid;
    s->tma_ok = L.tma != 0;
    s->tma_edge = L.tma_edge;
    s->tma_bytes_box = L.tma_bytes_box;
    s->tma_edge_bytes = L.tma_edge_bytes;
    s->tma_bytes = L.tma_bytes;
    s->lc.smem = L.smem;
    (void)EPB;
    s->d_pad = s->lc.grid * (int64_t)DPB;
    {   // bulk-copy data path: same tiles (DPB envs per CTA), T threads, everything staged in shared memory
        const size_t rs = f64 ? 8 : 4;
        // what bypasses shared memory (BulkSmem in gpd_step_bulk.cuh): shared memory per env bounds the tiles in flight per SM
        // measured (profiles/r02, 65,536 envs, FP32, 200-step windows): 8.95 / 8.77 / 8.62 us for direct = 0 / 1 / 2
        // (FP64 13.74 -> 13.31 us; 1 M envs unchanged within noise): default 2
        int direct = 2;
        if (const char* dv = getenv("GPD_BULK_DIRECT")) direct = atoi(dv) < 0 ? 0 : (atoi(dv) > 2 ? 2 : atoi(dv));
        s->bulk_direct = direct;
        // two tiles per CTA for chained FP32 launches that still leave >= 1.5 CTAs per SM (FP64: 13.2 us with one tile, 13.9 with two)
        s->bulk_tpc = (!f64 && L.grid >= 3 * 148) ? 2 : 1;
        if (const char* tv = getenv("GPD_BULK_TPC")) s->bulk_tpc = atoi(tv) < 1 ? 1 : (atoi(tv) > GPD_BULK_MAX_TPC ? GPD_BULK_MAX_TPC : atoi(tv));
        const size_t bsm = (size_t)DPB * s->W * 4 + (direct >= 2 ? 0 : 3 * (size_t)DPB * 4 * rs) +
                           (direct ? 0 : (size_t)DPB * 16 + 2 * (size_t)DPB * rs + 2 * (size_t)DPB * 4 + 2 * (size_t)DPB) + 8 * 32 +
                           (N > 1 ? 2 * (size_t)DPB * rs + (size_t)DPB * 4 + (size_t)(DPB / N) * 4 + 16 : 0);     // per-env reduction scratch
        // Eligible: single-drone RL env, 4-wide actions, whole-float4 rows, 16-row-aligned tiles that fit shared memory.
        // Default on for rows of at most 512 bytes (30 Hz: W = 72, 48 Hz: W = 108): measured 9.2 -> 8.6 us (FP32),
        // 16.1 -> 13.3 us (FP64) at 65,536 envs, 131 -> 121 us at 1 M envs, and at 48 Hz 11.35 -> 10.79 us once the state
        // vectors bypass shared memory (direct = 2; with everything staged the TMA-box kernel was ahead there).  Longer rows
        // (60 Hz and up) leave too few tiles per SM.  GPD_BULK=1 forces it where eligible, GPD_BULK=0 turns it off.
        const char* ev = getenv("GPD_BULK");
        // narrower actions (PID: A = 3, ONE_D_*: A = 1) slide their rows inside shared memory and take their actions per thread
        // multi-drone envs (MultiHover) too, unless downwash is on (two block barriers per substep: gpd::step_kernel); their
        // per-env arrays are written by the env's first drone, so they need direct == 2 like the narrow actions
        const bool eligible = !ctrl && s->W % 4 == 0 && DPB <= 128 && bsm <= (size_t)smem_optin &&
                              (N == 1 ? DPB % 16 == 0 && (A == 4 || direct == 2)
                                      : direct == 2 && DPB % N == 0 && !(cfg->physics_flags & GPD_PHY_DW));
        s->bulk_ok = eligible && (ev ? atoi(ev) != 0 : s->W * 4 <= 512);
        s->lc_bulk.threads = (DPB + 31) / 32 * 32; s->lc_bulk.grid = L.grid; s->lc_bulk.smem = bsm; s->lc_bulk.pdl = 0;   // whole warps
    }
    int bps_dbg = 0;
    double waves_dbg = 0;
    {   // programmatic dependent launch: measured to help only launches of at most ~2 CTAs per SM (the CTA launch and the
        // parameter fetch overlap the previous kernel's tail); with a full wave the early-resident CTAs all issue their
        // loads at the same instant after the wait and the burst costs more than the overlap gains
        // Per-CTA step sequencing (no whole-grid wait; every step kernel launched programmatically, so consecutive steps
        // overlap across the kernel boundary) pays one L2 round trip at each end of a CTA's life.  Measured (profiles/r02):
        // 65,536 envs 10.5 -> 9.2 us, FP64 23.9 -> 16.1 us, C3 35.0 -> 27.6 us, 262,144 envs 36.5 -> 35.2 us, but
        // 1 M envs 130.9 -> 134.1 us and C5 (2 M envs) 439 -> 457 us: with many waves the boundary is a small share of the
        // launch and the round trips cost more than the overlap gains.  Default: on for launches of at most 4 waves.
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
        int bps;
        if (s->bulk_ok)
            bps = cfg->precision == GPD_F64
                ? step_bulk_blocks_per_sm<double>(cfg->action_type, cfg->physics_flags, N, s->lc_bulk.threads, s->lc_bulk.smem)
                : step_bulk_blocks_per_sm<float>(cfg->action_type, cfg->physics_flags, N, s->lc_bulk.threads, s->lc_bulk.smem);
        else
            bps = cfg->precision == GPD_F64
                ? step_blocks_per_sm<double>(cfg->action_type, cfg->physics_flags, N, A, s->W, cfg->env_kind, s->lc.threads, s->lc.smem)
                : step_blocks_per_sm<float>(cfg->action_type, cfg->physics_flags, N, A, s->W, cfg->env_kind, s->lc.threads, s->lc.smem);
        const double waves = bps > 0 ? (double)s->lc.grid / ((double)bps * sms) : 1e9;
        const char* td = getenv("GPD_TILE_DEP");
        s->tile_dep = td ? (atoi(td) != 0 ? 1 : 0) : (waves <= 4.0 ? 1 : 0);
        const char* ev = getenv("GPD_PDL");
        s->lc.pdl = ev ? atoi(ev) : ((s->tile_dep || s->lc.grid <= 296) ? 1 : 0);
        s->lc_bulk.pdl = s->lc.pdl;
        bps_dbg = bps; waves_dbg = waves;
    }
    if (s->lc.grid > 0x7fffffffLL) { delete s; return fail(GPD_ERR_INVALID, "too many envs for one launch"); }
    int rc = cfg->precision == GPD_F64 ? build_args(s, s->a64) : build_args(s, s->a32);
    if (rc == GPD_OK && getenv("GPD_DEBUG_LAYOUT"))      // one line per handle: every create-time choice of the step's data path
        fprintf(stderr, "[gpd] %d CTAs/SM, %.2f waves: tile_dep %d, pdl %d, bulk path %d, tile %d, tiles %lld, tma %d, tma_edge %d, "
                "bulk_tpc %d, state_in_obs %d\n", bps_dbg, waves_dbg, s->tile_dep, s->lc.pdl, (int)s->bulk_ok, s->dpb,
                (long long)s->lc.grid, (int)s->tma_ok, s->tma_edge, s->bulk_tpc, s->a32.state_in_obs);
    if (rc == GPD_OK) { cudaError_t e = cudaMalloc((void**)&s->stats_out, 8 * sizeof(double)); if (e != cudaSuccess) rc = fail(GPD_ERR_ALLOC, "cudaMalloc failed"); }
    if (rc != GPD_OK) { gpd_destroy(s); return rc; }
    // start in the reset state (BaseAviary.__init__ ends with _housekeeping + _updateAndStoreKinematicInformation)
    rc = gpd_reset(s, nullptr, nullptr, nullptr, nullptr);
    if (rc == GPD_OK) { cudaError_t e = cudaDeviceSynchronize(); if (e != cudaSuccess) rc = fail(GPD_ERR_CUDA, "initial reset failed: %s", cudaGetErrorString(e)); }
    if (rc != GPD_OK) { gpd_destroy(s); return rc; }
    *out = s;
    return GPD_OK;
}

void gpd_destroy(gpd_sim* s)
{
    if (!s) return;
    cudaSetDevice(s->cfg.device);
    cudaDeviceSynchronize();
    for (void* p : s->allocs) cudaFree(p);
    cudaFree(s->h_act); cudaFree(s->h_obs[0]); cudaFree(s->h_obs[1]);
    cudaFree(s->h_tkin); cudaFree(s->h_mask); cudaFree(s->stats_out); cudaFree(s->stats_gather);
    cudaFree(s->init_bufs[0]); cudaFree(s->init_bufs[1]); cudaFree(s->target_buf);
    cudaFree(s->mir.d_kin_t); cudaFree(s->mir.d_full_t);
    delete s;
}

int gpd_obs_width(const gpd_sim* s) { return s ? s->W : fail(GPD_ERR_INVALID, "null handle"); }
int gpd_action_width(const gpd_sim* s) { return s ? s->A : fail(GPD_ERR_INVALID, "null handle"); }
int gpd_substeps(const gpd_sim* s) { return s ? s->S : fail(GPD_ERR_INVALID, "null handle"); }

int gpd_set_init_poses(gpd_sim* s, const double* xyz, const double* rpy, int per_env)
{
    if (!s || !xyz || !rpy) return fail(GPD_ERR_INVALID, "gpd_set_init_poses: null argument");
    CU(use_device(s->cfg.device));
    unchain(s, nullptr, true);
    return s->cfg.precision == GPD_F64 ? upload_init(s, s->a64, xyz, rpy, per_env) : upload_init(s, s->a32, xyz, rpy, per_env);
}

int gpd_set_targets(gpd_sim* s, const double* target_pos, int per_env)
{
    if (!s || !target_pos) return fail(GPD_ERR_INVALID, "gpd_set_targets: null argument");
    if (s->cfg.env_kind == GPD_ENV_CTRL) return fail(GPD_ERR_INVALID, "the Ctrl env has no target");
    CU(use_device(s->cfg.device));
    unchain(s, nullptr, true);
    return s->cfg.precision == GPD_F64 ? upload_targets(s, s->a64, target_pos, per_env) : upload_targets(s, s->a32, target_pos, per_env);
}

int gpd_reset(gpd_sim* s, const uint8_t* env_mask, const void* obs_prev, void* obs_out, void* stream)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    if (obs_out && obs_out == obs_prev) return fail(GPD_ERR_INVALID, "obs_prev must not alias obs_out");
    CU(use_device(s->cfg.device));
    unchain(s, stream);
    int rc = sync_state(s, stream);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (s->cfg.precision == GPD_F64) {
        StepArgs<double> a = s->a64;
        a.reset_mask = env_mask; a.obs_prev = (const float*)obs_prev; a.obs_out = obs_out;
        CU(launch_reset<double>(a, s->lc, st));
    } else {
        StepArgs<float> a = s->a32;
        a.reset_mask = env_mask; a.obs_prev = (const float*)obs_prev; a.obs_out = obs_out;
        CU(launch_reset<float>(a, s->lc, st));
    }
    if (obs_out) { s->last_obs = obs_out; ++s->obs_seq; }
    return GPD_OK;
}

// the bulk copies need 16-byte aligned actions / observations (see step_impl)
static bool bulk_step(const gpd_sim* s, const void* actions, const void* obs_prev, const void* obs_out)
{
    return s->bulk_ok && (((uintptr_t)actions | (uintptr_t)obs_prev | (uintptr_t)obs_out) & 15) == 0;
}

// Chained-state handles: the bulk step takes position and velocity of a chained tile from obs_prev, which must then be the
// observation this handle wrote last (or was given through gpd_note_latest_obs).  Any other step, or one on the per-thread
// kernel, must first move the state back into the arrays (sync_state), on a stream the whole step is ordered behind.
static bool step_needs_sync(const gpd_sim* s, const void* actions, const void* obs_prev, const void* obs_out)
{
    return s->a32.state_in_obs && (!bulk_step(s, actions, obs_prev, obs_out) || obs_prev != s->last_obs);
}

static int step_impl(gpd_sim* s, const void* actions, const void* obs_prev, void* obs_out, void* reward, uint8_t* terminated,
                     uint8_t* truncated, void* terminal_kin, float* kin_t, void* stream, int64_t kin_ld = 0,
                     bool host_io = false)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    if (!actions || !obs_out) return fail(GPD_ERR_INVALID, "gpd_step: actions and obs_out are required");
    if (obs_out == obs_prev) return fail(GPD_ERR_INVALID, "obs_prev must not alias obs_out");
    CU(use_device(s->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    CUtensorMap tp, to, te;
    bool have = false;
    // actions or observations that are not 16-byte aligned (step_into on offset views) take the per-thread kernel's scalar
    // variant (launch_step), which has no TMA path for 4-wide actions
    const bool al16 = (((uintptr_t)actions | (uintptr_t)obs_prev | (uintptr_t)obs_out) & 15) == 0;
    if (s->tma_ok && obs_prev && al16) {
        have = get_tmap(s, obs_prev, false, &tp) && get_tmap(s, obs_out, false, &to);
        if (have && s->tma_edge) have = get_tmap(s, obs_prev, true, &te);
    }
    const int use_tma = have ? 1 : 0;
    // the bulk copies need 16-byte aligned actions / observations (torch allocations and their rows are); anything else takes
    // the per-thread kernel.  Reward / flag arrays that are not (rows of a [T][E] uint8 trajectory buffer) only switch those
    // three outputs to plain stores: a sim keeps ONE kernel, so its FP32 results do not depend on the caller's buffer layout
    // (the two kernels agree bit for bit in FP64; in FP32 only up to the compiler's FMA contraction choices).
    const uintptr_t al_out = (uintptr_t)reward | (uintptr_t)terminated | (uintptr_t)truncated;
    const bool bulk = bulk_step(s, actions, obs_prev, obs_out);
    if (step_needs_sync(s, actions, obs_prev, obs_out)) {
        int rc = sync_state(s, stream);
        if (rc) return rc;
        unchain(s, stream);
    }
    const int out_plain = ((al_out & 15) != 0 || host_io) ? 1 : 0;     // outputs in mapped host memory: plain stores by the threads
    LaunchCfg lc = bulk ? s->lc_bulk : s->lc;
    const void* prev_sim = nullptr;     // handle of the step kernel this one is chained behind
    if (s->tile_dep) {
        // programmatic launch only when the caller opted in (gpd_set_step_chaining) and the library's previous launch on this
        // stream was a step kernel; otherwise plain stream order (the kernel still claims / publishes its tiles, so a
        // chained successor sequences correctly behind it)
        lc.pdl = (s->chaining && lc.pdl && g_chain.get(s->cfg.device, st, capture_id(st), &prev_sim)) ? 1 : 0;
    }
    // tiles of this launch and tiles per CTA (bulk kernel).  A launch chained behind a step of ANOTHER handle (independent env
    // sets in rotation) folds bulk_tpc tiles into one CTA (one buffer, claims up front, a tile published under the next tile's
    // loads: gpd_step_bulk.cuh): 8.6 -> 7.7 us per 65,536-env step.  One tile per CTA otherwise: alone on the machine a grid of
    // fewer, longer CTAs is only slower, and behind a step of the SAME handle the tiles depend on each other one to one, so the
    // finer grain overlaps better (7.1 vs 8.5 us).  The per-tile words make the two mappings interchangeable.
    const int64_t tiles = lc.grid;
    int tpc = 1;
    if (bulk && s->tile_dep && lc.pdl && s->bulk_tpc > 1 && prev_sim != (const void*)s) {
        tpc = s->bulk_tpc;
        lc.grid = (tiles + tpc - 1) / tpc;
    }
    if (s->cfg.precision == GPD_F64) {
        StepArgs<double> a = s->a64;
        a.actions = actions; a.obs_prev = (const float*)obs_prev; a.obs_out = obs_out; a.reward = (double*)reward;
        a.terminated = terminated; a.truncated = truncated; a.terminal_kin = (float*)terminal_kin; a.use_tma = use_tma;
        a.kin_t = kin_t; a.kin_ld = kin_ld > 0 ? kin_ld : s->D; a.out_plain = out_plain;
        a.tpc = tpc; a.tile_end = (int32_t)tiles;
        if (bulk) CU(launch_step_bulk<double>(a, lc, st));
        else CU(launch_step<double>(a, lc, have ? &tp : nullptr, have ? &to : nullptr, have && s->tma_edge ? &te : nullptr, st));
    } else {
        StepArgs<float> a = s->a32;
        a.actions = actions; a.obs_prev = (const float*)obs_prev; a.obs_out = obs_out; a.reward = (float*)reward;
        a.terminated = terminated; a.truncated = truncated; a.terminal_kin = (float*)terminal_kin; a.use_tma = use_tma;
        a.kin_t = kin_t; a.kin_ld = kin_ld > 0 ? kin_ld : s->D; a.out_plain = out_plain;
        a.tpc = tpc; a.tile_end = (int32_t)tiles;
        if (bulk) CU(launch_step_bulk<float>(a, lc, st));
        else CU(launch_step<float>(a, lc, have ? &tp : nullptr, have ? &to : nullptr, have && s->tma_edge ? &te : nullptr, st));
    }
    s->last_obs = obs_out;
    ++s->obs_seq;
    g_chain.set(s->cfg.device, st, true, capture_id(st), s);
    return GPD_OK;
}

int gpd_set_step_chaining(gpd_sim* s, int enable)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    s->chaining = enable ? 1 : 0;
    return GPD_OK;
}

int gpd_step(gpd_sim* s, const void* actions, const void* obs_prev, void* obs_out,
             void* reward, uint8_t* terminated, uint8_t* truncated, void* terminal_kin, void* stream)
{
    return step_impl(s, actions, obs_prev, obs_out, reward, terminated, truncated, terminal_kin, nullptr, stream);
}

// ---- host-buffer paths -------------------------------------------------------------------------------------------------
struct HostSizes { size_t rs, act_b, obs_b, obs_pad, pack_b, E, rew_pad, flag_pad; };
static HostSizes host_sizes(const gpd_sim* s)
{
    HostSizes z;
    const bool ctrl = s->cfg.env_kind == GPD_ENV_CTRL;
    z.rs = s->cfg.precision == GPD_F64 ? 8 : 4;
    z.act_b = (size_t)s->D * s->A * (ctrl ? z.rs : 4);
    z.obs_b = (size_t)s->D * s->W * (ctrl ? z.rs : 4);
    z.E = (size_t)s->cfg.num_envs;
    z.obs_pad = (z.obs_b + 15) & ~size_t(15);     // keeps the reward block aligned for Real stores
    z.pack_b = z.obs_pad + z.E * z.rs + 2 * z.E;
    z.rew_pad = (z.E * z.rs + 15) & ~size_t(15);  // mirror staging: reward | terminated | truncated, each 16-byte aligned
    z.flag_pad = (z.E + 15) & ~size_t(15);
    return z;
}

// Device staging of the host paths, all-or-nothing: a failed allocation leaves the handle exactly as it was.
static int ensure_host_path(gpd_sim* s)
{
    if (s->h_obs[0]) return GPD_OK;
    const HostSizes z = host_sizes(s);
    // each ping-pong slot is one packed block [obs | reward | terminated | truncated]: when the caller's host arrays are
    // laid out the same way (the Python facade allocates them so) the whole result travels in ONE device-to-host copy
    void *act = nullptr, *o0 = nullptr, *o1 = nullptr, *tk = nullptr, *mk = nullptr;
    cudaError_t e = cudaMalloc(&act, z.act_b);
    if (e == cudaSuccess) e = cudaMalloc(&o0, z.pack_b + 64);
    if (e == cudaSuccess) e = cudaMalloc(&o1, z.pack_b + 64);
    if (e == cudaSuccess) e = cudaMalloc(&tk, (size_t)s->D * 12 * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&mk, z.E);
    if (e == cudaSuccess) e = cudaMemset(tk, 0, (size_t)s->D * 12 * sizeof(float));
    if (e != cudaSuccess) {
        cudaFree(act); cudaFree(o0); cudaFree(o1); cudaFree(tk); cudaFree(mk);
        return fail(GPD_ERR_ALLOC, "host-path staging allocation failed: %s", cudaGetErrorString(e));
    }
    s->h_act = act; s->h_obs[0] = o0; s->h_obs[1] = o1; s->h_tkin = (float*)tk; s->h_mask = (uint8_t*)mk;
    return GPD_OK;
}

int gpd_step_host(gpd_sim* s, const void* actions, void* obs_out, void* reward,
                  uint8_t* terminated, uint8_t* truncated, void* terminal_kin, void* stream)
{
    if (!s || !actions || !obs_out) return fail(GPD_ERR_INVALID, "gpd_step_host: null argument");
    CU(use_device(s->cfg.device));
    int rc = ensure_host_path(s);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const HostSizes z = host_sizes(s);
    CU(cudaMemcpyAsync(s->h_act, actions, z.act_b, cudaMemcpyHostToDevice, st));
    int nxt = s->h_cur ^ 1;
    char* pack = (char*)s->h_obs[nxt];
    void* d_rew = pack + z.obs_pad;
    uint8_t* d_term = (uint8_t*)(pack + z.obs_pad + z.E * z.rs);
    uint8_t* d_trunc = d_term + z.E;
    rc = gpd_step(s, s->h_act, s->h_has_prev ? s->h_obs[s->h_cur] : nullptr, s->h_obs[nxt], d_rew, d_term, d_trunc,
                  terminal_kin ? s->h_tkin : nullptr, stream);
    if (rc) return rc;
    s->h_cur = nxt; s->h_has_prev = true;
    const bool packed = reward == (char*)obs_out + z.obs_pad && (void*)terminated == (char*)reward + z.E * z.rs &&
                        truncated == terminated + z.E;
    if (packed) {
        CU(cudaMemcpyAsync(obs_out, pack, z.pack_b, cudaMemcpyDeviceToHost, st));
    } else {
        CU(cudaMemcpyAsync(obs_out, pack, z.obs_b, cudaMemcpyDeviceToHost, st));
        if (reward) CU(cudaMemcpyAsync(reward, d_rew, z.E * z.rs, cudaMemcpyDeviceToHost, st));
        if (terminated) CU(cudaMemcpyAsync(terminated, d_term, z.E, cudaMemcpyDeviceToHost, st));
        if (truncated) CU(cudaMemcpyAsync(truncated, d_trunc, z.E, cudaMemcpyDeviceToHost, st));
    }
    if (terminal_kin) CU(cudaMemcpyAsync(terminal_kin, s->h_tkin, (size_t)s->D * 12 * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return GPD_OK;
}

int gpd_reset_host(gpd_sim* s, const uint8_t* env_mask, void* obs_out, void* stream)
{
    if (!s || !obs_out) return fail(GPD_ERR_INVALID, "gpd_reset_host: null argument");
    CU(use_device(s->cfg.device));
    int rc = ensure_host_path(s);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const HostSizes z = host_sizes(s);
    if (env_mask) CU(cudaMemcpyAsync(s->h_mask, env_mask, z.E, cudaMemcpyHostToDevice, st));
    int nxt = s->h_cur ^ 1;
    rc = gpd_reset(s, env_mask ? s->h_mask : nullptr, s->h_has_prev ? s->h_obs[s->h_cur] : nullptr, s->h_obs[nxt], stream);
    if (rc) return rc;
    s->h_cur = nxt; s->h_has_prev = true;
    CU(cudaMemcpyAsync(obs_out, s->h_obs[nxt], z.obs_b, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return GPD_OK;
}

// ---- host mirror (see struct Mirror) -----------------------------------------------------------------------------------
int gpd_mirror_alloc(int64_t rows, int64_t row_len, float** log_out)
{
    if (!log_out || rows < 1 || row_len < 1) return fail(GPD_ERR_INVALID, "gpd_mirror_alloc: bad argument");
    *log_out = nullptr;
    void* p = nullptr;
    const size_t bytes = (size_t)rows * (size_t)row_len * sizeof(float);
    cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable | cudaHostAllocMapped);
    if (e != cudaSuccess)
        return fail(e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver ? GPD_ERR_NO_DEVICE : GPD_ERR_ALLOC,
                    "cudaHostAlloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    memset(p, 0, bytes);
    *log_out = (float*)p;
    return GPD_OK;
}

int gpd_mirror_free(float* log)
{
    if (log) CU(cudaFreeHost(log));
    return GPD_OK;
}

int gpd_mirror_attach(gpd_sim* s, float* log, int64_t rows, int64_t row_len, int64_t col0)
{
    if (!s || !log) return fail(GPD_ERR_INVALID, "gpd_mirror_attach: null argument");
    if (s->cfg.env_kind == GPD_ENV_CTRL)
        return fail(GPD_ERR_INVALID, "the Ctrl observation has no action ring: use gpd_step_host (every byte of it is device-computed)");
    if (rows < s->W + s->A || col0 < 0 || row_len < col0 + s->D)
        return fail(GPD_ERR_INVALID, "gpd_mirror_attach: the log needs at least W + A = %d rows and col0 + D = %lld columns",
                    s->W + s->A, (long long)(col0 + s->D));
    CU(use_device(s->cfg.device));
    int rc = ensure_host_path(s);
    if (rc) return rc;
    if (!s->mir.d_kin_t) {
        void* k = nullptr;
        cudaError_t e = cudaMalloc(&k, (size_t)12 * s->D * sizeof(float));
        if (e != cudaSuccess) return fail(GPD_ERR_ALLOC, "cudaMalloc failed: %s", cudaGetErrorString(e));
        s->mir.d_kin_t = (float*)k;
    }
    Mirror& m = s->mir;
    m.log = log; m.rows = rows; m.ld = row_len; m.col0 = col0;
    m.row = 0; m.valid = false; m.pending = false;
    {
        void* dl = nullptr;
        m.d_log = (cudaHostGetDevicePointer(&dl, log, 0) == cudaSuccess) ? (float*)dl : nullptr;
        if (!m.d_log) cudaGetLastError();
        if (const char* ev = getenv("GPD_MIRROR_ZEROCOPY")) m.zero_copy = atoi(ev) != 0;
    }
    return GPD_OK;
}

int64_t gpd_mirror_row(const gpd_sim* s)
{
    if (!s || !s->mir.log) return fail(GPD_ERR_INVALID, "no host mirror attached");
    return s->mir.row;
}

// Device alias of a caller's host pointer when the memory is pinned and mapped (cudaHostAlloc / cudaHostRegister, e.g. torch's
// pin_memory), else nullptr.  Asked every step (~1 us per call): a cached answer could outlive the caller's allocation.
static void* host_alias(const void* host)
{
    if (!host) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost) return at.devicePointer;
    cudaGetLastError();
    return nullptr;
}

// device [nrows][D] (contiguous) -> log rows [row0, row0 + nrows), this handle's columns
static cudaError_t mirror_rows_d2h(gpd_sim* s, int64_t row0, const float* d_src, int nrows, cudaStream_t st)
{
    Mirror& m = s->mir;
    float* dst = m.log + row0 * m.ld + m.col0;
    if (m.ld == s->D)
        return cudaMemcpyAsync(dst, d_src, (size_t)nrows * s->D * sizeof(float), cudaMemcpyDeviceToHost, st);
    return cudaMemcpy2DAsync(dst, (size_t)m.ld * sizeof(float), d_src, (size_t)s->D * sizeof(float), (size_t)s->D * sizeof(float),
                             (size_t)nrows, cudaMemcpyDeviceToHost, st);
}

// Rebuilds the window rows [row, row + W) from a device observation (or zeroes the ring when there is none yet).
static int mirror_refresh(gpd_sim* s, const void* d_obs, int64_t row, cudaStream_t st)
{
    Mirror& m = s->mir;
    if (!d_obs) {       // no observation yet: all-zero ring (BaseRLAviary.py:153-154); the kin rows are written by the step
        CU(cudaStreamSynchronize(st));
        for (int64_t r = row; r < row + s->W; ++r) memset(m.log + r * m.ld + m.col0, 0, (size_t)s->D * sizeof(float));
        return GPD_OK;
    }
    if (!m.d_full_t) {
        void* f = nullptr;
        cudaError_t e = cudaMalloc(&f, (size_t)s->W * s->D * sizeof(float));
        if (e != cudaSuccess) return fail(GPD_ERR_ALLOC, "cudaMalloc failed: %s", cudaGetErrorString(e));
        m.d_full_t = (float*)f;
    }
    CU(launch_transpose_cols((const float*)d_obs, s->D, s->W, 0, s->W, m.d_full_t, s->D, st));
    CU(mirror_rows_d2h(s, row, m.d_full_t, s->W, st));
    return GPD_OK;
}

// newest action, host -> host: actions[d][A] into the A log rows that follow the window (transposed; streaming stores)
static void mirror_write_action(const gpd_sim* s, const float* act, int64_t row)
{
    const Mirror& m = s->mir;
    const int64_t D = s->D;
    const int A = s->A;
    float* r0 = m.log + row * m.ld + m.col0;
    if (A == 4 && ((uintptr_t)act & 15) == 0 && ((uintptr_t)r0 & 15) == 0 && (m.ld & 3) == 0) {
        float *q0 = r0, *q1 = r0 + m.ld, *q2 = r0 + 2 * m.ld, *q3 = r0 + 3 * m.ld;
        int64_t d = 0;
        for (; d + 4 <= D; d += 4) {
            __m128 a0 = _mm_load_ps(act + 4 * d), a1 = _mm_load_ps(act + 4 * d + 4), a2 = _mm_load_ps(act + 4 * d + 8),
                   a3 = _mm_load_ps(act + 4 * d + 12);
            _MM_TRANSPOSE4_PS(a0, a1, a2, a3);
            _mm_stream_ps(q0 + d, a0); _mm_stream_ps(q1 + d, a1); _mm_stream_ps(q2 + d, a2); _mm_stream_ps(q3 + d, a3);
        }
        for (; d < D; ++d) { q0[d] = act[4 * d]; q1[d] = act[4 * d + 1]; q2[d] = act[4 * d + 2]; q3[d] = act[4 * d + 3]; }
        _mm_sfence();
        return;
    }
    for (int k = 0; k < A; ++k) {
        float* q = r0 + (int64_t)k * m.ld;
        for (int64_t d = 0; d < D; ++d) q[d] = act[d * A + k];
    }
}

int gpd_step_mirror_begin(gpd_sim* s, const void* actions, const void* d_obs_prev, void* d_obs_out, void* reward,
                          uint8_t* terminated, uint8_t* truncated, void* terminal_kin, void* stream)
{
    if (!s || !actions) return fail(GPD_ERR_INVALID, "gpd_step_mirror: null argument");
    Mirror& m = s->mir;
    if (!m.log) return fail(GPD_ERR_INVALID, "gpd_step_mirror: no host mirror attached (gpd_mirror_attach)");
    if (m.pending) return fail(GPD_ERR_INVALID, "gpd_step_mirror_begin: the previous step was not completed (gpd_step_mirror_end)");
    CU(use_device(s->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const HostSizes z = host_sizes(s);
    const bool internal = d_obs_out == nullptr;      // NULL: the handle's own observation ping-pong
    int nxt = s->h_cur ^ 1;
    if (internal) {
        d_obs_prev = s->h_has_prev ? s->h_obs[s->h_cur] : nullptr;
        d_obs_out = s->h_obs[nxt];
    }
    // window maintenance: out of room -> back to row 0 (compaction); stale (the device chain moved without the mirror) -> in place
    const bool in_sync = m.valid && m.synced_seq == s->obs_seq && m.synced_obs == d_obs_prev;
    const bool no_room = m.row + s->A + s->W > m.rows;
    if (no_room || !in_sync) {
        if (no_room) m.row = 0;
        int rc = mirror_refresh(s, d_obs_prev, m.row, st);
        if (rc) return rc;
    }
    char* pack = (char*)s->h_obs[nxt] + z.obs_pad;    // reward / flags staging lives behind the internal observation slot
    void* d_rew = pack;
    const bool tight = z.rew_pad == z.E * z.rs && z.flag_pad == z.E;     // E % 16 == 0: the staging is [reward|term|trunc] packed
    uint8_t* d_term = (uint8_t*)(pack + z.rew_pad);
    uint8_t* d_trunc = d_term + z.flag_pad;
    // Zero-copy step: when the caller's arrays are pinned (the facade allocates them so) the step kernel itself reads the actions
    // from host memory and writes the 12 kin rows, reward and flags straight into the pinned log / result arrays over PCIe.
    // One kernel launch per step instead of launch + three DMA operations, each with its own start-up latency, and the
    // transfers run under the kernel instead of behind it.  Anything not pinned falls back to staging + copies, per array.
    bool host_done = false;
    if (m.zero_copy && m.d_log) {
        // [reward | terminated | truncated] in one block (the facade's layout): one look-up covers all three
        const bool one_block = reward && (void*)terminated == (char*)reward + z.E * z.rs && truncated == terminated + z.E;
        void* a_rew = host_alias(reward);
        void* a_term = one_block ? (a_rew ? (char*)a_rew + z.E * z.rs : nullptr) : host_alias(terminated);
        void* a_trunc = one_block ? (a_rew ? (char*)a_term + z.E : nullptr) : host_alias(truncated);
        void* a_tkin = terminal_kin ? host_alias(terminal_kin) : nullptr;
        const bool outs_ok = (!reward || a_rew) && (!terminated || a_term) && (!truncated || a_trunc) && (!terminal_kin || a_tkin);
        if (outs_ok) {
            const void* a_act = host_alias(actions);
            if (!a_act) {       // pageable actions: stage them, everything else stays zero-copy
                CU(cudaMemcpyAsync(s->h_act, actions, z.act_b, cudaMemcpyHostToDevice, st));
                a_act = s->h_act;
            }
            // Measured alternatives (profiles/r02/e2e_breakdown.jsonl): staging the actions with a DMA copy and keeping only the
            // outputs zero-copy 121 us of device time, kin rows by one DMA copy behind the kernel 110 us, everything by the
            // kernel 105 us (the link delivers ~42 GB/s device-to-host on this pool: 3.5 MB = 84 us is the floor)
            float* kin_rows = m.d_log + (m.row + s->A) * m.ld + m.col0;
            int rc = step_impl(s, a_act, d_obs_prev, d_obs_out, a_rew, (uint8_t*)a_term, (uint8_t*)a_trunc, a_tkin, kin_rows, stream,
                               m.ld, true);
            if (rc) return rc;
            host_done = true;
        }
    }
    if (!host_done) {
        CU(cudaMemcpyAsync(s->h_act, actions, z.act_b, cudaMemcpyHostToDevice, st));
        int rc = step_impl(s, s->h_act, d_obs_prev, d_obs_out, d_rew, d_term, d_trunc, terminal_kin ? s->h_tkin : nullptr, m.d_kin_t, stream);
        if (rc) return rc;
        // what the device computed: 12 kin rows into the slid window
        CU(mirror_rows_d2h(s, m.row + s->A, m.d_kin_t, 12, st));
    }
    if (internal) { s->h_cur = nxt; s->h_has_prev = true; }
    // reward and flags of every env (one packed copy when the caller's arrays are laid out like the staging)
    const bool packed = tight && reward && (void*)terminated == (char*)reward + z.E * z.rs && truncated == terminated + z.E;
    if (host_done) {
        // written by the kernel
    } else if (packed) {
        CU(cudaMemcpyAsync(reward, d_rew, z.E * z.rs + 2 * z.E, cudaMemcpyDeviceToHost, st));
    } else {
        if (reward) CU(cudaMemcpyAsync(reward, d_rew, z.E * z.rs, cudaMemcpyDeviceToHost, st));
        if (terminated) CU(cudaMemcpyAsync(terminated, d_term, z.E, cudaMemcpyDeviceToHost, st));
        if (truncated) CU(cudaMemcpyAsync(truncated, d_trunc, z.E, cudaMemcpyDeviceToHost, st));
    }
    if (terminal_kin && !host_done) CU(cudaMemcpyAsync(terminal_kin, s->h_tkin, (size_t)s->D * 12 * sizeof(float), cudaMemcpyDeviceToHost, st));
    m.pending = true;
    m.pending_obs = d_obs_out;
    m.pending_actions = (const float*)actions;
    return GPD_OK;
}

int gpd_step_mirror_end(gpd_sim* s, int64_t* first_row, void* stream)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    Mirror& m = s->mir;
    if (!m.pending) return fail(GPD_ERR_INVALID, "gpd_step_mirror_end without gpd_step_mirror_begin");
    m.pending = false;
    m.valid = false;
    // what the host already has: its own action, transposed into the newest ring rows while the device works
    mirror_write_action(s, m.pending_actions, m.row + s->W);
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    m.row += s->A;
    m.valid = true; m.synced_seq = s->obs_seq; m.synced_obs = m.pending_obs;
    if (first_row) *first_row = m.row;
    return GPD_OK;
}

int gpd_step_mirror(gpd_sim* s, const void* actions, const void* d_obs_prev, void* d_obs_out, void* reward,
                    uint8_t* terminated, uint8_t* truncated, void* terminal_kin, int64_t* first_row, void* stream)
{
    int rc = gpd_step_mirror_begin(s, actions, d_obs_prev, d_obs_out, reward, terminated, truncated, terminal_kin, stream);
    if (rc) return rc;
    return gpd_step_mirror_end(s, first_row, stream);
}

int gpd_reset_mirror(gpd_sim* s, const uint8_t* env_mask, const void* d_obs_prev, void* d_obs_out, int64_t* first_row, void* stream)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    Mirror& m = s->mir;
    if (!m.log) return fail(GPD_ERR_INVALID, "gpd_reset_mirror: no host mirror attached (gpd_mirror_attach)");
    if (m.pending) return fail(GPD_ERR_INVALID, "gpd_reset_mirror: a step is in flight (gpd_step_mirror_end)");
    CU(use_device(s->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    const HostSizes z = host_sizes(s);
    const bool internal = d_obs_out == nullptr;
    int nxt = s->h_cur ^ 1;
    if (internal) {
        d_obs_prev = s->h_has_prev ? s->h_obs[s->h_cur] : nullptr;
        d_obs_out = s->h_obs[nxt];
    }
    const bool in_sync = m.valid && m.synced_seq == s->obs_seq && m.synced_obs == d_obs_prev;
    if (env_mask) CU(cudaMemcpyAsync(s->h_mask, env_mask, z.E, cudaMemcpyHostToDevice, st));
    int rc = gpd_reset(s, env_mask ? s->h_mask : nullptr, d_obs_prev, d_obs_out, stream);
    if (rc) return rc;
    if (internal) { s->h_cur = nxt; s->h_has_prev = true; }
    m.valid = false;
    if (in_sync) {      // the ring survives a reset (BaseRLAviary.py:153-154): only the 12 kin rows change, the window does not move
        CU(launch_transpose_cols((const float*)d_obs_out, s->D, s->W, 0, 12, m.d_kin_t, s->D, st));
        CU(mirror_rows_d2h(s, m.row, m.d_kin_t, 12, st));
    } else {
        if (m.row + s->W > m.rows) m.row = 0;
        rc = mirror_refresh(s, d_obs_out, m.row, st);
        if (rc) return rc;
    }
    CU(cudaStreamSynchronize(st));
    m.valid = true; m.synced_seq = s->obs_seq; m.synced_obs = d_obs_out;
    if (first_row) *first_row = m.row;
    return GPD_OK;
}

int gpd_get_state(gpd_sim* s, void* state20, void* rpy_rates, void* pid_state, int32_t* step_counter, void* stream)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    CU(use_device(s->cfg.device));
    unchain(s, stream);
    int rc = sync_state(s, stream);
    if (rc) return rc;
    if (s->cfg.precision == GPD_F64)
        CU(launch_get_state<double>(s->a64, (const float*)s->last_obs, (double*)state20, (double*)rpy_rates, (double*)pid_state, step_counter, (cudaStream_t)stream));
    else
        CU(launch_get_state<float>(s->a32, (const float*)s->last_obs, (float*)state20, (float*)rpy_rates, (float*)pid_state, step_counter, (cudaStream_t)stream));
    return GPD_OK;
}

int gpd_note_latest_obs(gpd_sim* s, const void* obs)
{
    if (!s || !obs) return fail(GPD_ERR_INVALID, "gpd_note_latest_obs: null argument");
    s->last_obs = obs;
    ++s->obs_seq;                 // the caller replaced the latest observation: a host mirror must be rebuilt from it
    return GPD_OK;
}

int gpd_set_state(gpd_sim* s, const void* state20, const void* rpy_rates, const void* pid_state,
                  const int32_t* step_counter, void* stream)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    CU(use_device(s->cfg.device));
    unchain(s, stream);
    int rc = sync_state(s, stream);
    if (rc) return rc;
    if (s->cfg.precision == GPD_F64)
        CU(launch_set_state<double>(s->a64, (const double*)state20, (const double*)rpy_rates, (const double*)pid_state, step_counter, (cudaStream_t)stream));
    else
        CU(launch_set_state<float>(s->a32, (const float*)state20, (const float*)rpy_rates, (const float*)pid_state, step_counter, (cudaStream_t)stream));
    return GPD_OK;
}

int gpd_pid_compute(int device, int precision, const gpd_pid_params* pid, int64_t n, double control_timestep,
                    const void* cur_pos, const void* cur_quat, const void* cur_vel, const void* target_pos,
                    const void* target_rpy, const void* target_vel, const void* target_rpy_rates,
                    void* pid_state, void* rpm_out, void* pos_e_out, void* yaw_e_out, void* stream)
{
    if (!pid || !cur_pos || !cur_quat || !cur_vel || !target_pos || !pid_state || !rpm_out || n < 0)
        return fail(GPD_ERR_INVALID, "gpd_pid_compute: null argument");
    if (n == 0) return GPD_OK;
    CU(use_device(device));
    if (precision == GPD_F64) {
        DevPid<double> c; fill_pid(*pid, c);
        CU(launch_pid<double>(c, n, control_timestep, (const double*)cur_pos, (const double*)cur_quat, (const double*)cur_vel,
                              (const double*)target_pos, (const double*)target_rpy, (const double*)target_vel,
                              (const double*)target_rpy_rates, (double*)pid_state, (double*)rpm_out, (double*)pos_e_out,
                              (double*)yaw_e_out, (cudaStream_t)stream));
    } else if (precision == GPD_F32) {
        DevPid<float> c; fill_pid(*pid, c);
        CU(launch_pid<float>(c, n, (float)control_timestep, (const float*)cur_pos, (const float*)cur_quat, (const float*)cur_vel,
                             (const float*)target_pos, (const float*)target_rpy, (const float*)target_vel,
                             (const float*)target_rpy_rates, (float*)pid_state, (float*)rpm_out, (float*)pos_e_out,
                             (float*)yaw_e_out, (cudaStream_t)stream));
    } else return fail(GPD_ERR_INVALID, "bad precision");
    return GPD_OK;
}

int gpd_force_ground_effect(int device, int precision, const gpd_drone_params* d, int64_t n, const void* rpm,
                            const void* pos, const void* quat, void* out, uint8_t* applied, void* stream)
{
    if (!d || !rpm || !pos || !quat || !out || n < 0) return fail(GPD_ERR_INVALID, "gpd_force_ground_effect: null argument");
    if (n == 0) return GPD_OK;
    CU(use_device(device));
    if (precision == GPD_F64) { DevDrone<double> P; fill_drone(*d, P);
        CU(launch_ground_effect<double>(P, n, (const double*)rpm, (const double*)pos, (const double*)quat, (double*)out, applied, (cudaStream_t)stream)); }
    else { DevDrone<float> P; fill_drone(*d, P);
        CU(launch_ground_effect<float>(P, n, (const float*)rpm, (const float*)pos, (const float*)quat, (float*)out, applied, (cudaStream_t)stream)); }
    return GPD_OK;
}

int gpd_force_drag(int device, int precision, const gpd_drone_params* d, int64_t n, const void* rpm,
                   const void* quat, const void* vel, void* out, void* stream)
{
    if (!d || !rpm || !quat || !vel || !out || n < 0) return fail(GPD_ERR_INVALID, "gpd_force_drag: null argument");
    if (n == 0) return GPD_OK;
    CU(use_device(device));
    if (precision == GPD_F64) { DevDrone<double> P; fill_drone(*d, P);
        CU(launch_drag<double>(P, n, (const double*)rpm, (const double*)quat, (const double*)vel, (double*)out, (cudaStream_t)stream)); }
    else { DevDrone<float> P; fill_drone(*d, P);
        CU(launch_drag<float>(P, n, (const float*)rpm, (const float*)quat, (const float*)vel, (float*)out, (cudaStream_t)stream)); }
    return GPD_OK;
}

int gpd_force_downwash(int device, int precision, const gpd_drone_params* d, int64_t num_envs, int32_t num_drones,
                       const void* pos, void* out, void* stream)
{
    if (!d || !pos || !out || num_envs < 0 || num_drones < 1) return fail(GPD_ERR_INVALID, "gpd_force_downwash: bad argument");
    if (num_envs == 0) return GPD_OK;
    CU(use_device(device));
    if (precision == GPD_F64) { DevDrone<double> P; fill_drone(*d, P);
        CU(launch_downwash<double>(P, num_envs, num_drones, (const double*)pos, (double*)out, (cudaStream_t)stream)); }
    else { DevDrone<float> P; fill_drone(*d, P);
        CU(launch_downwash<float>(P, num_envs, num_drones, (const float*)pos, (float*)out, (cudaStream_t)stream)); }
    return GPD_OK;
}

int gpd_set_timeline_buffer(gpd_sim* s, unsigned long long* dev_buf)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    s->a32.timeline = dev_buf;
    s->a64.timeline = dev_buf;
    return GPD_OK;
}

int gpd_grid_size(const gpd_sim* s) { return s ? (int)s->lc.grid : fail(GPD_ERR_INVALID, "null handle"); }

int gpd_rollout_pid(gpd_sim* s, int32_t n_ctrl_steps, const void* waypoints, int32_t n_wp,
                    int32_t* wp_counters, void* action, void* stream)
{
    if (!s || !waypoints || !wp_counters || !action || n_wp < 1 || n_ctrl_steps < 0)
        return fail(GPD_ERR_INVALID, "gpd_rollout_pid: bad argument");
    if (s->cfg.env_kind != GPD_ENV_CTRL) return fail(GPD_ERR_INVALID, "gpd_rollout_pid needs the Ctrl env");
    if (s->cfg.drone.model == GPD_RACE) return fail(GPD_ERR_INVALID, "DSLPIDControl requires CF2X or CF2P");
    if (s->cfg.physics_flags & GPD_PHY_DW) return fail(GPD_ERR_INVALID, "gpd_rollout_pid does not support downwash");
    CU(use_device(s->cfg.device));
    unchain(s, stream);
    if (s->cfg.precision == GPD_F64)
        CU(launch_rollout_pid<double>(s->a64, n_ctrl_steps, (const double*)waypoints, n_wp, wp_counters, (double*)action, (cudaStream_t)stream));
    else
        CU(launch_rollout_pid<float>(s->a32, n_ctrl_steps, (const float*)waypoints, n_wp, wp_counters, (float*)action, (cudaStream_t)stream));
    return GPD_OK;
}

int gpd_rollout(gpd_sim* s, int32_t n_steps, const void* actions, const void* obs_prev, void* obs_out,
                void* reward, uint8_t* terminated, uint8_t* truncated, void* traj, void* terminal_kin, void* stream)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    if (n_steps < 1) return fail(GPD_ERR_INVALID, "gpd_rollout: n_steps must be >= 1");
    if (!actions || !obs_out) return fail(GPD_ERR_INVALID, "gpd_rollout: actions and obs_out are required");
    const bool ctrl = s->cfg.env_kind == GPD_ENV_CTRL;
    if (ctrl) obs_prev = nullptr;
    if (obs_out == obs_prev || obs_out == actions || (traj && (traj == obs_out || traj == actions)) ||
        (terminal_kin && (terminal_kin == obs_out || terminal_kin == traj)))
        return fail(GPD_ERR_INVALID, "gpd_rollout: aliased buffers");
    if (((uintptr_t)actions | (uintptr_t)obs_prev | (uintptr_t)obs_out | (uintptr_t)traj | (uintptr_t)terminal_kin) & 15)
        return fail(GPD_ERR_INVALID, "gpd_rollout: actions, observations, traj and terminal_kin must be 16-byte aligned");
    CU(use_device(s->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    unchain(s, stream);                 // the next step is not launched programmatically behind the rollout
    int rc = sync_state(s, stream);     // chained-state tiles back into the arrays: the rollout reads and writes those
    if (rc) return rc;
    // the step kernel's tiles without its DMA warp: one statistics slot per CTA, as gpd_create allocated them
    LaunchCfg lc{};
    lc.threads = s->lc.threads - s->copy_threads;
    lc.grid = s->lc.grid;
    lc.smem = smem_bytes(s->cfg.precision == GPD_F64, false, s->cfg.num_drones > 1, s->dpb, s->dpb / s->cfg.num_drones);
    if (s->cfg.precision == GPD_F64) {
        StepArgs<double> a = s->a64;
        a.actions = actions; a.obs_prev = (const float*)obs_prev; a.obs_out = obs_out; a.reward = (double*)reward;
        a.terminated = terminated; a.truncated = truncated; a.terminal_kin = (float*)terminal_kin;
        CU(launch_rollout<double>(a, n_steps, traj, lc, st));
    } else {
        StepArgs<float> a = s->a32;
        a.actions = actions; a.obs_prev = (const float*)obs_prev; a.obs_out = obs_out; a.reward = (float*)reward;
        a.terminated = terminated; a.truncated = truncated; a.terminal_kin = (float*)terminal_kin;
        CU(launch_rollout<float>(a, n_steps, traj, lc, st));
    }
    s->last_obs = obs_out;
    ++s->obs_seq;
    return GPD_OK;
}

int gpd_plan(gpd_sim* s, int32_t n_steps, int32_t n_samples, const void* actions, const void* targets, double gamma,
             void* returns, int32_t* done_step, void* reward, void* final_kin, void* stream)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    if (s->cfg.env_kind == GPD_ENV_CTRL) return fail(GPD_ERR_INVALID, "gpd_plan: the Ctrl env has no reward to plan on");
    if (n_steps < 1 || n_samples < 1) return fail(GPD_ERR_INVALID, "gpd_plan: n_steps and n_samples must be >= 1");
    if (!std::isfinite(gamma) || gamma < 0.0 || gamma > 1.0) return fail(GPD_ERR_INVALID, "gpd_plan: gamma must be in [0, 1]");
    if (!actions || !returns) return fail(GPD_ERR_INVALID, "gpd_plan: actions and returns are required");
    if (((uintptr_t)actions | (uintptr_t)final_kin) & 15)
        return fail(GPD_ERR_INVALID, "gpd_plan: actions and final_kin must be 16-byte aligned");
    const void* outs[4] = { returns, done_step, reward, final_kin };
    for (int j = 0; j < 4; ++j) {
        if (!outs[j]) continue;
        if (outs[j] == actions || outs[j] == targets) return fail(GPD_ERR_INVALID, "gpd_plan: aliased buffers");
        for (int k = j + 1; k < 4; ++k)
            if (outs[j] == outs[k]) return fail(GPD_ERR_INVALID, "gpd_plan: aliased buffers");
    }
    // whole copies per CTA (MULTI) or DPB copies per CTA, as the rollout's tiles
    const int N = s->cfg.num_drones;
    const int64_t copies = s->cfg.num_envs * (int64_t)n_samples;
    const int64_t per_cta = N > 1 ? s->dpb / N : s->dpb;
    LaunchCfg lc{};
    lc.threads = s->lc.threads - s->copy_threads;
    lc.grid = (copies + per_cta - 1) / per_cta;
    lc.smem = smem_bytes(s->cfg.precision == GPD_F64, false, N > 1, s->dpb, s->dpb / N);
    if (lc.grid > INT32_MAX) return fail(GPD_ERR_INVALID, "gpd_plan: %lld copies need more than INT32_MAX CTAs", (long long)copies);
    CU(use_device(s->cfg.device));
    cudaStream_t st = (cudaStream_t)stream;
    unchain(s, stream);                 // the next step is not launched programmatically behind the plan
    int rc = sync_state(s, stream);     // chained-state tiles back into the arrays: the plan reads the state from there
    if (rc) return rc;
    if (s->cfg.precision == GPD_F64)
        CU(plan_launch<double>(s, s->a64, n_steps, n_samples, actions, targets, gamma, returns, done_step, reward, final_kin, lc, st));
    else
        CU(plan_launch<float>(s, s->a32, n_steps, n_samples, actions, targets, gamma, returns, done_step, reward, final_kin, lc, st));
    return GPD_OK;
}

int64_t gpd_plan_grad_tape_bytes(const gpd_sim* s, int32_t n_steps, int32_t n_samples)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    if (n_steps < 1 || n_samples < 1) return fail(GPD_ERR_INVALID, "gpd_plan_grad_tape_bytes: n_steps and n_samples must be >= 1");
    const int64_t b = plan_grad_tape_bytes(s, n_steps, n_samples);
    if (b < 0) return fail(GPD_ERR_INVALID, "gpd_plan_grad_tape_bytes: the tape does not fit in 63 bits");
    return b;
}

int gpd_plan_grad(gpd_sim* s, int32_t n_steps, int32_t n_samples, const void* actions, const void* targets, double gamma,
                  void* returns, int32_t* done_step, void* grad_actions, void* tape, int64_t tape_bytes, void* stream)
{
    if (!s) return fail(GPD_ERR_INVALID, "null handle");
    const gpd_config& c = s->cfg;
    if (c.env_kind == GPD_ENV_CTRL) return fail(GPD_ERR_INVALID, "gpd_plan_grad: the Ctrl env has no reward to plan on");
    if (c.action_type != GPD_ACT_RPM && c.action_type != GPD_ACT_ONE_D_RPM)
        return fail(GPD_ERR_INVALID, "gpd_plan_grad: only the RPM and ONE_D_RPM actions are differentiated (no DSLPID adjoint)");
    if (c.physics_flags != 0)
        return fail(GPD_ERR_INVALID, "gpd_plan_grad: only Physics.DYN (physics_flags 0) is differentiated, no force models");
    if (n_steps < 1 || n_samples < 1) return fail(GPD_ERR_INVALID, "gpd_plan_grad: n_steps and n_samples must be >= 1");
    if (!std::isfinite(gamma) || gamma < 0.0 || gamma > 1.0) return fail(GPD_ERR_INVALID, "gpd_plan_grad: gamma must be in [0, 1]");
    if (!actions || !returns || !grad_actions || !tape)
        return fail(GPD_ERR_INVALID, "gpd_plan_grad: actions, returns, grad_actions and tape are required");
    if (((uintptr_t)actions | (uintptr_t)tape) & 15)
        return fail(GPD_ERR_INVALID, "gpd_plan_grad: actions and tape must be 16-byte aligned");
    const int64_t need = plan_grad_tape_bytes(s, n_steps, n_samples);
    if (need < 0 || tape_bytes < need)
        return fail(GPD_ERR_INVALID, "gpd_plan_grad: tape_bytes %lld < %lld", (long long)tape_bytes, (long long)need);
    const void* bufs[6] = { actions, targets, returns, done_step, grad_actions, tape };
    for (int j = 0; j < 6; ++j)
        for (int k = j + 1; k < 6; ++k)
            if (bufs[j] && bufs[j] == bufs[k]) return fail(GPD_ERR_INVALID, "gpd_plan_grad: aliased buffers");
    const int N = c.num_drones;
    const int64_t copies = c.num_envs * (int64_t)n_samples;
    const int64_t per_cta = N > 1 ? s->dpb / N : s->dpb;
    LaunchCfg lc{};
    lc.threads = s->lc.threads - s->copy_threads;
    lc.grid = (copies + per_cta - 1) / per_cta;
    lc.smem = smem_bytes(c.precision == GPD_F64, false, N > 1, s->dpb, s->dpb / N);
    if (lc.grid > INT32_MAX) return fail(GPD_ERR_INVALID, "gpd_plan_grad: %lld copies need more than INT32_MAX CTAs", (long long)copies);
    CU(use_device(c.device));
    cudaStream_t st = (cudaStream_t)stream;
    unchain(s, stream);                 // the next step is not launched programmatically behind the plan
    int rc = sync_state(s, stream);     // chained-state tiles back into the arrays: the plan reads the state from there
    if (rc) return rc;
    if (c.precision == GPD_F64)
        CU(plan_grad_launch<double>(s, s->a64, n_steps, n_samples, actions, targets, gamma, returns, done_step, grad_actions, tape, lc, st));
    else
        CU(plan_grad_launch<float>(s, s->a32, n_steps, n_samples, actions, targets, gamma, returns, done_step, grad_actions, tape, lc, st));
    return GPD_OK;
}

int gpd_count_nonfinite(gpd_sim* s, long long* out_host, void* stream)
{
    if (!s || !out_host) return fail(GPD_ERR_INVALID, "gpd_count_nonfinite: null argument");
    CU(use_device(s->cfg.device));
    unchain(s, stream);
    int rc = sync_state(s, stream);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* cnt = (unsigned long long*)s->stats_out;       // reuse the 64-byte scratch
    CU(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), st));
    if (s->cfg.precision == GPD_F64) CU(launch_nonfinite<double>(s->a64, cnt, st));
    else CU(launch_nonfinite<float>(s->a32, cnt, st));
    unsigned long long h = 0;
    CU(cudaMemcpyAsync(&h, cnt, sizeof h, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *out_host = (long long)h;
    return GPD_OK;
}

// ---- NCCL, bound at run time: the library never links against libnccl; a process that passes a communicator has it loaded ----
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*CommCount)(const ncclComm_t, int*) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};

static const NcclApi* nccl_api()
{
    static NcclApi api;
    static bool tried = false;
    if (tried) return api.ok ? &api : nullptr;
    tried = true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);     // the copy the process already uses (e.g. torch's)
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return nullptr;
    api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))dlsym(h, "ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))dlsym(h, "ncclCommDestroy");
    api.CommCount = (decltype(api.CommCount))dlsym(h, "ncclCommCount");
    api.AllGather = (decltype(api.AllGather))dlsym(h, "ncclAllGather");
    api.GetErrorString = (decltype(api.GetErrorString))dlsym(h, "ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.CommCount && api.AllGather && api.GetErrorString;
    return api.ok ? &api : nullptr;
}

#define NC(api, call)                                                                                    \
    do {                                                                                                 \
        ncclResult_t _r = (call);                                                                        \
        if (_r != ncclSuccess) return fail(GPD_ERR_CUDA, "%s failed: %s", #call, (api)->GetErrorString(_r)); \
    } while (0)

int gpd_nccl_unique_id(char id_out[GPD_NCCL_UNIQUE_ID_BYTES])
{
    if (!id_out) return fail(GPD_ERR_INVALID, "gpd_nccl_unique_id: null argument");
    const NcclApi* n = nccl_api();
    if (!n) return fail(GPD_ERR_INVALID, "libnccl.so.2 could not be loaded: %s", dlerror());
    static_assert(sizeof(ncclUniqueId) == GPD_NCCL_UNIQUE_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    NC(n, n->GetUniqueId(&id));
    memcpy(id_out, &id, sizeof id);
    return GPD_OK;
}

int gpd_nccl_comm_init(const char id[GPD_NCCL_UNIQUE_ID_BYTES], int rank, int world_size, int device, void** comm_out)
{
    if (!id || !comm_out || world_size < 1 || rank < 0 || rank >= world_size) return fail(GPD_ERR_INVALID, "gpd_nccl_comm_init: bad argument");
    *comm_out = nullptr;
    const NcclApi* n = nccl_api();
    if (!n) return fail(GPD_ERR_INVALID, "libnccl.so.2 could not be loaded: %s", dlerror());
    CU(use_device(device));
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof uid);
    ncclComm_t c = nullptr;
    NC(n, n->CommInitRank(&c, world_size, uid, rank));
    *comm_out = c;
    return GPD_OK;
}

int gpd_nccl_comm_destroy(void* comm)
{
    if (!comm) return GPD_OK;
    const NcclApi* n = nccl_api();
    if (!n) return fail(GPD_ERR_INVALID, "libnccl.so.2 could not be loaded");
    NC(n, n->CommDestroy((ncclComm_t)comm));
    return GPD_OK;
}

int gpd_episode_stats(gpd_sim* s, double out[8], int clear, void* nccl_comm, void* stream)
{
    if (!s || !out) return fail(GPD_ERR_INVALID, "gpd_episode_stats: null argument");
    for (int k = 0; k < 8; ++k) out[k] = 0.0;
    if (!s->cfg.auto_reset) return fail(GPD_ERR_INVALID, "episode statistics are kept only with auto_reset");
    CU(use_device(s->cfg.device));
    unchain(s, stream);
    cudaStream_t st = (cudaStream_t)stream;
    StatSlot* slots = s->cfg.precision == GPD_F64 ? s->a64.p.stat_slots : s->a32.p.stat_slots;
    CU(launch_stats(slots, s->lc.grid, s->stats_out, clear, slots, st));
    const double* result = s->stats_out;
    if (nccl_comm) {    // job-wide: ONE collective (all-gather of the 8 doubles of every rank) + a rank-order combine on the device
        const NcclApi* n = nccl_api();
        if (!n) return fail(GPD_ERR_INVALID, "a communicator was passed but libnccl.so.2 could not be loaded");
        int nranks = 0;
        NC(n, n->CommCount((ncclComm_t)nccl_comm, &nranks));
        if (nranks > s->stats_gather_ranks) {
            CU(cudaStreamSynchronize(st));
            cudaFree(s->stats_gather);
            s->stats_gather = nullptr; s->stats_gather_ranks = 0;
            CU(cudaMalloc((void**)&s->stats_gather, (size_t)(nranks + 1) * 8 * sizeof(double)));
            s->stats_gather_ranks = nranks;
        }
        NC(n, n->AllGather(s->stats_out, s->stats_gather, 8, ncclFloat64, (ncclComm_t)nccl_comm, st));
        double* combined = s->stats_gather + (size_t)nranks * 8;
        CU(launch_stats_combine(s->stats_gather, nranks, combined, st));
        result = combined;
    }
    CU(cudaMemcpyAsync(out, result, 8 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (out[0] == 0.0) { out[4] = 0.0; out[5] = 0.0; }
    return GPD_OK;
}

int gpd_adjacency(gpd_sim* s, double neighbourhood_radius, void* out, void* stream)
{
    if (!s || !out) return fail(GPD_ERR_INVALID, "gpd_adjacency: null argument");
    CU(use_device(s->cfg.device));
    unchain(s, stream);
    int rc = sync_state(s, stream);
    if (rc) return rc;
    if (s->cfg.precision == GPD_F64) CU(launch_adjacency<double>(s->a64, neighbourhood_radius, (double*)out, (cudaStream_t)stream));
    else CU(launch_adjacency<float>(s->a32, (float)neighbourhood_radius, (float*)out, (cudaStream_t)stream));
    return GPD_OK;
}

}  // extern "C"
