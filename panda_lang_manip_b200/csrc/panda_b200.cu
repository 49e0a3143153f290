// panda_b200.cu -- C ABI of libpanda_b200.so (include/panda_b200.h): handle management, SoA state allocation, snapshots,
// kernel dispatch, the host-buffer entry points and the HER reward kernels.  No CPU fallback: every entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <memory>
#include <string>
#include <type_traits>
#include <utility>
#include <variant>
#include <vector>
#include "panda_b200.h"
#include "panda_kernels.cuh"
#include "panda_model.h"
#include "panda_scene.h"
#include "panda_render.h"
#include "panda_motion.cuh"

namespace pg {
long long g_launches = 0;
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
static int cuda_fail(cudaError_t e, const char* what) { return fail(PG_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e)); }
#define PG_CUDA(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_, #x); } while (0)

template <typename T, int TASK> cudaError_t configure_step(void);       // panda_step_task.cu
template <typename T> cudaError_t configure_bare(void);                 // panda_bare.cu
template <typename T> void launch_render_setup(const EnvDev<T>& E, const RenderScene& R, RenderPrim* prims, cudaStream_t st);   // panda_render.cu
void launch_render(const RenderPrim* prims, const RenderCamera& C, int n_envs, float* depth, unsigned char* rgba, unsigned char* seg, float* points, unsigned char* valid, cudaStream_t st);
template <typename T> void launch_motion_move(const EnvDev<T>& E, const MotionPlan& P, const double* goal, const double* goal_quat, const unsigned char* mask, cudaStream_t st);   // panda_motion.cu
void launch_motion_gripper(const MotionPlan& P, double finger, int steps, const unsigned char* mask, cudaStream_t st);
template <typename T> void launch_motion_step(const EnvDev<T>& E, const MotionPlan& P, int act_dim, int* remaining, cudaStream_t st);
#define PG_DECL(T, K)                                                                                        \
    extern template void launch_step<T, K>(const EnvDev<T>&, int, const StepIO&, cudaStream_t);              \
    extern template void launch_reset<T, K>(const EnvDev<T>&, const ResetIO&, cudaStream_t);                 \
    extern template cudaError_t configure_step<T, K>(void);
PG_DECL(float, 0) PG_DECL(float, 1) PG_DECL(float, 2) PG_DECL(float, 3) PG_DECL(float, 4) PG_DECL(float, 5)
PG_DECL(double, 0) PG_DECL(double, 1) PG_DECL(double, 2) PG_DECL(double, 3) PG_DECL(double, 4) PG_DECL(double, 5)

// The kernels are templates over the task: calls f(std::integral_constant<int, K>()) for the K of Ks equal to the runtime id
// (nothing if none is).  Only the listed Ks are instantiated.
template <int... Ks, typename F> static void dispatch(int id, F&& f) {
    (void)((id == Ks && (f(std::integral_constant<int, Ks>()), true)) || ...);
}
// goal layouts: 3-D position (tasks 0-3, thr 0.05), Stack 6-D (thr 0.1), Flip quaternion (thr 0.2); the goal kernels exist per layout
static int goal_layout(int task) { return task == TASK_STACK || task == TASK_FLIP ? task : 0; }
// f(float()) for PG_F32 goal arrays, f(double()) otherwise
template <typename F> static auto with_dtype(int dtype, F&& f) { return dtype == PG_F32 ? f(float()) : f(double()); }
static bool valid_task(int task) { return task >= 0 && task <= 5; }
static bool valid_reward_type(int reward_type) { return reward_type >= 0 && reward_type <= 1; }

// One CUDA resource: freed when its owner goes out of scope (a NULL one is not).  Move-only; the raw value is `p`.
template <typename P, cudaError_t (*Free)(P)> struct Own {
    P p{};
    Own() = default;
    Own(Own&& o) noexcept : p(o.p) { o.p = P{}; }
    Own& operator=(Own&& o) noexcept { std::swap(p, o.p); return *this; }
    ~Own() { if (p) Free(p); }
};
using DevBuf = Own<void*, cudaFree>;
using PinnedBuf = Own<void*, cudaFreeHost>;
using Stream = Own<cudaStream_t, cudaStreamDestroy>;
using Event = Own<cudaEvent_t, cudaEventDestroy>;

// page-locked (cudaHostAlloc / cudaHostRegister / pg_host_pin) host memory can be the source / target of an async copy directly
static bool host_pinned(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}
// The host ends of an async copy to or from a caller's host buffer: a page-locked buffer is copied directly, any other one goes
// through pinned staging memory -- copied there before the upload (host_source), or out of it after the stream is synchronised
// (host_target, then copy_back).  A NULL output is not copied.
static const void* host_source(const void* user, void* stage, size_t bytes) { return host_pinned(user) ? user : memcpy(stage, user, bytes); }
static void* host_target(void* user, void* stage) { return user && !host_pinned(user) ? stage : user; }
static void copy_back(void* user, const void* target, size_t bytes) { if (target != user) memcpy(user, target, bytes); }

// Staging of the host-buffer entry points: a private stream, one device input and one device output buffer, and a pinned mirror of
// each.  It only grows: a direction that is too small is re-allocated 25 % larger than asked for, and its capacity is recorded only
// once both of its buffers exist, so the next reserve after a failed one allocates again instead of using a half-built stage.
struct Staging {
    unsigned flags = cudaStreamNonBlocking;     // of the stream
    Stream st; DevBuf d_in, d_out; PinnedBuf h_in, h_out; size_t cap_in = 0, cap_out = 0;
    long long allocs = 0;                       // (re)allocations so far, one per direction
    int reserve(size_t in_bytes, size_t out_bytes) {
        if (!st.p) PG_CUDA(cudaStreamCreateWithFlags(&st.p, flags));
        const int rc = in_bytes > cap_in ? grow(d_in, h_in, cap_in, in_bytes) : PG_OK;
        return rc == PG_OK && out_bytes > cap_out ? grow(d_out, h_out, cap_out, out_bytes) : rc;
    }
    int grow(DevBuf& d, PinnedBuf& h, size_t& cap, size_t bytes) {
        PG_CUDA(cudaStreamSynchronize(st.p));
        cap = 0; d = DevBuf(); h = PinnedBuf();
        const size_t c = bytes + bytes / 4;
        PG_CUDA(cudaMalloc(&d.p, c)); PG_CUDA(cudaMallocHost(&h.p, c));
        cap = c; allocs++;
        return PG_OK;
    }
};
}  // namespace pg

using namespace pg;

struct pg_env {
    int task, ctrl, reward, n, device;
    int obs_dim, goal_dim, act_dim, max_steps, state_dim, nobj;
    DevBuf blob; size_t blob_bytes = 0;               // one allocation: q, qd, obj, goal, steps, episode, ret, stats
    std::variant<EnvDev<float>, EnvDev<double>> env;  // the state in blob: EnvDev<float> for PG_F32 handles, EnvDev<double> for PG_F64
    std::map<int, DevBuf> snaps; int next_snap = 0;
    DevBuf prims; RenderScene rscene;                 // analytic renderer: per-env primitive lists (allocated at the first pg_render)
    std::vector<DevBuf> snap_pool;                    // buffers of removed snapshots, reused by the next save (no allocation in a save / remove loop)
    // env groups: sorted batches are cut into groups of consecutive envs, each advanced on its own stream, so that the tail of
    // one group's launch (a few contact-heavy blocks) overlaps with the other groups' launches instead of idling the GPU
    DevBuf dbg;
    int groups = 1; Stream gstream[8]; Event ev_fork, ev_join[8];
    int segments = 4;                                 // launches per step for sorted batches (see pg_create)
    // pg_step_host's staging, on a blocking stream: like work on a caller's stream, it is ordered after what the legacy default stream holds
    Staging host{cudaStreamDefault};
    ~pg_env() { cudaSetDevice(device); }               // the members are freed after this body runs, on the handle's device
};

// f(E) with the handle's state
template <typename F> static auto with_env(pg_env* e, F&& f) { return std::visit(f, e->env); }
// One thread per env on `stream`: f(E, grid, st) launches a BLOCK-wide kernel over the bound state E.
template <typename F> static int launch_per_env(pg_env* e, void* stream, F&& f) {
    PG_CUDA(cudaSetDevice(e->device));
    const int grid = (e->n + BLOCK - 1) / BLOCK;
    with_env(e, [&](auto& E) { f(E, grid, (cudaStream_t)stream); });
    g_launches++;
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
// stats[first, first + count) to the host (see EnvDev::stats)
static int read_stats(pg_env* e, int first, int count, double* out) {
    PG_CUDA(cudaSetDevice(e->device));
    const double* stats = with_env(e, [](auto& E) { return E.stats; });
    PG_CUDA(cudaMemcpy(out, stats + first, count * sizeof(double), cudaMemcpyDeviceToHost));
    return PG_OK;
}

template <typename T> static void bind(EnvDev<T>& E, pg_env* e, char* base, unsigned long long seed, long long id0) {
    const size_t n = (size_t)e->n;
    E.n = e->n; E.reward_type = e->reward; E.id0 = id0; E.seed = seed;
    size_t off = 0;
    auto take = [&](size_t bytes) { char* p = base + off; off += (bytes + 255) & ~(size_t)255; return p; };
    E.stats = (double*)take(8 * sizeof(double));
    E.q = (T*)take(9 * n * sizeof(T)); E.qd = (T*)take(9 * n * sizeof(T));
    E.obj = (T*)take((size_t)(e->nobj > 0 ? e->nobj : 1) * 13 * n * sizeof(T));
    E.goal = (double*)take(6 * n * sizeof(double));
    E.target = (T*)take(9 * n * sizeof(T));
    E.motor = (T*)take((e->task == PG_TASK_BARE ? 36 : 0) * n * sizeof(T));
    E.steps = (int*)take(n * sizeof(int)); E.episode = (unsigned*)take(n * sizeof(unsigned)); E.ret = (float*)take(n * sizeof(float));
    E.ccount = (unsigned short*)take(n * sizeof(unsigned short)); E.perm = (int*)take(n * sizeof(int));
    E.hist = (int*)take(((n + PERM_CHUNK - 1) / PERM_CHUNK + 8) * PERM_BUCKETS * sizeof(int));
    e->blob_bytes = off;
}

template <typename E, bool WANT_REWARD> static void launch_reward(int task, const E* ag, const E* dg, float* reward, unsigned char* success, long long m, int reward_type, double thr, cudaStream_t st) {
    const int vec_ok = (((uintptr_t)ag | (uintptr_t)dg) & 15) == 0;
    long long blocks = (m / 2 + 255) / 256 + 1;
    int grid = (int)(blocks < 148LL * 32 ? blocks : 148LL * 32);   // grid-stride; capped at a multiple of the SM count
    dispatch<0, 4, 5>(goal_layout(task), [&](auto L) {
        reward_kernel<E, L, WANT_REWARD><<<grid, 256, 0, st>>>(ag, dg, reward, success, m, reward_type, vec_ok, thr);
    });
    g_launches++;
}

// widest load (bytes) every row start allows: base pointers and the row pitch must both be multiples of it; a load that reaches past
// the row's G elements (16-byte loads on 6-D fp32 rows) needs the padding to exist, i.e. pitch >= the loaded span
template <typename E> static int her_vector_bytes(int G, const void* a, const void* b, long long pitch) {
    const uintptr_t bits = (uintptr_t)a | (uintptr_t)b | (uintptr_t)(pitch * (long long)sizeof(E));
    for (int vb = 16; vb > (int)sizeof(E); vb >>= 1) {
        const int ev = vb / (int)sizeof(E), span = (G + ev - 1) / ev * ev;
        if ((bits & (uintptr_t)(vb - 1)) == 0 && span <= pitch) return vb;
    }
    return (int)sizeof(E);
}
template <typename E, int TASK> static void launch_her_task(const E* next_ag, const E* dg, const long long* src, const long long* goal_src, E* dg_out, E* ag_out, float* reward,
                                                            long long m, long long pitch, int reward_type, double thr, cudaStream_t st) {
    const long long per_block = 256LL * HER_INFLIGHT;
    const int grid = (int)std::min<long long>((m + per_block - 1) / per_block, 148LL * 32);
    const int vb = her_vector_bytes<E>(task_goal_dim(TASK), next_ag, dg, pitch);
    if (vb == 16) her_relabel_kernel<E, TASK, 16><<<grid, 256, 0, st>>>(next_ag, dg, src, goal_src, dg_out, ag_out, reward, m, pitch, reward_type, thr);
    else if (vb == 8) her_relabel_kernel<E, TASK, 8><<<grid, 256, 0, st>>>(next_ag, dg, src, goal_src, dg_out, ag_out, reward, m, pitch, reward_type, thr);
    else her_relabel_kernel<E, TASK, (int)sizeof(E)><<<grid, 256, 0, st>>>(next_ag, dg, src, goal_src, dg_out, ag_out, reward, m, pitch, reward_type, thr);
    g_launches++;
}
template <typename E> static void launch_her(int task, const E* next_ag, const E* dg, const long long* src, const long long* goal_src, E* dg_out, E* ag_out, float* reward,
                                             long long m, long long pitch, int reward_type, double thr, cudaStream_t st) {
    dispatch<0, 4, 5>(goal_layout(task), [&](auto L) {
        launch_her_task<E, L>(next_ag, dg, src, goal_src, dg_out, ag_out, reward, m, pitch, reward_type, thr, st);
    });
}

// Host-buffer mode of a step (pg_step_host): every env group copies its own action rows in before its first launch and its own
// output rows out after its last one, on its own stream -- group g's device-to-host copies overlap group g+1's kernels.
struct HostIO { const float* act; float* obs; float* ag; float* dg; float* rew; unsigned char* term; unsigned char* trunc; };
// E: a copy of the handle's bound state, adjusted per launch
template <typename T> static int step_impl(pg_env* e, EnvDev<T> E, const float* actions, const float* target_quat, float* obs, float* ag, float* dg, float* reward,
                                           unsigned char* terminated, unsigned char* truncated, int auto_reset, float* contacts, unsigned char* contact_count,
                                           cudaStream_t stream, const HostIO* hio) {
    PG_CUDA(cudaSetDevice(e->device));
    // Contact-aware scheduling (see perm_*_kernel): large batches are re-sorted by their contact state before every launch, and a
    // step is cut into `segments` launches of consecutive sub-steps so that envs which make contact mid-step are regrouped; small
    // batches keep the identity map, one launch per step and the tiled I/O path.  Results do not depend on either choice.
    const bool use_perm = e->n >= 4096;
    const int segs = use_perm ? e->segments : 1;
    const unsigned short* key = E.ccount;
    int* hist = E.hist;
    int* perm = E.perm;
    if (!use_perm) E.perm = nullptr;
    // host mode pipelines the copies against the env groups the configuration already has (measured: on one GPU the single-stream
    // Reach-joints configuration loses 5 % when cut into 4 groups only to overlap 0.2 ms of copies)
    const int groups = use_perm ? e->groups : 1;
    // group g owns the envs (and thread slots) [g * gsize, min(n, (g + 1) * gsize)), gsize a multiple of the sort chunk
    const int gsize = ((e->n + groups - 1) / groups + PERM_CHUNK - 1) / PERM_CHUNK * PERM_CHUNK;
    const size_t A = e->act_dim, O = e->obs_dim, G = e->goal_dim;
    if (groups > 1) PG_CUDA(cudaEventRecord(e->ev_fork.p, stream));
    for (int g = 0; g < groups; g++) {
        const int t0 = g * gsize, cnt = std::min(e->n, t0 + gsize) - t0;
        if (cnt <= 0) break;
        cudaStream_t st = groups > 1 ? e->gstream[g].p : stream;
        if (groups > 1) PG_CUDA(cudaStreamWaitEvent(st, e->ev_fork.p, 0));
        if (hio) PG_CUDA(cudaMemcpyAsync(const_cast<float*>(actions) + t0 * A, hio->act + t0 * A, (size_t)cnt * A * sizeof(float), cudaMemcpyHostToDevice, st));
        E.t0 = t0; E.tcount = cnt;
        const int nchunks = (cnt + PERM_CHUNK - 1) / PERM_CHUNK;
        int* ghist = hist + (size_t)(t0 / PERM_CHUNK + g) * PERM_BUCKETS;
        const int nsub = E.P.nsub;
        for (int sg = 0; sg < segs; sg++) {
            StepIO io{target_quat, actions, obs, ag, dg, reward, terminated, truncated, auto_reset, sg * nsub / segs, (sg + 1) * nsub / segs,
                      contacts, contact_count};
            if (io.s0 == io.s1) continue;       // fewer sub-steps than segments
            if (use_perm) {
                perm_hist_kernel<<<nchunks, PERM_THREADS, 0, st>>>(key + t0, ghist, cnt);
                perm_scatter_kernel<<<nchunks, PERM_THREADS, 0, st>>>(key + t0, ghist, perm + t0, cnt, nchunks, t0);
                g_launches += 2;
            }
            dispatch<0, 1, 2, 3, 4, 5>(e->task, [&](auto K) { launch_step<T, K>(E, e->ctrl, io, st); });
        }
        if (hio) {
            if (hio->obs) PG_CUDA(cudaMemcpyAsync(hio->obs + t0 * O, obs + t0 * O, (size_t)cnt * O * sizeof(float), cudaMemcpyDeviceToHost, st));
            if (hio->ag) PG_CUDA(cudaMemcpyAsync(hio->ag + t0 * G, ag + t0 * G, (size_t)cnt * G * sizeof(float), cudaMemcpyDeviceToHost, st));
            if (hio->dg) PG_CUDA(cudaMemcpyAsync(hio->dg + t0 * G, dg + t0 * G, (size_t)cnt * G * sizeof(float), cudaMemcpyDeviceToHost, st));
            if (hio->rew) PG_CUDA(cudaMemcpyAsync(hio->rew + t0, reward + t0, (size_t)cnt * sizeof(float), cudaMemcpyDeviceToHost, st));
            if (hio->term) PG_CUDA(cudaMemcpyAsync(hio->term + t0, terminated + t0, (size_t)cnt, cudaMemcpyDeviceToHost, st));
            if (hio->trunc) PG_CUDA(cudaMemcpyAsync(hio->trunc + t0, truncated + t0, (size_t)cnt, cudaMemcpyDeviceToHost, st));
        }
        if (groups > 1) { PG_CUDA(cudaEventRecord(e->ev_join[g].p, st)); PG_CUDA(cudaStreamWaitEvent(stream, e->ev_join[g].p, 0)); }
    }
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

extern "C" {

const char* pg_last_error(void) { return g_err.c_str(); }
long long pg_kernel_launches(void) { return g_launches; }

static int check_device(int device, const char* who) {
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) return fail(PG_ERR_CUDA, std::string(who) + ": no CUDA device (" + cudaGetErrorString(ce) + "); this library has no CPU path");
    if (device < 0 || device >= ndev) return fail(PG_ERR_ARG, std::string(who) + ": bad device index");
    PG_CUDA(cudaSetDevice(device));
    return PG_OK;
}
// the bound state for `precision`, its allocation and the model; the caller fills the scene and the task parameters
static int alloc_state(pg_env* e, int precision, unsigned long long seed, long long env_id_offset, const double base[3]) {
    with_dtype(precision, [&](auto x) { e->env.emplace<EnvDev<decltype(x)>>(); });
    return with_env(e, [&](auto& E) -> int {
        using T = std::remove_pointer_t<decltype(E.q)>;
        bind(E, e, nullptr, seed, env_id_offset);
        cudaError_t err = cudaMalloc(&e->blob.p, e->blob_bytes);
        if (err != cudaSuccess) return cuda_fail(err, "cudaMalloc(state)");
        PG_CUDA(cudaMemset(e->blob.p, 0, e->blob_bytes));
        bind(E, e, (char*)e->blob.p, seed, env_id_offset); E.M = make_model<T>(base);
        // the > 48 kB dynamic shared memory opt-in is per function and per device: done for this handle's device, errors reported
        cudaError_t ce = cudaSuccess;
        if (e->task == PG_TASK_BARE) ce = configure_bare<T>();
        else dispatch<0, 1, 2, 3, 4, 5>(e->task, [&](auto K) { ce = configure_step<T, K>(); });
        if (ce != cudaSuccess) return cuda_fail(ce, "cudaFuncSetAttribute(step kernel shared memory)");
        return PG_OK;
    });
}

int pg_create(int task, int control_type, int reward_type, int num_envs, int device, unsigned long long seed, long long env_id_offset,
              int precision, pg_env** out) {
    if (!out) return fail(PG_ERR_ARG, "pg_create: out is NULL");
    if (!valid_task(task) || control_type < 0 || control_type > 1 || !valid_reward_type(reward_type) || num_envs <= 0 || precision < 0 || precision > 1)
        return fail(PG_ERR_ARG, "pg_create: bad task / control_type / reward_type / num_envs / precision");
    int rc = check_device(device, "pg_create"); if (rc != PG_OK) return rc;
    auto e = std::make_unique<pg_env>();
    e->task = task; e->ctrl = control_type; e->reward = reward_type; e->n = num_envs; e->device = device;
    e->nobj = task_nobj(task); e->obs_dim = task_obs_dim(task); e->goal_dim = task_goal_dim(task); e->act_dim = task_act_dim(task, control_type);
    e->max_steps = task_max_steps(task); e->state_dim = 18 + 13 * e->nobj + e->goal_dim + 1;
    const double base[3] = {-0.6, 0.0, 0.0};   // panda_tasks.py:26,43,60,77,94,111
    rc = alloc_state(e.get(), precision, seed, env_id_offset, base); if (rc != PG_OK) return rc;
    const bool light = e->nobj == 0 && control_type == CTRL_JOINTS;
    e->segments = light ? 4 : 20;
    { const char* v = getenv("PG_DEBUG_TIMING"); if (v && v[0] == '1') { PG_CUDA(cudaMalloc(&e->dbg.p, (size_t)e->n * 2 * sizeof(long long))); PG_CUDA(cudaMemset(e->dbg.p, 0, (size_t)e->n * 2 * sizeof(long long))); } }
    with_env(e.get(), [&](auto& E) {
        using T = std::remove_pointer_t<decltype(E.q)>;
        E.S = make_scene<T>(task); E.P = make_task_params(task); E.dbg = (long long*)e->dbg.p;
    });
    // measured defaults (profiles/r1_notes.md): contact scenes and ee control re-sort before every sub-step and run 4 env groups (2 for ee-controlled Reach);
    // joint-controlled Reach (few contacts) keeps 4 launches per step on one stream
    e->groups = (num_envs >= 16384 && !light) ? (e->nobj == 0 ? 2 : 4) : 1;
    if (e->groups > 1) {
        PG_CUDA(cudaEventCreateWithFlags(&e->ev_fork.p, cudaEventDisableTiming));
        for (int g = 0; g < e->groups; g++) { PG_CUDA(cudaStreamCreateWithFlags(&e->gstream[g].p, cudaStreamNonBlocking)); PG_CUDA(cudaEventCreateWithFlags(&e->ev_join[g].p, cudaEventDisableTiming)); }
    }
    rc = pg_reset(e.get(), nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr); if (rc != PG_OK) return rc;
    PG_CUDA(cudaDeviceSynchronize());
    *out = e.release();
    return PG_OK;
}

int pg_create_bare(int num_envs, int device, int precision, const double* robot_base, int n_bodies, const double* bodies, const double* table_rect,
                   const double* ground_z, pg_env** out) {
    if (!out) return fail(PG_ERR_ARG, "pg_create_bare: out is NULL");
    if (num_envs <= 0 || precision < 0 || precision > 1 || n_bodies < 0 || n_bodies > MAXOBJ || (n_bodies > 0 && !bodies))
        return fail(PG_ERR_ARG, "pg_create_bare: bad num_envs / precision / n_bodies (at most 2 free bodies)");
    for (int o = 0; o < n_bodies; o++) {
        const double* b = bodies + 13 * o;
        if ((b[0] != SH_BOX && b[0] != SH_CYL) || !(b[1] > 0) || !(b[2] > 0) || !(b[3] > 0) || !(b[4] > 0) || !(b[5] >= 0))
            return fail(PG_ERR_ARG, "pg_create_bare: body rows are [shape(0 box,1 z-cylinder) hx hy hz mass(>0) mu pos3 quat4]");
    }
    double pose[MAXOBJ][7];                     // the bodies' creation poses, quaternions normalised
    for (int o = 0; o < n_bodies; o++) {
        const double* b = bodies + 13 * o;
        const double nq = sqrt(b[9] * b[9] + b[10] * b[10] + b[11] * b[11] + b[12] * b[12]);
        if (!(nq > 0)) return fail(PG_ERR_ARG, "pg_create_bare: zero quaternion");
        for (int k = 0; k < 7; k++) pose[o][k] = k < 3 ? b[6 + k] : b[6 + k] / nq;
    }
    int rc = check_device(device, "pg_create_bare"); if (rc != PG_OK) return rc;
    auto e = std::make_unique<pg_env>();
    e->task = PG_TASK_BARE; e->ctrl = CTRL_JOINTS; e->reward = 0; e->n = num_envs; e->device = device;
    e->nobj = n_bodies; e->obs_dim = 0; e->goal_dim = 0; e->act_dim = 0; e->max_steps = 0; e->state_dim = 18 + 13 * n_bodies + 1;
    // a world without a robot still carries one (the kernels are built around it): it is parked 1 km up, out of reach of everything
    const double parked[3] = {0.0, 0.0, 1000.0};
    rc = alloc_state(e.get(), precision, 0, 0, robot_base ? robot_base : parked); if (rc != PG_OK) return rc;
    Scene<double> S = make_scene<double>(TASK_REACH);
    S.nobj = n_bodies;
    for (int o = 0; o < n_bodies; o++) { const double* b = bodies + 13 * o; scene_set_obj(S, o, (int)b[0], b[1], b[2], b[3], b[4], b[5]); }
    if (table_rect) { S.table_x0 = table_rect[0]; S.table_x1 = table_rect[1]; S.table_y0 = table_rect[2]; S.table_y1 = table_rect[3]; }
    else { S.table_x0 = 1.0; S.table_x1 = -1.0; S.table_y0 = 1.0; S.table_y1 = -1.0; }     // empty rectangle: no table
    S.ground_z = ground_z ? *ground_z : -1e30;                                               // no plane: nothing to land on
    with_env(e.get(), [&](auto& E) {
        using T = std::remove_pointer_t<decltype(E.q)>;
        E.S = scene_cast<T>(S); E.P = make_task_params(TASK_REACH);
    });
    // initial state: joints at 0 (loadURDF), bodies at their creation poses, velocity motors (target 0, max impulse 1 per sub-step)
    std::vector<double> st((size_t)num_envs * e->state_dim, 0.0), mot((size_t)num_envs * 45, 0.0);
    for (int i = 0; i < num_envs; i++) {
        double* r = st.data() + (size_t)i * e->state_dim;
        for (int o = 0; o < n_bodies; o++) std::copy(pose[o], pose[o] + 7, r + 18 + 13 * o);
        for (int d = 0; d < 9; d++) { double* m = mot.data() + ((size_t)i * 9 + d) * 5; m[0] = 0.0; m[1] = 1.0; m[2] = 0.0; m[3] = 0.0; m[4] = 1.0 * 500.0; }
    }
    DevBuf d_st, d_mot;
    cudaError_t ce = cudaMalloc(&d_st.p, st.size() * sizeof(double)); if (ce == cudaSuccess) ce = cudaMalloc(&d_mot.p, mot.size() * sizeof(double));
    if (ce == cudaSuccess) ce = cudaMemcpy(d_st.p, st.data(), st.size() * sizeof(double), cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = cudaMemcpy(d_mot.p, mot.data(), mot.size() * sizeof(double), cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) return cuda_fail(ce, "pg_create_bare: initial state upload");
    rc = pg_set_state(e.get(), (const double*)d_st.p, nullptr, nullptr); if (rc != PG_OK) return rc;
    rc = pg_set_motors(e.get(), (const double*)d_mot.p, nullptr, nullptr); if (rc != PG_OK) return rc;
    ce = cudaDeviceSynchronize(); if (ce != cudaSuccess) return cuda_fail(ce, "pg_create_bare");
    *out = e.release();
    return PG_OK;
}

int pg_destroy(pg_env* e) { delete e; return PG_OK; }

int pg_dims(const pg_env* e, int* obs_dim, int* goal_dim, int* action_dim, int* max_episode_steps, int* state_dim) {
    if (!e) return fail(PG_ERR_ARG, "pg_dims: NULL handle");
    if (obs_dim) *obs_dim = e->obs_dim; if (goal_dim) *goal_dim = e->goal_dim; if (action_dim) *action_dim = e->act_dim;
    if (max_episode_steps) *max_episode_steps = e->max_steps; if (state_dim) *state_dim = e->state_dim;
    return PG_OK;
}

int pg_reset(pg_env* e, const unsigned char* mask, const unsigned long long* seeds, const double* goal_override, const double* object_override, float* obs, float* ag,
             float* dg, void* stream) {
    if (!e) return fail(PG_ERR_ARG, "pg_reset: NULL handle");
    if (e->task == PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_reset: a bare world has no task to reset; use pg_set_state");
    PG_CUDA(cudaSetDevice(e->device));
    ResetIO io{mask, goal_override, object_override, obs, ag, dg, seeds};
    with_env(e, [&](auto& E) {
        using T = std::remove_pointer_t<decltype(E.q)>;
        dispatch<0, 1, 2, 3, 4, 5>(e->task, [&](auto K) { launch_reset<T, K>(E, io, (cudaStream_t)stream); });
    });
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}

int pg_set_action_scale(pg_env* e, double ee_scale, double finger_scale) {
    if (!e || !(ee_scale > 0) || !(finger_scale > 0)) return fail(PG_ERR_ARG, "pg_set_action_scale: bad argument");
    with_env(e, [&](auto& E) { E.M.ee_scale = ee_scale; E.M.finger_scale = finger_scale; });
    return PG_OK;
}
int pg_set_task_params(pg_env* e, double distance_threshold, const double* goal_range_low, const double* goal_range_high, const double* obj_range_low, const double* obj_range_high) {
    if (!e || e->task == PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_set_task_params: needs a task handle");
    if (!(distance_threshold >= 0)) return fail(PG_ERR_ARG, "pg_set_task_params: distance_threshold must be >= 0");
    TaskParams P = with_env(e, [](auto& E) { return E.P; });
    P.thr64 = distance_threshold; P.thr32 = (float)distance_threshold;
    for (int k = 0; k < 3; k++) { if (goal_range_low) P.goal_lo[k] = goal_range_low[k]; if (goal_range_high) P.goal_hi[k] = goal_range_high[k]; }
    for (int k = 0; k < 2; k++) { if (obj_range_low) P.obj_lo[k] = obj_range_low[k]; if (obj_range_high) P.obj_hi[k] = obj_range_high[k]; }
    for (int k = 0; k < 3; k++) if (!(P.goal_lo[k] <= P.goal_hi[k])) return fail(PG_ERR_ARG, "pg_set_task_params: goal range low > high");
    for (int k = 0; k < 2; k++) if (!(P.obj_lo[k] <= P.obj_hi[k])) return fail(PG_ERR_ARG, "pg_set_task_params: object range low > high");
    with_env(e, [&](auto& E) { E.P = P; });
    return PG_OK;
}
int pg_set_substeps(pg_env* e, int n_substeps) {
    if (!e || e->task == PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_set_substeps: needs a task handle (bare worlds pass the count to pg_sim_step)");
    if (n_substeps < 1 || n_substeps > 1000) return fail(PG_ERR_ARG, "pg_set_substeps: 1 <= n_substeps <= 1000");
    with_env(e, [&](auto& E) { E.P.nsub = n_substeps; });
    return PG_OK;
}
int pg_step(pg_env* e, const float* actions, const float* target_quat, float* obs, float* ag, float* dg, float* reward, unsigned char* terminated,
            unsigned char* truncated, int auto_reset, float* contacts, unsigned char* contact_count, void* stream) {
    if (!e || !actions) return fail(PG_ERR_ARG, "pg_step: NULL handle or actions");
    if (e->task == PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_step: a bare world is advanced with pg_sim_step");
    if (target_quat && e->ctrl != CTRL_EE) return fail(PG_ERR_ARG, "pg_step: a target orientation needs ee control");
    return with_env(e, [&](auto& E) {
        return step_impl(e, E, actions, target_quat, obs, ag, dg, reward, terminated, truncated, auto_reset, contacts, contact_count, (cudaStream_t)stream, nullptr);
    });
}
int pg_max_contacts(const pg_env* e, int* per_env) {
    if (!e || !per_env) return fail(PG_ERR_ARG, "pg_max_contacts: NULL argument");
    if (e->task == PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_max_contacts: bare worlds have no contact report");
    *per_env = max_contacts(e->nobj);
    return PG_OK;
}

int pg_host_pin(void* ptr, size_t bytes) {
    if (!ptr || bytes == 0) return fail(PG_ERR_ARG, "pg_host_pin: bad argument");
    PG_CUDA(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
    return PG_OK;
}
int pg_host_unpin(void* ptr) {
    if (!ptr) return fail(PG_ERR_ARG, "pg_host_unpin: NULL");
    PG_CUDA(cudaHostUnregister(ptr));
    return PG_OK;
}

int pg_step_host(pg_env* e, const float* actions, float* obs, float* ag, float* dg, float* reward, unsigned char* terminated, unsigned char* truncated, int auto_reset) {
    if (!e || !actions) return fail(PG_ERR_ARG, "pg_step_host: NULL handle or actions");
    if (e->task == PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_step_host: a bare world is advanced with pg_sim_step");
    PG_CUDA(cudaSetDevice(e->device));
    const size_t n = (size_t)e->n, O = e->obs_dim, G = e->goal_dim, act_bytes = n * e->act_dim * sizeof(float);
    // the outputs share one device slab and its pinned mirror: obs | ag | dg | reward | terminated | truncated
    void* user[6] = {obs, ag, dg, reward, terminated, truncated};
    const size_t bytes[6] = {n * O * sizeof(float), n * G * sizeof(float), n * G * sizeof(float), n * sizeof(float), n, n};
    size_t off[7] = {0};
    for (int k = 0; k < 6; k++) off[k + 1] = off[k] + bytes[k];
    Staging& s = e->host;
    int rc = s.reserve(act_bytes, off[6]); if (rc != PG_OK) return rc;
    char* dev = (char*)s.d_out.p;
    void* host[6];
    for (int k = 0; k < 6; k++) host[k] = host_target(user[k], (char*)s.h_out.p + off[k]);
    HostIO hio{(const float*)host_source(actions, s.h_in.p, act_bytes), (float*)host[0], (float*)host[1], (float*)host[2], (float*)host[3],
               (unsigned char*)host[4], (unsigned char*)host[5]};
    rc = with_env(e, [&](auto& E) {
        return step_impl(e, E, (float*)s.d_in.p, nullptr, (float*)(dev + off[0]), (float*)(dev + off[1]), (float*)(dev + off[2]), (float*)(dev + off[3]),
                         (unsigned char*)(dev + off[4]), (unsigned char*)(dev + off[5]), auto_reset, nullptr, nullptr, s.st.p, &hio);
    });
    if (rc != PG_OK) return rc;
    PG_CUDA(cudaStreamSynchronize(s.st.p));
    for (int k = 0; k < 6; k++) copy_back(user[k], host[k], bytes[k]);
    return PG_OK;
}

int pg_compute_reward(int task, int reward_type, double threshold, const void* ag, const void* dg, float* reward, long long m, int dtype, void* stream) {
    if (m == 0) return PG_OK;       // an empty batch is valid (its pointers may be NULL)
    if (!valid_task(task) || !valid_reward_type(reward_type) || !ag || !dg || !reward || m < 0 || !(threshold >= 0)) return fail(PG_ERR_ARG, "pg_compute_reward: bad argument");
    with_dtype(dtype, [&](auto x) {
        using E = decltype(x);
        launch_reward<E, true>(task, (const E*)ag, (const E*)dg, reward, nullptr, m, reward_type, threshold, (cudaStream_t)stream);
    });
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
int pg_is_success(int task, double threshold, const void* ag, const void* dg, unsigned char* success, long long m, int dtype, void* stream) {
    if (m == 0) return PG_OK;
    if (!valid_task(task) || !ag || !dg || !success || m < 0 || !(threshold >= 0)) return fail(PG_ERR_ARG, "pg_is_success: bad argument");
    with_dtype(dtype, [&](auto x) {
        using E = decltype(x);
        launch_reward<E, false>(task, (const E*)ag, (const E*)dg, nullptr, success, m, 0, threshold, (cudaStream_t)stream);
    });
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
int pg_her_relabel(int task, int reward_type, double threshold, const void* next_ag, const void* dg, long long pitch, const long long* src, const long long* goal_src,
                   void* dg_out, void* ag_out, float* reward, long long m, int dtype, void* stream) {
    if (m == 0) return PG_OK;
    if (!valid_task(task) || !valid_reward_type(reward_type) || !next_ag || !dg || !src || !goal_src || !dg_out || !reward || m < 0 || !(threshold >= 0))
        return fail(PG_ERR_ARG, "pg_her_relabel: bad argument");
    if (pitch < task_goal_dim(task)) return fail(PG_ERR_ARG, "pg_her_relabel: the row pitch is smaller than the goal dimension");
    with_dtype(dtype, [&](auto x) {
        using E = decltype(x);
        launch_her<E>(task, (const E*)next_ag, (const E*)dg, src, goal_src, (E*)dg_out, (E*)ag_out, reward, m, pitch, reward_type, threshold, (cudaStream_t)stream);
    });
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
// Host-array entry points (the path stable-baselines3's HerReplayBuffer takes through env_method("compute_reward"), reference
// panda_gym/envs/core.py:226, examples/train_push.py:1-12).  They stage through one Staging per device: after the first call of a
// given size there is no allocation, its stream carries H2D -> kernel -> D2H, one stream synchronisation at the end.  The stages
// are never destroyed: at process exit the CUDA runtime may be gone before static destructors run.
static Staging* const device_stages = new Staging[64];
long long pg_host_stage_allocations(void) {
    long long allocs = 0;
    for (int d = 0; d < 64; d++) allocs += device_stages[d].allocs;
    return allocs;
}
static int reward_host(bool want_reward, int task, int reward_type, double thr, const void* ag, const void* dg, void* result, long long m, int dtype, int device) {
    if (device < 0 || device >= 64) return fail(PG_ERR_ARG, "host path: bad device index");
    int rc = check_device(device, "host path"); if (rc != PG_OK) return rc;
    const size_t es = with_dtype(dtype, [](auto x) { return sizeof(x); }), bytes = (size_t)m * task_goal_dim(task) * es, out_bytes = (size_t)m * (want_reward ? 4 : 1);
    const size_t dg_off = (bytes + 255) & ~(size_t)255;      // dg 256-byte aligned like ag: reward_kernel's 16-byte loads need both
    Staging& s = device_stages[device];
    rc = s.reserve(dg_off + bytes, out_bytes); if (rc != PG_OK) return rc;
    char *d_in = (char*)s.d_in.p, *h_in = (char*)s.h_in.p;
    PG_CUDA(cudaMemcpyAsync(d_in, host_source(ag, h_in, bytes), bytes, cudaMemcpyHostToDevice, s.st.p));
    PG_CUDA(cudaMemcpyAsync(d_in + dg_off, host_source(dg, h_in + dg_off, bytes), bytes, cudaMemcpyHostToDevice, s.st.p));
    rc = want_reward ? pg_compute_reward(task, reward_type, thr, d_in, d_in + dg_off, (float*)s.d_out.p, m, dtype, s.st.p)
                     : pg_is_success(task, thr, d_in, d_in + dg_off, (unsigned char*)s.d_out.p, m, dtype, s.st.p);
    if (rc != PG_OK) return rc;
    void* host = host_target(result, s.h_out.p);
    PG_CUDA(cudaMemcpyAsync(host, s.d_out.p, out_bytes, cudaMemcpyDeviceToHost, s.st.p));
    PG_CUDA(cudaStreamSynchronize(s.st.p));
    copy_back(result, host, out_bytes);
    return PG_OK;
}
int pg_compute_reward_host(int task, int reward_type, double threshold, const void* ag, const void* dg, float* reward, long long m, int dtype, int device) {
    if (m == 0) return PG_OK;
    if (!valid_task(task) || !valid_reward_type(reward_type) || !ag || !dg || !reward || m < 0 || !(threshold >= 0)) return fail(PG_ERR_ARG, "pg_compute_reward_host: bad argument");
    return reward_host(true, task, reward_type, threshold, ag, dg, reward, m, dtype, device);
}
int pg_is_success_host(int task, double threshold, const void* ag, const void* dg, unsigned char* success, long long m, int dtype, int device) {
    if (m == 0) return PG_OK;
    if (!valid_task(task) || !ag || !dg || !success || m < 0 || !(threshold >= 0)) return fail(PG_ERR_ARG, "pg_is_success_host: bad argument");
    return reward_host(false, task, 0, threshold, ag, dg, success, m, dtype, device);
}

// Snapshots are stream-ordered: one device-to-device copy of the handle's single SoA allocation, enqueued on the caller's stream
// (the env groups' streams are joined back to that stream by every pg_step, so ordering on it is sufficient).  No device-wide
// synchronisation, no allocation when a removed snapshot's buffer can be reused -> a save / K x (restore, step) / remove loop can
// be captured in a CUDA graph after its first, warm-up execution.
int pg_save_state(pg_env* e, int* state_id, void* stream) {
    if (!e || !state_id) return fail(PG_ERR_ARG, "pg_save_state: NULL argument");
    PG_CUDA(cudaSetDevice(e->device));
    DevBuf p;
    if (!e->snap_pool.empty()) { p = std::move(e->snap_pool.back()); e->snap_pool.pop_back(); }
    else PG_CUDA(cudaMalloc(&p.p, e->blob_bytes));
    cudaError_t ce = cudaMemcpyAsync(p.p, e->blob.p, e->blob_bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    if (ce != cudaSuccess) { e->snap_pool.push_back(std::move(p)); return cuda_fail(ce, "cudaMemcpyAsync(snapshot)"); }
    *state_id = e->next_snap++; e->snaps[*state_id] = std::move(p);
    return PG_OK;
}
int pg_restore_state(pg_env* e, int state_id, void* stream) {
    if (!e) return fail(PG_ERR_ARG, "pg_restore_state: NULL handle");
    auto it = e->snaps.find(state_id);
    if (it == e->snaps.end()) return fail(PG_ERR_STATE, "pg_restore_state: unknown state id " + std::to_string(state_id));
    PG_CUDA(cudaSetDevice(e->device));
    PG_CUDA(cudaMemcpyAsync(e->blob.p, it->second.p, e->blob_bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return PG_OK;
}
// The buffer goes back to the handle's pool: copies that still read or write it are ordered before any later reuse as long as the
// caller keeps using the same stream for the handle (the contract of every entry point).
int pg_remove_state(pg_env* e, int state_id) {
    if (!e) return fail(PG_ERR_ARG, "pg_remove_state: NULL handle");
    auto it = e->snaps.find(state_id);
    if (it == e->snaps.end()) return fail(PG_ERR_STATE, "pg_remove_state: unknown state id " + std::to_string(state_id));
    e->snap_pool.push_back(std::move(it->second)); e->snaps.erase(it);
    return PG_OK;
}

int pg_get_state(pg_env* e, double* state, void* stream) {
    if (!e || !state) return fail(PG_ERR_ARG, "pg_get_state: NULL argument");
    return launch_per_env(e, stream, [&](auto& E, int grid, cudaStream_t st) { get_state_kernel<<<grid, BLOCK, 0, st>>>(E, e->nobj, e->goal_dim, state); });
}
int pg_set_state(pg_env* e, const double* state, const unsigned char* mask, void* stream) {
    if (!e || !state) return fail(PG_ERR_ARG, "pg_set_state: NULL argument");
    return launch_per_env(e, stream, [&](auto& E, int grid, cudaStream_t st) { set_state_kernel<<<grid, BLOCK, 0, st>>>(E, e->nobj, e->goal_dim, state, mask); });
}
static int launch_ik(pg_env* e, int link, const double* position, const double* orientation, double* joint_angles, int out7, void* stream) {
    return launch_per_env(e, stream, [&](auto& E, int grid, cudaStream_t st) { ik_kernel<<<grid, BLOCK, 0, st>>>(E, link, position, orientation, joint_angles, out7); });
}
int pg_inverse_kinematics(pg_env* e, const double* position, const double* orientation, double* joint_angles, void* stream) {
    if (!e || !position || !orientation || !joint_angles) return fail(PG_ERR_ARG, "pg_inverse_kinematics: NULL argument");
    return launch_ik(e, 11, position, orientation, joint_angles, 1, stream);
}
int pg_inverse_kinematics_link(pg_env* e, int link, const double* position, const double* orientation, double* joint_angles, void* stream) {
    if (!e || !position || !orientation || !joint_angles) return fail(PG_ERR_ARG, "pg_inverse_kinematics_link: NULL argument");
    if (link < 0 || link > 11) return fail(PG_ERR_ARG, "pg_inverse_kinematics_link: link must be 0..11");
    return launch_ik(e, link, position, orientation, joint_angles, 0, stream);
}
int pg_get_link_state(pg_env* e, int link, double* out, void* stream) {
    if (!e || !out) return fail(PG_ERR_ARG, "pg_get_link_state: NULL argument");
    if (link < 0 || link > 11) return fail(PG_ERR_ARG, "pg_get_link_state: link must be 0..11");
    return launch_per_env(e, stream, [&](auto& E, int grid, cudaStream_t st) { link_state_kernel<<<grid, BLOCK, 0, st>>>(E, link, out); });
}
int pg_set_motors(pg_env* e, const double* motors, const unsigned char* mask, void* stream) {
    if (!e || !motors) return fail(PG_ERR_ARG, "pg_set_motors: NULL argument");
    if (e->task != PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_set_motors: task handles derive their motor targets from the action inside pg_step (Panda.set_action); raw motors exist on bare worlds");
    return launch_per_env(e, stream, [&](auto& E, int grid, cudaStream_t st) { set_motors_kernel<<<grid, BLOCK, 0, st>>>(E, motors, mask); });
}
int pg_get_motors(pg_env* e, double* motors, void* stream) {
    if (!e || !motors) return fail(PG_ERR_ARG, "pg_get_motors: NULL argument");
    if (e->task != PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_get_motors: bare worlds only");
    return launch_per_env(e, stream, [&](auto& E, int grid, cudaStream_t st) { get_motors_kernel<<<grid, BLOCK, 0, st>>>(E, motors); });
}
int pg_sim_step(pg_env* e, int n_substeps, void* stream) {
    if (!e || n_substeps < 0) return fail(PG_ERR_ARG, "pg_sim_step: bad argument");
    if (e->task != PG_TASK_BARE) return fail(PG_ERR_ARG, "pg_sim_step: task handles step through pg_step (controller + sub-steps + observation in one call)");
    if (n_substeps == 0) return PG_OK;
    PG_CUDA(cudaSetDevice(e->device));
    with_env(e, [&](auto& E) { launch_bare_step(E, e->nobj, n_substeps, (cudaStream_t)stream); });
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
static void fill_render_scene(pg_env* e) {
    RenderScene& R = e->rscene;
    memset(&R, 0, sizeof R);
    Scene<double> S; double bz;
    with_env(e, [&](auto& E) { S = scene_cast<double>(E.S); bz = E.M.base[2]; });
    R.nobj = e->nobj;
    R.has_table = S.table_x0 < S.table_x1; R.table[0] = (float)S.table_x0; R.table[1] = (float)S.table_x1; R.table[2] = (float)S.table_y0; R.table[3] = (float)S.table_y1; R.table_height = 0.4f;
    R.has_plane = S.ground_z > -1e29; R.plane_z = (float)S.ground_z;
    R.has_robot = bz < 500.0;                                  // a bare world without a robot parks it 1 km up
    const float bc[3] = {-0.04f, 0.0f, 0.07f}, bh[3] = {0.11f, 0.1f, 0.07f};     // panda_link0: approximate extents (its mesh is not available)
    for (int k = 0; k < 3; k++) { R.base_c[k] = bc[k]; R.base_h[k] = bh[k]; }
    for (int l = 0; l < 7; l++) for (int k = 0; k < 3; k++) { R.link_c[l][k] = (float)kLinks[l].com[k]; R.link_h[l][k] = (float)(0.5 * kLinks[l].box[k]); }
    const int rb_link[3] = {8, 9, 10};
    for (int b = 0; b < 3; b++) for (int k = 0; k < 3; k++) { R.link_c[rb_link[b]][k] = (float)S.rb_c[b][k]; R.link_h[rb_link[b]][k] = (float)S.rb_h[b][k]; }
}
int pg_render(pg_env* e, int width, int height, const double* camera, int crop, float* depth, unsigned char* rgba, unsigned char* segmentation, float* points,
              unsigned char* valid, void* stream) {
    if (!e || !camera || width <= 0 || height <= 0 || width > 4096 || height > 4096) return fail(PG_ERR_ARG, "pg_render: bad argument");
    if (valid && !points) return fail(PG_ERR_ARG, "pg_render: valid is the point cloud's mask, it needs points");
    PG_CUDA(cudaSetDevice(e->device));
    if (!e->prims.p) { PG_CUDA(cudaMalloc(&e->prims.p, (size_t)e->n * RENDER_MAX_PRIMS * sizeof(RenderPrim))); fill_render_scene(e); }
    // b3ComputeViewMatrixFromYawPitchRoll (up axis 2) + computeProjectionMatrixFOV(fov 60, near 0.1, far 100): pybullet.py:90-102
    const double rad = 0.01745329251994329547, yaw = camera[4] * rad, pitch = camera[5] * rad, roll = camera[6] * rad, dist = camera[3];
    const double cy = cos(yaw), sy = sin(yaw), cr = cos(roll), sr = sin(roll), cp = cos(pitch), sp = sin(pitch);
    // eyeRot.setEulerZYX(yaw, roll, pitch): R = Rz(yaw) Ry(roll) Rx(pitch)
    const double Rm[3][3] = {{cy * cr, cy * sr * sp - sy * cp, cy * sr * cp + sy * sp}, {sy * cr, sy * sr * sp + cy * cp, sy * sr * cp - cy * sp}, {-sr, cr * sp, cr * cp}};
    double eye[3], up[3], f[3], sv[3], u[3];
    for (int k = 0; k < 3; k++) { eye[k] = Rm[k][1] * -dist + camera[k]; up[k] = Rm[k][2]; f[k] = camera[k] - eye[k]; }
    double fl = sqrt(f[0] * f[0] + f[1] * f[1] + f[2] * f[2]);
    if (!(fl > 0)) return fail(PG_ERR_ARG, "pg_render: camera distance must be > 0");
    for (int k = 0; k < 3; k++) f[k] /= fl;
    sv[0] = f[1] * up[2] - f[2] * up[1]; sv[1] = f[2] * up[0] - f[0] * up[2]; sv[2] = f[0] * up[1] - f[1] * up[0];
    double sl = sqrt(sv[0] * sv[0] + sv[1] * sv[1] + sv[2] * sv[2]);
    for (int k = 0; k < 3; k++) sv[k] /= sl;
    u[0] = sv[1] * f[2] - sv[2] * f[1]; u[1] = sv[2] * f[0] - sv[0] * f[2]; u[2] = sv[0] * f[1] - sv[1] * f[0];
    RenderCamera C; memset(&C, 0, sizeof C);
    C.width = width; C.height = height; C.crop = crop;
    for (int k = 0; k < 3; k++) { C.eye[k] = (float)eye[k]; C.fwd[k] = (float)f[k]; C.right[k] = (float)sv[k]; C.up[k] = (float)u[k]; }
    C.tan_half_fov = (float)tan(30.0 * rad); C.aspect = (float)width / (float)height; C.near = 0.1f; C.far = 100.0f;
    const double l[3] = {0.35, -0.25, 0.9}; const double ll = sqrt(l[0] * l[0] + l[1] * l[1] + l[2] * l[2]);
    for (int k = 0; k < 3; k++) C.light[k] = (float)(l[k] / ll);
    const unsigned char col[RENDER_ID_ROBOT + 1][4] = {{0, 0, 0, 255}, {38, 38, 38, 255}, {242, 242, 242, 255},
                                                      {(unsigned char)(e->task == PG_TASK_STACK ? 26 : (e->task == PG_TASK_FLIP ? 255 : 26)), (unsigned char)(e->task == PG_TASK_STACK ? 26 : (e->task == PG_TASK_FLIP ? 255 : 230)),
                                                       (unsigned char)(e->task == PG_TASK_STACK ? 230 : (e->task == PG_TASK_FLIP ? 255 : 26)), 255},
                                                      {26, 230, 26, 255}, {235, 235, 235, 255}};     // plane 0.15, table 0.95, objects (tasks/ *.py rgba_color), robot
    memcpy(C.color, col, sizeof col);
    C.background[0] = 223; C.background[1] = 54; C.background[2] = 45; C.background[3] = 255;          // pybullet.py:28 default background_color
    with_env(e, [&](auto& E) { launch_render_setup(E, e->rscene, (RenderPrim*)e->prims.p, (cudaStream_t)stream); });
    launch_render((const RenderPrim*)e->prims.p, C, e->n, depth, rgba, segmentation, points, valid, (cudaStream_t)stream);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
int pg_get_ee_pose(pg_env* e, double* pose, void* stream) {
    if (!e || !pose) return fail(PG_ERR_ARG, "pg_get_ee_pose: NULL argument");
    return launch_per_env(e, stream, [&](auto& E, int grid, cudaStream_t st) { ee_pose_kernel<<<grid, BLOCK, 0, st>>>(E, pose); });
}
int pg_debug_schedule(pg_env* e, unsigned short* key_host, int* perm_host) {
    if (!e || !key_host || !perm_host) return fail(PG_ERR_ARG, "pg_debug_schedule: NULL argument");
    PG_CUDA(cudaSetDevice(e->device));
    const unsigned short* key = nullptr; const int* perm = nullptr;
    with_env(e, [&](auto& E) { key = E.ccount; perm = E.perm; });
    PG_CUDA(cudaMemcpy(key_host, key, (size_t)e->n * sizeof(unsigned short), cudaMemcpyDeviceToHost));
    PG_CUDA(cudaMemcpy(perm_host, perm, (size_t)e->n * sizeof(int), cudaMemcpyDeviceToHost));
    return PG_OK;
}
int pg_debug_timing(pg_env* e, long long* out) {
    if (!e || !out) return fail(PG_ERR_ARG, "pg_debug_timing: NULL argument");
    if (!e->dbg.p) return fail(PG_ERR_ARG, "pg_debug_timing: create the handle with PG_DEBUG_TIMING=1 in the environment");
    PG_CUDA(cudaSetDevice(e->device));
    PG_CUDA(cudaDeviceSynchronize());
    PG_CUDA(cudaMemcpy(out, e->dbg.p, (size_t)e->n * 2 * sizeof(long long), cudaMemcpyDeviceToHost));
    return PG_OK;
}
int pg_contact_overflows(pg_env* e, long long* count) {
    if (!e || !count) return fail(PG_ERR_ARG, "pg_contact_overflows: NULL argument");
    double d = 0;
    const int rc = read_stats(e, 5, 1, &d);
    if (rc == PG_OK) *count = (long long)d;
    return rc;
}
int pg_diverged(pg_env* e, long long* count) {
    if (!e || !count) return fail(PG_ERR_ARG, "pg_diverged: NULL argument");
    double d = 0;
    const int rc = read_stats(e, 4, 1, &d);
    if (rc == PG_OK) *count = (long long)d;
    return rc;
}
int pg_stats(pg_env* e, double out[4]) {
    if (!e || !out) return fail(PG_ERR_ARG, "pg_stats: NULL argument");
    return read_stats(e, 0, 4, out);
}

}  // extern "C"

// Motion primitives: one allocation holds the plan rows (MotionPlan) and the step's scratch actions / orientations.
struct pg_motion {
    int n, device;
    DevBuf blob;
    MotionPlan P;
    ~pg_motion() { cudaSetDevice(device); }          // blob is freed after this body runs, on the plan's device
};
// the checks every motion entry point makes on its (plan, env) pair
static int motion_env(pg_motion* m, pg_env* e, const char* who) {
    if (!m || !e) return fail(PG_ERR_ARG, std::string(who) + ": NULL plan or env");
    if (m->n != e->n || m->device != e->device) return fail(PG_ERR_ARG, std::string(who) + ": the plan was created for another batch size or device");
    if (e->task == PG_TASK_BARE) return fail(PG_ERR_STATE, std::string(who) + ": a bare world has no ee action to drive");
    if (e->ctrl != CTRL_EE) return fail(PG_ERR_STATE, std::string(who) + ": the motion primitives need an ee-controlled handle");
    return PG_OK;
}

extern "C" {

int pg_motion_create(int num_envs, int device, pg_motion** out) {
    if (!out) return fail(PG_ERR_ARG, "pg_motion_create: out is NULL");
    if (num_envs <= 0) return fail(PG_ERR_ARG, "pg_motion_create: num_envs must be > 0");
    int rc = check_device(device, "pg_motion_create"); if (rc != PG_OK) return rc;
    const size_t n = (size_t)num_envs;
    const size_t f_bytes = MP_ROWS * n * sizeof(double), i_bytes = 3 * n * sizeof(int), act_bytes = 4 * n * sizeof(float), quat_bytes = 4 * n * sizeof(float);
    auto m = std::make_unique<pg_motion>();
    m->n = num_envs; m->device = device;
    cudaError_t ce = cudaMalloc(&m->blob.p, f_bytes + i_bytes + act_bytes + quat_bytes);
    if (ce == cudaSuccess) ce = cudaMemset(m->blob.p, 0, f_bytes + i_bytes + act_bytes + quat_bytes);      // every env idle
    if (ce != cudaSuccess) return cuda_fail(ce, "pg_motion_create");
    char* b = (char*)m->blob.p;
    m->P.n = num_envs;
    m->P.f = (double*)b; b += f_bytes;
    m->P.kind = (int*)b; m->P.step = m->P.kind + n; m->P.count = m->P.kind + 2 * n; b += i_bytes;
    m->P.act = (float*)b; b += act_bytes;
    m->P.quat = (float*)b;
    *out = m.release();
    return PG_OK;
}
int pg_motion_destroy(pg_motion* m) { delete m; return PG_OK; }
int pg_motion_move(pg_motion* m, pg_env* e, const double* goal_pos, const double* goal_quat, const unsigned char* mask, void* stream) {
    int rc = motion_env(m, e, "pg_motion_move"); if (rc != PG_OK) return rc;
    if (!goal_pos || !goal_quat) return fail(PG_ERR_ARG, "pg_motion_move: NULL goal_pos or goal_quat");
    PG_CUDA(cudaSetDevice(e->device));
    with_env(e, [&](auto& E) { launch_motion_move(E, m->P, goal_pos, goal_quat, mask, (cudaStream_t)stream); });
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
int pg_motion_gripper(pg_motion* m, pg_env* e, double finger_action, int steps, const unsigned char* mask, void* stream) {
    if (steps < 0) return fail(PG_ERR_ARG, "pg_motion_gripper: steps must be >= 0");
    int rc = motion_env(m, e, "pg_motion_gripper"); if (rc != PG_OK) return rc;
    if (task_block_gripper(e->task)) return fail(PG_ERR_STATE, "pg_motion_gripper: this task blocks the gripper (Reach, Push, Slide have no finger action)");
    PG_CUDA(cudaSetDevice(e->device));
    launch_motion_gripper(m->P, finger_action, steps, mask, (cudaStream_t)stream);
    PG_CUDA(cudaGetLastError());
    return PG_OK;
}
int pg_motion_step(pg_motion* m, pg_env* e, float* obs, float* ag, float* dg, float* reward, unsigned char* terminated, unsigned char* truncated,
                   int* remaining, void* stream) {
    int rc = motion_env(m, e, "pg_motion_step"); if (rc != PG_OK) return rc;
    PG_CUDA(cudaSetDevice(e->device));
    return with_env(e, [&](auto& E) {
        launch_motion_step(E, m->P, e->act_dim, remaining, (cudaStream_t)stream);
        return step_impl(e, E, m->P.act, m->P.quat, obs, ag, dg, reward, terminated, truncated, 0, nullptr, nullptr, (cudaStream_t)stream, nullptr);
    });
}

}  // extern "C"
