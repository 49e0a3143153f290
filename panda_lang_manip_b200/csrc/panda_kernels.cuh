// panda_kernels.cuh -- the CUDA kernels: one thread per environment, structure-of-arrays state in HBM, I/O rows staged
// through shared memory so that every global access is a coalesced (and where aligned, 16-byte) transaction, the whole
// env step (controller, 20 sub-steps, observation, reward, optional auto-reset) fused into one launch so the state is read
// once and written once per step.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "panda_env.cuh"

namespace pg {

constexpr int BLOCK = 128;
// envs per block of the step kernel (a block is what the SM schedules and frees: smaller blocks release their shared memory and warp
// slots as soon as their own envs are done)
constexpr int STEP_BLOCK = 128;

template <typename T> struct EnvDev {
    int n;                       // environments on this device
    int reward_type;
    long long id0;               // global index of env 0 (RNG key)
    unsigned long long seed;
    T* q;                        // [9][n]
    T* qd;                       // [9][n]
    T* obj;                      // [nobj][13][n]  pos3 quat4 lin3 ang3
    double* goal;                // [6][n] task goal, float64 whatever the simulation precision (core.py:285-288 evaluates success / reward against the float64 goal)
    T* target;                   // [9][n] motor targets of the step in flight (only live between the segments of a cut step); bare worlds: the motors' target angles
    T* motor;                    // bare worlds only: [4][9][n] position gain, velocity gain, target velocity, max impulse per sub-step (setJointMotorControlArray state)
    int* steps;                  // [n] steps since reset (TimeLimit)
    unsigned* episode;           // [n] episodes started (RNG counter)
    float* ret;                  // [n] running episode return
    double* stats;               // [6] episodes, successes, return sum, length sum, diverged envs, contact candidates dropped at the cap
    int* perm;                   // [n] thread -> env map of the next launch (contact-heavy envs first), or NULL
    int t0, tcount;              // sorted path: this launch covers the thread slots [t0, t0 + tcount) of perm (one env group)
    unsigned short* ccount;      // [n] scheduling key written by the env's last launch (see KEY_* in panda_env.cuh)
    long long* dbg;              // [n][2] per-thread-slot (cycles spent in env_step, key) of the last launch, or NULL (PG_DEBUG_TIMING=1)
    int* hist;                   // [ceil(n/1024)][24] scratch of the bucket sort
    Model<T> M;
    Scene<T> S;
    TaskParams P;
};
struct StepIO {
    const float* target_quat;    // [n,4] (x,y,z,w) EE target orientation for ee control, or NULL = (1,0,0,0)
    const float* actions; float* obs; float* ag; float* dg; float* reward; unsigned char* terminated; unsigned char* truncated;
    int auto_reset;
    int s0, s1;                  // sub-step range of this launch: [0, nsub) = a whole step
    float* contacts;             // [n, max_contacts(nobj), REPORT_WORDS] contact report of the step's last sub-step, or NULL
    unsigned char* contact_count;   // [n] its rows per env, or NULL
};
struct ResetIO {
    const unsigned char* mask; const double* goal_override; const double* object_override; float* obs; float* ag; float* dg;
    const unsigned long long* seeds;   // [n] per-env seeds (RobotTaskEnv.reset(seed=k), core.py:240-244: equal seeds give equal draws), or NULL = the handle's stream
};

// ---------------------------------------------------------------------------------------------- Philox4x32-10
struct Philox {
    uint32_t c[4], k[2], out[4]; int have;
    __device__ Philox(unsigned long long seed, unsigned long long env, uint32_t episode) {
        k[0] = (uint32_t)seed; k[1] = (uint32_t)(seed >> 32); c[0] = (uint32_t)env; c[1] = (uint32_t)(env >> 32); c[2] = episode; c[3] = 0; have = 0;
    }
    __device__ void round4() {
        uint32_t a[4] = {c[0], c[1], c[2], c[3]}, key[2] = {k[0], k[1]};
#pragma unroll
        for (int r = 0; r < 10; r++) {
            uint32_t hi0 = __umulhi(0xD2511F53u, a[0]), lo0 = 0xD2511F53u * a[0], hi1 = __umulhi(0xCD9E8D57u, a[2]), lo1 = 0xCD9E8D57u * a[2];
            uint32_t n0 = hi1 ^ a[1] ^ key[0], n1 = lo1, n2 = hi0 ^ a[3] ^ key[1], n3 = lo0;
            a[0] = n0; a[1] = n1; a[2] = n2; a[3] = n3; key[0] += 0x9E3779B9u; key[1] += 0xBB67AE85u;
        }
        out[0] = a[0]; out[1] = a[1]; out[2] = a[2]; out[3] = a[3]; c[3]++; have = 4;
    }
    __device__ uint32_t next() { if (have == 0) round4(); return out[4 - have--]; }
    __device__ double uniform() { uint32_t a = next() >> 5, b = next() >> 6; return (a * 67108864.0 + b) * (1.0 / 9007199254740992.0); }   // 53 bits, [0,1)
    __device__ double uniform(double lo, double hi) { return lo + (hi - lo) * uniform(); }
    __device__ double normal() { double u1 = 1.0 - uniform(), u2 = uniform(); return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2); }
};

// ---------------------------------------------------------------------------------------------- I/O tiles
// rows [row0, row0 + BS) of a row-major [n, W] array <-> per-thread registers, through shared memory
template <int W, typename E, int BS = BLOCK> __device__ __forceinline__ void tile_load(E* s, const E* g, long long row0, int n, E* reg) {
    const long long base = row0 * W;
    const int cnt = (int)min((long long)BS, (long long)n - row0) * W;
    if (sizeof(E) == 4 && ((uintptr_t)(g + base) & 15) == 0) {
        const int c4 = cnt >> 2;
        for (int i = threadIdx.x; i < c4; i += BS) reinterpret_cast<float4*>(s)[i] = __ldg(reinterpret_cast<const float4*>(g + base) + i);
        for (int i = (c4 << 2) + threadIdx.x; i < cnt; i += BS) s[i] = g[base + i];
    } else {
        for (int i = threadIdx.x; i < cnt; i += BS) s[i] = g[base + i];
    }
    __syncthreads();
    if ((int)threadIdx.x * W < cnt) {
#pragma unroll
        for (int k = 0; k < W; k++) reg[k] = s[threadIdx.x * W + k];
    }
    __syncthreads();
}
// `write` is per-thread: rows whose thread passes write=false keep their previous contents
template <int W, typename E, int BS = BLOCK> __device__ __forceinline__ void tile_store(E* s, E* g, long long row0, int n, const E* reg, bool all_write, bool write) {
    if (g == nullptr) return;
    const long long base = row0 * W;
    const int cnt = (int)min((long long)BS, (long long)n - row0) * W;
    if (!all_write) {   // masked rows: each thread writes its own row directly
        if (write && (int)threadIdx.x * W < cnt) {
#pragma unroll
            for (int k = 0; k < W; k++) g[base + threadIdx.x * W + k] = reg[k];
        }
        return;
    }
    if ((int)threadIdx.x * W < cnt) {
#pragma unroll
        for (int k = 0; k < W; k++) s[threadIdx.x * W + k] = reg[k];
    }
    __syncthreads();
    if (sizeof(E) == 4 && ((uintptr_t)(g + base) & 15) == 0) {
        const int c4 = cnt >> 2;
        for (int i = threadIdx.x; i < c4; i += BS) reinterpret_cast<float4*>(g + base)[i] = reinterpret_cast<const float4*>(s)[i];
        for (int i = (c4 << 2) + threadIdx.x; i < cnt; i += BS) g[base + i] = s[i];
    } else {
        for (int i = threadIdx.x; i < cnt; i += BS) g[base + i] = s[i];
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------- SoA state access
template <typename T, int NOBJ> __device__ __forceinline__ void load_state(const EnvDev<T>& E, int i, T* q, T* qd, Obj<T>* ob) {
    const int n = E.n;
#pragma unroll
    for (int d = 0; d < ND; d++) { q[d] = E.q[d * n + i]; qd[d] = E.qd[d * n + i]; }
#pragma unroll
    for (int o = 0; o < NOBJ; o++) {
        const T* p = E.obj + (size_t)o * 13 * n + i;
        ob[o].pos = mk<T>(p[0], p[n], p[2 * n]); ob[o].qx = p[3 * n]; ob[o].qy = p[4 * n]; ob[o].qz = p[5 * n]; ob[o].qw = p[6 * n];
        ob[o].lin = mk<T>(p[7 * n], p[8 * n], p[9 * n]); ob[o].ang = mk<T>(p[10 * n], p[11 * n], p[12 * n]);
    }
}
template <typename T> __device__ __forceinline__ void load_goal(const EnvDev<T>& E, int i, double* goal) {
#pragma unroll
    for (int k = 0; k < 6; k++) goal[k] = E.goal[k * E.n + i];
}
template <typename T, int NOBJ> __device__ __forceinline__ void store_state(const EnvDev<T>& E, int i, const T* q, const T* qd, const Obj<T>* ob) {
    const int n = E.n;
#pragma unroll
    for (int d = 0; d < ND; d++) { E.q[d * n + i] = q[d]; E.qd[d * n + i] = qd[d]; }
#pragma unroll
    for (int o = 0; o < NOBJ; o++) {
        T* p = E.obj + (size_t)o * 13 * n + i;
        p[0] = ob[o].pos.x; p[n] = ob[o].pos.y; p[2 * n] = ob[o].pos.z; p[3 * n] = ob[o].qx; p[4 * n] = ob[o].qy; p[5 * n] = ob[o].qz; p[6 * n] = ob[o].qw;
        p[7 * n] = ob[o].lin.x; p[8 * n] = ob[o].lin.y; p[9 * n] = ob[o].lin.z; p[10 * n] = ob[o].ang.x; p[11 * n] = ob[o].ang.y; p[12 * n] = ob[o].ang.z;
    }
}

// ---------------------------------------------------------------------------------------------- reset
// Task.reset + Panda.reset for one env: neutral joints, zero velocity, sampled (or overridden) goal and object placement.
// Distributions: reach.py:22-23,51-54; push.py:69-87; slide.py:23-24,73-91; pick_and_place.py:65-85; stack.py:94-119;
// flip.py:63-80 (goal: uniform rotation, drawn from the device stream instead of scipy's unseeded global RNG).
template <typename T, int TASK>
__device__ __forceinline__ void env_reset(const EnvDev<T>& E, int i, uint32_t episode, const double* goal_ov, const double* obj_ov, T* q, T* qd, Obj<T>* ob, double* goal,
                                          const unsigned long long* seeds = nullptr) {
    constexpr int NOBJ = task_nobj(TASK);
    constexpr int G = task_goal_dim(TASK);
    const double neutral[ND] = {0.00, 0.41, 0.00, -1.85, 0.00, 2.26, 0.79, 0.00, 0.00};   // panda.py:45
#pragma unroll
    for (int d = 0; d < ND; d++) { q[d] = (T)neutral[d]; qd[d] = T(0); }
    // RNG stream: (handle seed, global env id, episode) -- or, for a seeded reset, the env's own seed alone, so that equal seeds
    // give equal goals / placements whatever the env index (test/seed_test.py semantics)
    Philox rng(seeds ? seeds[i] : E.seed, seeds ? 0xA5A5A5A5ull : (unsigned long long)(E.id0 + i), seeds ? 0u : episode);
    const TaskParams& P = E.P;
    double g[6] = {0, 0, 0, 0, 0, 0}, op[6] = {0, 0, 0, 0, 0, 0};
    const double z0 = TASK == TASK_SLIDE ? 0.03 : 0.02;         // object_size / 2: the height at which goals and objects sit on the table
    if (TASK == TASK_FLIP) { double a = rng.normal(), b = rng.normal(), c = rng.normal(), d = rng.normal(), nn = 1.0 / sqrt(a * a + b * b + c * c + d * d); g[0] = a * nn; g[1] = b * nn; g[2] = c * nn; g[3] = d * nn; }
    else {
        g[0] = rng.uniform(P.goal_lo[0], P.goal_hi[0]); g[1] = rng.uniform(P.goal_lo[1], P.goal_hi[1]);
        double z = (TASK == TASK_REACH || TASK == TASK_PICK_AND_PLACE) ? rng.uniform(P.goal_lo[2], P.goal_hi[2]) : 0.0;
        if (TASK == TASK_PICK_AND_PLACE && rng.uniform() < 0.3) z = 0.0;                       // pick_and_place.py:74-76: 30 % of the goals lie on the table
        g[2] = (TASK == TASK_REACH ? 0.0 : z0) + z;
        if (TASK == TASK_STACK) { g[3] = g[0]; g[4] = g[1]; g[5] = 0.06; }                    // stack.py:102-108: both goals share the noise
    }
#pragma unroll
    for (int o = 0; o < NOBJ; o++) {
        op[3 * o] = rng.uniform(P.obj_lo[0], P.obj_hi[0]); op[3 * o + 1] = rng.uniform(P.obj_lo[1], P.obj_hi[1]);
        op[3 * o + 2] = o == 1 ? 0.06 : z0;
    }
    if (goal_ov) {
#pragma unroll
        for (int k = 0; k < G; k++) g[k] = goal_ov[(size_t)i * G + k];
    }
    if (obj_ov) {
#pragma unroll
        for (int k = 0; k < 3 * NOBJ; k++) op[k] = obj_ov[(size_t)i * 3 * NOBJ + k];
    }
#pragma unroll
    for (int k = 0; k < 6; k++) goal[k] = g[k];
#pragma unroll
    for (int o = 0; o < NOBJ; o++) {
        ob[o].pos = mk<T>((T)op[3 * o], (T)op[3 * o + 1], (T)op[3 * o + 2]); ob[o].qx = T(0); ob[o].qy = T(0); ob[o].qz = T(0); ob[o].qw = T(1);
        ob[o].lin = mk<T>(T(0), T(0), T(0)); ob[o].ang = mk<T>(T(0), T(0), T(0));
    }
}

template <typename T, int TASK>
__global__ void __launch_bounds__(BLOCK) reset_kernel(const __grid_constant__ EnvDev<T> E, const ResetIO io) {
    constexpr int NOBJ = task_nobj(TASK), O = task_obs_dim(TASK), G = task_goal_dim(TASK);
    const long long row0 = (long long)blockIdx.x * BLOCK;
    const int i = (int)row0 + threadIdx.x;
    const bool valid = i < E.n;
    const bool mine = valid && (io.mask == nullptr || io.mask[i] != 0);
    float obs[O], ag[G], dg[G];
    if (mine) {
        T q[ND], qd[ND]; double goal[6]; Obj<T> ob[NOBJ > 0 ? NOBJ : 1];
        uint32_t ep = E.episode[i] + 1u;
        env_reset<T, TASK>(E, i, ep, io.goal_override, io.object_override, q, qd, ob, goal, io.seeds);
        store_state<T, NOBJ>(E, i, q, qd, ob);
#pragma unroll
        for (int k = 0; k < 6; k++) E.goal[k * E.n + i] = goal[k];
        E.steps[i] = 0; E.episode[i] = ep; E.ret[i] = 0.0f; E.ccount[i] = 0;
        env_observe<T, TASK>(E.M, q, qd, q, ob, goal, obs, ag, dg);
    }
    tile_store<O>((float*)nullptr, io.obs, row0, E.n, obs, false, mine);
    tile_store<G>((float*)nullptr, io.ag, row0, E.n, ag, false, mine);
    tile_store<G>((float*)nullptr, io.dg, row0, E.n, dg, false, mine);
}

// ---------------------------------------------------------------------------------------------- step
// Contact-aware scheduling.  Contact handling is the expensive, data-dependent part of a sub-step; with envs mapped to threads
// in index order nearly every warp holds a few envs in contact and runs that code at ~10% lane utilisation.  Before each launch
// the envs are therefore bucket-sorted by the key their previous launch wrote (KEY_* in panda_env.cuh): full-limit-sweep envs,
// envs with robot contacts, near ones, by contact count and solver cap -- heaviest first so the long blocks start early.
// This packs envs that will execute the same contact code into the same warps.  Two passes over 1024-env chunks.
constexpr int PERM_BUCKETS = 336, PERM_CHUNK = 1024, PERM_THREADS = 384;
__device__ __forceinline__ int perm_bucket(unsigned short key) {
    const int n = key & 0x1f, robot = (key >> 5) & 1, capped = (key >> 6) & 1, near = (key >> 7) & 1, full = (key >> 9) & 1;
    const int nq = n <= 10 ? n : 11 + min((n - 11) >> 2, 2);        // 0..13
    const int ngen = (key >> 10) & 15;
    const int cls = ngen > 0 ? 3 + min((ngen - 1) >> 1, 2) : (robot ? 2 : near);     // far, near, robot on table only, 1-2 / 3-4 / 5+ generic contacts
    return ((full * 6 + cls) * 14 + nq) * 2 + capped;
}
// pass 1: per-chunk bucket histogram
static __global__ void __launch_bounds__(PERM_THREADS) perm_hist_kernel(const unsigned short* __restrict__ key, int* __restrict__ hist, int n) {
    __shared__ int s_h[PERM_BUCKETS];
    if (threadIdx.x < PERM_BUCKETS) s_h[threadIdx.x] = 0;
    __syncthreads();
    const int base = blockIdx.x * PERM_CHUNK;
    for (int i = base + threadIdx.x; i < min(n, base + PERM_CHUNK); i += PERM_THREADS) atomicAdd(&s_h[perm_bucket(key[i])], 1);
    __syncthreads();
    if (threadIdx.x < PERM_BUCKETS) hist[blockIdx.x * PERM_BUCKETS + threadIdx.x] = s_h[threadIdx.x];
}
// pass 2: bucket-major offsets (heaviest bucket first; chunks in order inside a bucket) and scatter.  The order inside one chunk's
// slice of a bucket is arbitrary: the map only decides which thread runs which env, never a result.
// key / perm point at the group's first env / thread slot, id0 is that env's index
static __global__ void __launch_bounds__(PERM_THREADS) perm_scatter_kernel(const unsigned short* __restrict__ key, const int* __restrict__ hist, int* __restrict__ perm, int n, int nchunks, int id0) {
    __shared__ int s_pos[PERM_BUCKETS], s_warp[PERM_THREADS / 32];
    // thread t owns bucket PERM_BUCKETS-1-t (descending order): total over all chunks, prefix over the chunks before this one
    const int b = PERM_BUCKETS - 1 - (int)threadIdx.x;
    int tot = 0, pre = 0;
    if (b >= 0) for (int c = 0; c < nchunks; c++) { int h = hist[c * PERM_BUCKETS + b]; tot += h; if (c < (int)blockIdx.x) pre += h; }
    int x = tot;                                    // inclusive scan of the totals in descending bucket order
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, d); if ((threadIdx.x & 31) >= d) x += y; }
    if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = x;
    __syncthreads();
    int carry = 0;
    for (int w = 0; w < (int)(threadIdx.x >> 5); w++) carry += s_warp[w];
    if (b >= 0) s_pos[b] = carry + x - tot + pre;
    __syncthreads();
    const int base = blockIdx.x * PERM_CHUNK;
    for (int i = base + threadIdx.x; i < min(n, base + PERM_CHUNK); i += PERM_THREADS) perm[atomicAdd(&s_pos[perm_bucket(key[i])], 1)] = id0 + i;
}
template <int W, typename E> __device__ __forceinline__ void row_load(const E* g, int i, E* reg) {
#pragma unroll
    for (int k = 0; k < W; k++) reg[k] = g[(size_t)i * W + k];
}
template <int W, typename E> __device__ __forceinline__ void row_store(E* g, int i, const E* reg) {
    if (g == nullptr) return;
#pragma unroll
    for (int k = 0; k < W; k++) g[(size_t)i * W + k] = reg[k];
}

// Dynamic shared memory per block: solver_slots() words per thread of solver state (Jx + contact records, word-interleaved), aliased with
// the I/O row tile that is only live before and after the simulation phase.
// Threads per block: 128, except where the solver slab of 128 envs would exceed the 227 kB a block may own (fp64 parity mode on the
// two-object scene: 416 slots x 8 B x 128 = 426 kB) -- those run 32-env blocks.
constexpr size_t SMEM_LIMIT = 227 * 1024;
template <typename T, int TASK> constexpr int step_block() { return (size_t)solver_slots(task_nobj(TASK)) * STEP_BLOCK * sizeof(T) <= SMEM_LIMIT ? STEP_BLOCK : 32; }
template <typename T, int TASK, int CTRL> constexpr size_t step_smem_bytes() {
    constexpr int O = task_obs_dim(TASK), G = task_goal_dim(TASK), NA = task_act_dim(TASK, CTRL), BS = step_block<T, TASK>();
    constexpr int W = O > NA ? (O > G ? O : G) : (NA > G ? NA : G);
    constexpr size_t solver = (size_t)solver_slots(task_nobj(TASK)) * BS * sizeof(T), tile = (size_t)W * BS * sizeof(float);
    return solver > tile ? solver : tile;
}
template <typename T, int TASK, int CTRL>
__global__ void __launch_bounds__((step_block<T, TASK>())) step_kernel(const __grid_constant__ EnvDev<T> E, const StepIO io) {
    constexpr int NOBJ = task_nobj(TASK), O = task_obs_dim(TASK), G = task_goal_dim(TASK), NA = task_act_dim(TASK, CTRL), BS = step_block<T, TASK>();
    static_assert(step_smem_bytes<T, TASK, CTRL>() <= SMEM_LIMIT, "solver slab exceeds the per-block shared memory of sm_100");
    extern __shared__ __align__(16) unsigned char s_raw[];
    float* s_io = reinterpret_cast<float*>(s_raw);
    __shared__ double s_stats[6];
    const long long row0 = (long long)blockIdx.x * BS;
    const bool mapped = E.perm != nullptr;               // launch-uniform
    const int t = (int)row0 + threadIdx.x;
    const bool valid = t < (mapped ? E.tcount : E.n);
    const int i = (valid && mapped) ? E.perm[E.t0 + t] : t;
    if (threadIdx.x < 6) s_stats[threadIdx.x] = 0.0;
    __syncthreads();                                     // s_stats is zeroed before any warp can atomicAdd into it
    const bool first = io.s0 == 0, last = io.s1 == E.P.nsub;      // launch-uniform
    float act[NA];
    if (first) { if (mapped) { if (valid) row_load<NA>(io.actions, i, act); } else tile_load<NA, float, BS>(s_io, io.actions, row0, E.n, act); }
    float obs[O], ag[G], dg[G], reward = 0.0f;
    unsigned char term = 0, trunc = 0;
    if (valid) {
        T q[ND], qd[ND], target[ND], qc[ND]; Obj<T> ob[NOBJ > 0 ? NOBJ : 1];
        Contacts<T> C;
        C.st.base = reinterpret_cast<T*>(s_raw) + threadIdx.x; C.st.stride = BS; C.dropped = 0;
        load_state<T, NOBJ>(E, i, q, qd, ob);
        if (!first) {
#pragma unroll
            for (int d = 0; d < ND; d++) target[d] = E.target[d * E.n + i];
        }
        int sched_key = E.ccount[i];                // in: KEY_FULL of the previous key; out: this launch's key
        float tquat[4];
        if (first && io.target_quat) row_load<4>(io.target_quat, i, tquat);
        const long long clk0 = E.dbg ? clock64() : 0;
        env_step_sim<T, TASK, CTRL>(E.M, E.S, q, qd, ob, act, (first && io.target_quat) ? tquat : nullptr, C, sched_key, target, qc, io.s0, io.s1, E.P.nsub);
        if (E.dbg) { E.dbg[2 * (size_t)(E.t0 + t)] = clock64() - clk0; unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid)); E.dbg[2 * (size_t)(E.t0 + t) + 1] = (long long)sched_key | ((long long)smid << 16); }
        if (C.dropped > 0) atomicAdd(&s_stats[5], (double)C.dropped);
        if (last) {     // the report of the step that just ended: the records are still in this thread's column of the slab, before any reset
            if (io.contacts) {
                float* rows = io.contacts + (size_t)i * (max_contacts(NOBJ) * REPORT_WORDS);
                for (int c = 0; c < C.n; c++) contact_report_row(E.S, C, c, rows + c * REPORT_WORDS);
            }
            if (io.contact_count) io.contact_count[i] = (unsigned char)C.n;
        }
        double goal[6];
        if (last) {     // the goal is only needed now: loaded after the simulation so that it does not occupy registers across the solver
            load_goal(E, i, goal);
            env_step_finish<T, TASK>(E.M, E.reward_type, q, qd, qc, ob, goal, E.P.thr64, obs, ag, dg, reward, term);
        }
        if (last) {
            int steps = E.steps[i] + 1;
            trunc = steps >= task_max_steps(TASK);
            float ret = E.ret[i] + reward;
            // divergence guard: a non-finite state is counted and, with auto-reset, the episode is cut (truncated) and the env restarted
            T chk = T(0);
#pragma unroll
            for (int d = 0; d < ND; d++) chk += q[d] + qd[d];
#pragma unroll
            for (int o = 0; o < NOBJ; o++) chk += ob[o].pos.x + ob[o].pos.y + ob[o].pos.z + ob[o].qw + ob[o].lin.x + ob[o].lin.y + ob[o].lin.z + ob[o].ang.x + ob[o].ang.y + ob[o].ang.z;
            if (!(fabs(chk) < T(1e30))) { atomicAdd(&s_stats[4], 1.0); if (io.auto_reset) { trunc = 1; term = 0; reward = 0.0f; ret = E.ret[i]; } }
            if (io.auto_reset && (term || trunc)) {
                atomicAdd(&s_stats[0], 1.0); atomicAdd(&s_stats[1], (double)term); atomicAdd(&s_stats[2], (double)ret); atomicAdd(&s_stats[3], (double)steps);
                uint32_t ep = E.episode[i] + 1u;
                env_reset<T, TASK>(E, i, ep, nullptr, nullptr, q, qd, ob, goal);
#pragma unroll
                for (int k = 0; k < 6; k++) E.goal[k * E.n + i] = goal[k];
                E.episode[i] = ep; steps = 0; ret = 0.0f; sched_key = 0;
                env_observe<T, TASK>(E.M, q, qd, q, ob, goal, obs, ag, dg);
            }
            E.steps[i] = steps; E.ret[i] = ret;
        } else {
#pragma unroll
            for (int d = 0; d < ND; d++) E.target[d * E.n + i] = target[d];
        }
        store_state<T, NOBJ>(E, i, q, qd, ob);
        E.ccount[i] = (unsigned short)sched_key;
    }
    if (!last) {        // (launch-uniform) only the overflow counter can be non-zero before the step's last segment
        __syncthreads();
        if (threadIdx.x == 5 && s_stats[5] != 0.0) atomicAdd(&E.stats[5], s_stats[5]);
        return;
    }
    __syncthreads();    // the solver slab is dead for every thread of the block: reuse it as the output tile
    if (mapped) {
        if (valid) { row_store<O>(io.obs, i, obs); row_store<G>(io.ag, i, ag); row_store<G>(io.dg, i, dg); }
    } else {
        tile_store<O, float, BS>(s_io, io.obs, row0, E.n, obs, true, valid);
        tile_store<G, float, BS>(s_io, io.ag, row0, E.n, ag, true, valid);
        tile_store<G, float, BS>(s_io, io.dg, row0, E.n, dg, true, valid);
    }
    if (valid) {
        if (io.reward) io.reward[i] = reward;
        if (io.terminated) io.terminated[i] = term;
        if (io.truncated) io.truncated[i] = trunc;
    }
    __syncthreads();
    if (threadIdx.x < 6 && s_stats[threadIdx.x] != 0.0) atomicAdd(&E.stats[threadIdx.x], s_stats[threadIdx.x]);
}

// ---------------------------------------------------------------------------------------------- raw state exchange / IK
// rows [q(9) qd(9) | per object pos3 quat4 lin3 ang3 | goal(G) | episode step] in float64; nobj / G are runtime (task and bare handles)
template <typename T>
__global__ void __launch_bounds__(BLOCK) get_state_kernel(const __grid_constant__ EnvDev<T> E, int nobj, int G, double* out) {
    const int SD = 18 + 13 * nobj + G + 1;
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= E.n) return;
    double* r = out + (size_t)i * SD; const int n = E.n;
    for (int d = 0; d < ND; d++) { r[d] = E.q[d * n + i]; r[9 + d] = E.qd[d * n + i]; }
    for (int k = 0; k < 13 * nobj; k++) r[18 + k] = E.obj[(size_t)k * n + i];
    for (int k = 0; k < G; k++) r[18 + 13 * nobj + k] = E.goal[k * n + i];
    r[SD - 1] = E.steps[i];
}
template <typename T>
__global__ void __launch_bounds__(BLOCK) set_state_kernel(const __grid_constant__ EnvDev<T> E, int nobj, int G, const double* in, const unsigned char* mask) {
    const int SD = 18 + 13 * nobj + G + 1;
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= E.n || (mask && !mask[i])) return;
    const double* r = in + (size_t)i * SD; const int n = E.n;
    for (int d = 0; d < ND; d++) { E.q[d * n + i] = (T)r[d]; E.qd[d * n + i] = (T)r[9 + d]; }
    for (int k = 0; k < 13 * nobj; k++) E.obj[(size_t)k * n + i] = (T)r[18 + k];
    for (int k = 0; k < G; k++) E.goal[k * n + i] = r[18 + 13 * nobj + k];
    E.steps[i] = (int)r[SD - 1];
}
// calculateInverseKinematics (pybullet.py:479-497) on `link` from the current joint state: target [n,3] + quaternion [n,4] (normalised
// here; the reference's KAT test/pybullet_test.py:265 passes an un-normalised one) -> 9 joint values.  link 11 with out7 != 0 is the
// env path's fixed instance (ik_ee, 7 arm angles per row).
template <typename T>
__global__ void __launch_bounds__(BLOCK) ik_kernel(const __grid_constant__ EnvDev<T> E, int link, const double* pos, const double* quat, double* out, int out7) {
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= E.n) return;
    T q[ND], tq[4], o[ND];
    for (int d = 0; d < ND; d++) q[d] = E.q[d * E.n + i];
    double nn = 0; for (int k = 0; k < 4; k++) nn += quat[(size_t)i * 4 + k] * quat[(size_t)i * 4 + k];
    nn = 1.0 / sqrt(nn);
    for (int k = 0; k < 4; k++) tq[k] = (T)(quat[(size_t)i * 4 + k] * nn);
    const V3<T> p = mk<T>((T)pos[(size_t)i * 3], (T)pos[(size_t)i * 3 + 1], (T)pos[(size_t)i * 3 + 2]);
    if (out7) { ik_ee(E.M, q, p, tq, o); for (int d = 0; d < 7; d++) out[(size_t)i * 7 + d] = (double)o[d]; }
    else { ik_link(E.M, link, q, p, tq, o); for (int d = 0; d < ND; d++) out[(size_t)i * ND + d] = (double)o[d]; }
}
// getLinkState for any link 0..11 (pybullet.py:351-400): rows [pos3 quat4 lin3 ang3] float64; pose from the link-transform cache
// FK(q - qd dt), velocity from the fresh state rotated by the cached basis (SURVEY App. B.5)
template <typename T>
__global__ void __launch_bounds__(BLOCK) link_state_kernel(const __grid_constant__ EnvDev<T> E, int link, double* out) {
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= E.n) return;
    T q[ND], qd[ND], qc[ND], qt[4];
    for (int d = 0; d < ND; d++) { q[d] = E.q[d * E.n + i]; qd[d] = E.qd[d * E.n + i]; qc[d] = q[d] - qd[d] * Consts<T>::dt; }
    V3<T> p, l, a;
    link_state(E.M, link, q, qd, qc, p, qt, l, a);
    double* r = out + (size_t)i * 13;
    r[0] = p.x; r[1] = p.y; r[2] = p.z; r[3] = qt[0]; r[4] = qt[1]; r[5] = qt[2]; r[6] = qt[3];
    r[7] = l.x; r[8] = l.y; r[9] = l.z; r[10] = a.x; r[11] = a.y; r[12] = a.z;
}

// ---------------------------------------------------------------------------------------------- bare world (the sim facade without a task)
// What the reference's PyBullet facade is when used directly (panda_gym/pybullet.py: loadURDF + create_box + control_joints + step;
// its own tests test/pybullet_test.py:56-65,110-204 do exactly that): a robot whose nine motors are whatever
// setJointMotorControlArray left them (after loadURDF: velocity motors, target 0, max impulse 1 -- SURVEY App. B.1), up to two
// free bodies, optional table / ground plane, and `nsub` x stepSimulation per call.  One thread per world; same sub-step code as the
// env path (env_substep) with the generic motor rows.
constexpr int BARE_BLOCK = 32;
template <typename T, int NOBJ> constexpr size_t bare_smem_bytes() { return (size_t)solver_slots(NOBJ) * BARE_BLOCK * sizeof(T); }
template <typename T, int NOBJ>
__global__ void __launch_bounds__(BARE_BLOCK) bare_step_kernel(const __grid_constant__ EnvDev<T> E, int nsub) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int i = blockIdx.x * BARE_BLOCK + threadIdx.x;
    if (i >= E.n) return;
    const int n = E.n;
    T q[ND], qd[ND], target[ND], mot[27]; Obj<T> ob[NOBJ > 0 ? NOBJ : 1];
    Contacts<T> C;
    C.st.base = reinterpret_cast<T*>(s_raw) + threadIdx.x; C.st.stride = BARE_BLOCK; C.dropped = 0;
    load_state<T, NOBJ>(E, i, q, qd, ob);
    Model<T> M = E.M;
#pragma unroll
    for (int d = 0; d < ND; d++) {
        target[d] = E.target[d * n + i];
        mot[d] = E.motor[(0 * ND + d) * (size_t)n + i]; mot[9 + d] = E.motor[(1 * ND + d) * (size_t)n + i]; mot[18 + d] = E.motor[(2 * ND + d) * (size_t)n + i];
        M.max_imp[d] = E.motor[(3 * ND + d) * (size_t)n + i];
    }
    bool full_sweep = true, limits_active = false;
    for (int s = 0; s < nsub; s++) env_substep<T, NOBJ, false, true>(M, E.S, q, qd, target, ob, C, full_sweep, limits_active, mot);
    store_state<T, NOBJ>(E, i, q, qd, ob);
    E.steps[i] += 1;
}
// motors of the worlds whose mask byte is set (NULL = all): rows [9][5] = position gain, velocity gain, target angle, target
// velocity, max force (N or N m; the impulse limit per sub-step is force x dt)
template <typename T>
__global__ void __launch_bounds__(BLOCK) set_motors_kernel(const __grid_constant__ EnvDev<T> E, const double* in, const unsigned char* mask) {
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= E.n || (mask && !mask[i])) return;
    const size_t n = E.n;
    for (int d = 0; d < ND; d++) {
        const double* r = in + ((size_t)i * ND + d) * 5;
        E.motor[(0 * ND + d) * n + i] = (T)r[0]; E.motor[(1 * ND + d) * n + i] = (T)r[1]; E.target[d * n + i] = (T)r[2];
        E.motor[(2 * ND + d) * n + i] = (T)r[3]; E.motor[(3 * ND + d) * n + i] = (T)(r[4] * (double)Consts<T>::dt);
    }
}
template <typename T>
__global__ void __launch_bounds__(BLOCK) get_motors_kernel(const __grid_constant__ EnvDev<T> E, double* out) {
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= E.n) return;
    const size_t n = E.n;
    for (int d = 0; d < ND; d++) {
        double* r = out + ((size_t)i * ND + d) * 5;
        r[0] = E.motor[(0 * ND + d) * n + i]; r[1] = E.motor[(1 * ND + d) * n + i]; r[2] = E.target[d * n + i];
        r[3] = E.motor[(2 * ND + d) * n + i]; r[4] = (double)E.motor[(3 * ND + d) * n + i] / (double)Consts<T>::dt;
    }
}

// End-effector (link 11) pose from the CURRENT joint state (getLinkState with computeForwardKinematics, the fork's
// get_ee_orientation): rows [x y z qx qy qz qw] in float64.
template <typename T>
__global__ void __launch_bounds__(BLOCK) ee_pose_kernel(const __grid_constant__ EnvDev<T> E, double* out) {
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= E.n) return;
    T q[ND];
    for (int d = 0; d < ND; d++) q[d] = E.q[d * E.n + i];
    V3<T> p; T qt[4]; ee_pose(E.M, q, p, qt);
    double* r = out + (size_t)i * 7;
    r[0] = p.x; r[1] = p.y; r[2] = p.z; r[3] = qt[0]; r[4] = qt[1]; r[5] = qt[2]; r[6] = qt[3];
}

// ---------------------------------------------------------------------------------------------- HER compute_reward / is_success
// HBM-bound: M rows of two [M,G] arrays in, 4 (reward) or 1 (success) bytes out.  Each thread owns RPT consecutive rows chosen so
// that RPT*G elements are a whole number of 16-byte words: the rows are fetched with streaming 16-byte loads straight into
// registers (3 per array in flight per thread, no shared-memory round trip, no barrier), a warp covers one contiguous span.
template <typename E, int G> struct RewardTile {
    static constexpr int V = 16 / sizeof(E);                                   // elements per 16-byte word
    static constexpr int RPT = (G % V == 0) ? 1 : ((2 * G) % V == 0 ? 2 : 4);  // rows per thread
    static constexpr int NV = RPT * G / V;                                     // 16-byte words per thread and array
};
template <typename E, int TASK, bool WANT_REWARD>
__global__ void __launch_bounds__(256) reward_kernel(const E* __restrict__ ag, const E* __restrict__ dg, float* __restrict__ reward, unsigned char* __restrict__ success, long long m, int reward_type, int vec_ok, double threshold) {
    constexpr int G = task_goal_dim(TASK);
    using TL = RewardTile<E, G>;
    const E thr = (E)threshold;                  // compared in the dtype of the distance (numpy casts the Python-float threshold to it)
    const long long groups = vec_ok ? m / TL::RPT : 0;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (long long)gridDim.x * blockDim.x) {
        union { float4 v[TL::NV]; E e[TL::RPT * G]; } a, b;
        const float4* pa = reinterpret_cast<const float4*>(ag + g * TL::RPT * G);
        const float4* pb = reinterpret_cast<const float4*>(dg + g * TL::RPT * G);
#pragma unroll
        for (int k = 0; k < TL::NV; k++) { a.v[k] = __ldcs(pa + k); b.v[k] = __ldcs(pb + k); }
#pragma unroll
        for (int r = 0; r < TL::RPT; r++) {
            E d = goal_distance(TASK, a.e + r * G, b.e + r * G);
            if (WANT_REWARD) reward[g * TL::RPT + r] = reward_from_distance(reward_type, d, thr);
            else success[g * TL::RPT + r] = d < thr;
        }
    }
    // tail rows (and the whole array when the pointers are not 16-byte aligned)
    for (long long row = groups * TL::RPT + (long long)blockIdx.x * blockDim.x + threadIdx.x; row < m; row += (long long)gridDim.x * blockDim.x) {
        E a[G], b[G];
#pragma unroll
        for (int k = 0; k < G; k++) { a[k] = ag[row * G + k]; b[k] = dg[row * G + k]; }
        E d = goal_distance(TASK, a, b);
        if (WANT_REWARD) reward[row] = reward_from_distance(reward_type, d, thr);
        else success[row] = d < thr;
    }
}

// HER relabelling fused with compute_reward -- the caller on the learner side of the step (reference: examples/train_push.py:1-12
// hands the env to stable-baselines3's HerReplayBuffer, which gathers `next_achieved_goal` rows as new goals and calls
// Task.compute_reward, tasks/*.py, on the relabelled batch).  For sampled transition j: the new desired goal is the next achieved
// goal of transition goal_src[j] (a later step of the same episode under the "future" strategy), or the stored desired goal when
// goal_src[j] < 0; the reward is recomputed from the transition's own next achieved goal and the new goal, in the reference's
// float32 arithmetic.  56 / 92 algorithmic bytes per transition (3-D / 6-D goals).
//
// The kernel is a random row gather: what it moves through DRAM is 32-byte sectors, not rows.  A row of G elements at a pitch of
// `pitch` elements is fetched with the widest loads its alignment allows (VB bytes each: 16 for 32-byte padded rows, 8 for dense
// 6-D fp32 rows, 4 otherwise) -- a dense 24-byte row is 3 requests instead of 6 and straddles two sectors half the time, a row
// padded to 32 bytes (pitch 8) is exactly one sector -- and every thread keeps HT transitions in flight (2 x HT independent row
// gathers issued before the first use), because a gather is bounded by the number of sectors in flight per SM, not by bandwidth.
template <typename E, int G, int VB> struct RowLoad {
    static constexpr int EV = VB / (int)sizeof(E);            // elements per load
    static constexpr int NV = (G + EV - 1) / EV;               // loads per row (the last one may read padding: only when pitch allows it)
    __device__ static __forceinline__ void load(const E* __restrict__ p, E* out) {
        if constexpr (VB == 16) {
            union { float4 v[NV]; E e[NV * EV]; } u;
#pragma unroll
            for (int k = 0; k < NV; k++) u.v[k] = __ldg(reinterpret_cast<const float4*>(p) + k);
#pragma unroll
            for (int k = 0; k < G; k++) out[k] = u.e[k];
        } else if constexpr (VB == 8) {
            union { float2 v[NV]; E e[NV * EV]; } u;
#pragma unroll
            for (int k = 0; k < NV; k++) u.v[k] = __ldg(reinterpret_cast<const float2*>(p) + k);
#pragma unroll
            for (int k = 0; k < G; k++) out[k] = u.e[k];
        } else {
#pragma unroll
            for (int k = 0; k < G; k++) out[k] = __ldg(p + k);
        }
    }
};
constexpr int HER_INFLIGHT = 4;      // transitions in flight per thread (two row gathers each)
template <typename E, int TASK, int VB>
__global__ void __launch_bounds__(256) her_relabel_kernel(const E* __restrict__ next_ag, const E* __restrict__ dg, const long long* __restrict__ src,
                                                          const long long* __restrict__ goal_src, E* __restrict__ dg_out, E* __restrict__ ag_out,
                                                          float* __restrict__ reward, long long m, long long pitch, int reward_type, double threshold) {
    constexpr int G = task_goal_dim(TASK), HT = HER_INFLIGHT;
    using RL = RowLoad<E, G, VB>;
    const E thr = (E)threshold;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long j0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; j0 < m; j0 += HT * stride) {
        long long s[HT], gs[HT];
#pragma unroll
        for (int h = 0; h < HT; h++) { const long long j = j0 + h * stride; const bool ok = j < m; s[h] = ok ? __ldcs(src + j) : 0; gs[h] = ok ? __ldcs(goal_src + j) : 0; }
        E a[HT][G], b[HT][G];
#pragma unroll
        for (int h = 0; h < HT; h++) {
            RL::load(next_ag + s[h] * pitch, a[h]);
            RL::load(gs[h] >= 0 ? next_ag + gs[h] * pitch : dg + s[h] * pitch, b[h]);
        }
#pragma unroll
        for (int h = 0; h < HT; h++) {
            const long long j = j0 + h * stride;
            if (j >= m) break;
            E d = goal_distance(TASK, a[h], b[h]);
            __stcs(reward + j, reward_from_distance(reward_type, d, thr));
#pragma unroll
            for (int k = 0; k < G; k++) { __stcs(dg_out + j * G + k, b[h][k]); if (ag_out) __stcs(ag_out + j * G + k, a[h][k]); }
        }
    }
}

// host-side launchers, instantiated per task in panda_step_task.cu
template <typename T, int TASK> void launch_step(const EnvDev<T>& E, int ctrl, const StepIO& io, cudaStream_t st);
template <typename T, int TASK> void launch_reset(const EnvDev<T>& E, const ResetIO& io, cudaStream_t st);
template <typename T> void launch_bare_step(const EnvDev<T>& E, int nobj, int nsub, cudaStream_t st);   // panda_bare.cu

}  // namespace pg
