// panda_env.cuh -- one environment step: action -> motor targets -> 20 sub-steps -> observation / goals / reward / success.
//
// Mirrors reference panda_gym/envs/core.py:280-289 (RobotTaskEnv.step), :229-238 (_get_obs),
// panda_gym/envs/robots/panda.py:52-119 (set_action, get_obs), the per-task get_obs / get_achieved_goal /
// is_success / compute_reward of panda_gym/envs/tasks/<task>.py and panda_gym/utils.py:4-30.
#pragma once
#include <string.h>
#include "panda_contact.cuh"

namespace pg {

enum { TASK_REACH = 0, TASK_PUSH = 1, TASK_SLIDE = 2, TASK_PICK_AND_PLACE = 3, TASK_STACK = 4, TASK_FLIP = 5 };
enum { CTRL_EE = 0, CTRL_JOINTS = 1 };
enum { REWARD_SPARSE = 0, REWARD_DENSE = 1 };

PG_HD constexpr int task_nobj(int task) { return task == TASK_REACH ? 0 : (task == TASK_STACK ? 2 : 1); }
PG_HD constexpr bool task_block_gripper(int task) { return task == TASK_REACH || task == TASK_PUSH || task == TASK_SLIDE; }   // panda_tasks.py:60,77,94
PG_HD constexpr int task_goal_dim(int task) { return task == TASK_STACK ? 6 : (task == TASK_FLIP ? 4 : 3); }
PG_HD constexpr int task_obs_dim(int task) { return (task_block_gripper(task) ? 6 : 7) + (task == TASK_REACH ? 0 : (task == TASK_STACK ? 24 : (task == TASK_FLIP ? 13 : 12))); }
PG_HD constexpr int task_act_dim(int task, int ctrl) { return (ctrl == CTRL_EE ? 3 : 7) + (task_block_gripper(task) ? 0 : 1); }
PG_HD constexpr int task_max_steps(int task) { return task == TASK_STACK ? 100 : 50; }   // panda_gym/__init__.py:18,46

// What the reference's task constructors take as keyword arguments (tasks/reach.py:15-23 distance_threshold, goal_range; push.py:12-25,
// slide.py:12-27, pick_and_place.py:13-29, stack.py:11-25, flip.py:13-24: goal_xy_range, goal_z_range, goal_x_offset, obj_xy_range) and
// PyBullet(n_substeps) (pybullet.py:26), as kernel parameters.  Ranges are the noise boxes added to the task's base goal / object height.
struct TaskParams {
    double goal_lo[3], goal_hi[3];  // goal noise box
    double obj_lo[2], obj_hi[2];    // object xy noise box
    double thr64; float thr32;      // distance_threshold (compared in the dtype of the distance, as numpy does)
    int nsub;                       // stepSimulation calls per env step
};
inline TaskParams make_task_params(int task) {
    TaskParams P;
    const double z_hi = task == 0 ? 0.3 : (task == 3 ? 0.2 : 0.0), x_off = task == 2 ? 0.4 : 0.0;
    P.goal_lo[0] = -0.15 + x_off; P.goal_hi[0] = 0.15 + x_off; P.goal_lo[1] = -0.15; P.goal_hi[1] = 0.15; P.goal_lo[2] = 0.0; P.goal_hi[2] = z_hi;
    P.obj_lo[0] = P.obj_lo[1] = -0.15; P.obj_hi[0] = P.obj_hi[1] = 0.15;
    P.thr64 = task == 4 ? 0.1 : (task == 5 ? 0.2 : 0.05); P.thr32 = (float)P.thr64; P.nsub = 20;
    return P;
}

// float32 arithmetic exactly as numpy evaluates it: no fused multiply-add (SURVEY App. A.4)
#ifdef __CUDA_ARCH__
PG_HD float f_sub(float a, float b) { return __fsub_rn(a, b); }
PG_HD float f_add(float a, float b) { return __fadd_rn(a, b); }
PG_HD float f_mul(float a, float b) { return __fmul_rn(a, b); }
PG_HD float f_sqrt(float a) { return __fsqrt_rn(a); }
PG_HD double d_sub(double a, double b) { return __dsub_rn(a, b); }
PG_HD double d_add(double a, double b) { return __dadd_rn(a, b); }
PG_HD double d_mul(double a, double b) { return __dmul_rn(a, b); }
PG_HD double d_sqrt(double a) { return __dsqrt_rn(a); }
#else
PG_HD float f_sub(float a, float b) { return a - b; }
PG_HD float f_add(float a, float b) { return a + b; }
PG_HD float f_mul(float a, float b) { return a * b; }
PG_HD float f_sqrt(float a) { return sqrtf(a); }
PG_HD double d_sub(double a, double b) { return a - b; }
PG_HD double d_add(double a, double b) { return a + b; }
PG_HD double d_mul(double a, double b) { return a * b; }
PG_HD double d_sqrt(double a) { return sqrt(a); }
#endif
PG_HD float threshold_f32(int task) { return task == TASK_STACK ? 0.1f : (task == TASK_FLIP ? 0.2f : 0.05f); }
PG_HD double threshold_f64(int task) { return task == TASK_STACK ? 0.1 : (task == TASK_FLIP ? 0.2 : 0.05); }
// utils.distance (np.linalg.norm(a-b, axis=-1): squares summed left to right) / utils.angle_distance row-wise (1 - <a,b>^2)
PG_HD float goal_distance(int task, const float* a, const float* b) {
    if (task == TASK_FLIP) {
        float s = f_add(f_add(f_mul(a[0], b[0]), f_mul(a[1], b[1])), f_add(f_mul(a[2], b[2]), f_mul(a[3], b[3])));
        return f_sub(1.0f, f_mul(s, s));
    }
    const int g = task_goal_dim(task);
    float d0 = f_sub(a[0], b[0]), acc = f_mul(d0, d0);
    for (int k = 1; k < g; k++) { float d = f_sub(a[k], b[k]); acc = f_add(acc, f_mul(d, d)); }
    return f_sqrt(acc);
}
PG_HD double goal_distance(int task, const double* a, const double* b) {
    if (task == TASK_FLIP) {
        double s = d_add(d_add(d_mul(a[0], b[0]), d_mul(a[1], b[1])), d_add(d_mul(a[2], b[2]), d_mul(a[3], b[3])));
        return d_sub(1.0, d_mul(s, s));
    }
    const int g = task_goal_dim(task);
    double d0 = d_sub(a[0], b[0]), acc = d_mul(d0, d0);
    for (int k = 1; k < g; k++) { double d = d_sub(a[k], b[k]); acc = d_add(acc, d_mul(d, d)); }
    return d_sqrt(acc);
}
// sparse: -(d > thr).astype(float32) -> -1.0 or -0.0;  dense: -d.astype(float32)
// ptxas 12.9 miscompiles `selp.f32 -1.0, -0.0` into an int->float conversion that yields +0.0, so the sign bit is OR-ed in
// through an opaque instruction after the {1.0, 0.0} select.
PG_HD float sparse_reward(bool beyond) {
#ifdef __CUDA_ARCH__
    unsigned mag = __float_as_uint(beyond ? 1.0f : 0.0f), bits;
    asm volatile("or.b32 %0, %1, 0x80000000;" : "=r"(bits) : "r"(mag));
    return __uint_as_float(bits);
#else
    const unsigned bits = beyond ? 0xBF800000u : 0x80000000u;
    float f; memcpy(&f, &bits, sizeof f); return f;
#endif
}
PG_HD float reward_from_distance(int reward_type, float d, float thr) { return reward_type == REWARD_SPARSE ? sparse_reward(d > thr) : -d; }
PG_HD float reward_from_distance(int reward_type, double d, double thr) { return reward_type == REWARD_SPARSE ? sparse_reward(d > thr) : -(float)d; }

// pybullet getEulerFromQuaternion (SURVEY App. B.4)
template <typename T> PG_HD void euler_from_quat(T x, T y, T z, T w, T* e) {
    T sarg = T(-2) * (x * z - w * y);
    const T hp = Consts<T>::pi / 2;
    if (sarg <= T(-0.99999)) { e[0] = T(0); e[1] = -hp; e[2] = 2 * atan2(x, -y); }
    else if (sarg >= T(0.99999)) { e[0] = T(0); e[1] = hp; e[2] = 2 * atan2(-x, y); }
    else {
        e[0] = atan2(2 * (y * z + w * x), w * w - x * x - y * y + z * z);
        e[1] = asin(sarg);
        e[2] = atan2(2 * (x * y + w * z), w * w + x * x - y * y - z * z);
    }
}

// _get_obs: robot obs (ee pos, ee vel[, finger width]) ++ task obs; achieved goal; desired goal
template <typename T, int TASK>
PG_HD void env_observe(const Model<T>& M, const T* q, const T* qd, const T* qc, const Obj<T>* ob, const double* goal, float* obs, float* ag, float* dg) {
    constexpr int NOBJ = task_nobj(TASK);
    V3<T> p, v; ee_observe(M, q, qd, qc, p, v);
    int n = 0;
    obs[n++] = (float)p.x; obs[n++] = (float)p.y; obs[n++] = (float)p.z;
    obs[n++] = (float)v.x; obs[n++] = (float)v.y; obs[n++] = (float)v.z;
    if (!task_block_gripper(TASK)) obs[n++] = (float)(q[7] + q[8]);
#pragma unroll
    for (int o = 0; o < NOBJ; o++) {
        obs[n++] = (float)ob[o].pos.x; obs[n++] = (float)ob[o].pos.y; obs[n++] = (float)ob[o].pos.z;
        if (TASK == TASK_FLIP) { obs[n++] = (float)ob[o].qx; obs[n++] = (float)ob[o].qy; obs[n++] = (float)ob[o].qz; obs[n++] = (float)ob[o].qw; }
        else { T e[3]; euler_from_quat(ob[o].qx, ob[o].qy, ob[o].qz, ob[o].qw, e); obs[n++] = (float)e[0]; obs[n++] = (float)e[1]; obs[n++] = (float)e[2]; }
        obs[n++] = (float)ob[o].lin.x; obs[n++] = (float)ob[o].lin.y; obs[n++] = (float)ob[o].lin.z;
        obs[n++] = (float)ob[o].ang.x; obs[n++] = (float)ob[o].ang.y; obs[n++] = (float)ob[o].ang.z;
    }
    if (TASK == TASK_REACH) { ag[0] = (float)p.x; ag[1] = (float)p.y; ag[2] = (float)p.z; }
    else if (TASK == TASK_FLIP) { ag[0] = (float)ob[0].qx; ag[1] = (float)ob[0].qy; ag[2] = (float)ob[0].qz; ag[3] = (float)ob[0].qw; }
    else {
#pragma unroll
        for (int o = 0; o < NOBJ; o++) { ag[3 * o] = (float)ob[o].pos.x; ag[3 * o + 1] = (float)ob[o].pos.y; ag[3 * o + 2] = (float)ob[o].pos.z; }
    }
#pragma unroll
    for (int k = 0; k < task_goal_dim(TASK); k++) dg[k] = (float)goal[k];
}

// Panda.set_action: clip, arm target from the ee displacement (IK) or the joint deltas, finger target
template <typename T, int TASK, int CTRL>
PG_HD void env_set_action(const Model<T>& M, const T* q, const T* qd, const float* action, const float* target_quat, T* target) {
    constexpr int NA = task_act_dim(TASK, CTRL);
    T a[NA];
#pragma unroll
    for (int k = 0; k < NA; k++) { T v = (T)action[k]; a[k] = v < T(-1) ? T(-1) : (v > T(1) ? T(1) : v); }
    if (CTRL == CTRL_EE) {
        // the EE position the reference reads is the cached one, FK(q - qd dt) (SURVEY App. B.5)
        T qc[ND];
#pragma unroll
        for (int d = 0; d < ND; d++) qc[d] = q[d] - qd[d] * Consts<T>::dt;
        Frame<T> F[7]; fk_arm(M, qc, F);
        V3<T> p = F[6].p + F[6].Z * M.eez;
        p.x += a[0] * M.ee_scale; p.y += a[1] * M.ee_scale; p.z += a[2] * M.ee_scale;
        if (p.z < T(0)) p.z = T(0);
        // target orientation: (1,0,0,0) as panda.py:89, or the caller's quaternion (the fork's panda_ori.py:72-99 euler_xyz target)
        T tq[4] = {T(1), T(0), T(0), T(0)};
        if (target_quat) {
            T n = T(0);
#pragma unroll
            for (int k = 0; k < 4; k++) { tq[k] = (T)target_quat[k]; n += tq[k] * tq[k]; }
            n = T(1) / sqrt(n);
#pragma unroll
            for (int k = 0; k < 4; k++) tq[k] *= n;
        }
        ik_ee(M, q, p, tq, target);
    } else {
#pragma unroll
        for (int d = 0; d < 7; d++) target[d] = q[d] + a[d] * M.ee_scale;
    }
    T w = task_block_gripper(TASK) ? T(0) : (q[7] + q[8]) + a[NA - 1] * M.finger_scale;
    target[7] = w / 2; target[8] = w / 2;
}

// Scheduling key (16 bits) written by every launch for the sort that precedes the next one: bits 0-4 contacts of the last sub-step,
// then: a robot box is in contact, the last solve ran all 50 sweeps, near a contact (or in contact earlier in the launch), an arm
// joint limit was engaged (the next launch starts with the full limit sweep); bits 10-13: generic contacts of the last sub-step
// (two-object scenes only: measured +6 % on Stack, -5 % on the one-object scenes, whose batches fragment over the extra buckets).
enum { KEY_ROBOT = 0x20, KEY_CAPPED = 0x40, KEY_NEAR = 0x80, KEY_FULL = 0x200 };

// RobotTaskEnv.step (core.py:280-289) evaluates is_success / compute_reward on (float32 achieved goal, FLOAT64 task goal): numpy promotes
// the difference to float64, so the in-step distance, its comparison with the threshold and the dense reward's cast -d.astype(float32)
// are float64 arithmetic on the float32-rounded achieved goal -- unlike compute_reward on two float32 arrays (the HER path, reward_kernel).
// The goal is therefore stored in float64 whatever the simulation precision.
template <int TASK>
PG_HD void step_reward(int reward_type, const float* ag, const double* goal, double thr, float& reward, unsigned char& success) {
    double a[task_goal_dim(TASK)];
#pragma unroll
    for (int k = 0; k < task_goal_dim(TASK); k++) a[k] = (double)ag[k];
    const double d = goal_distance(TASK, a, goal);
    success = d < thr;
    reward = reward_from_distance(reward_type, d, thr);
}

// The simulation part of RobotTaskEnv.step for one environment, or the sub-step range [s0, s1) of it (a step may be cut into segments so
// that the envs can be re-sorted in between; the motor targets travel through `target`).  q/qd/ob are updated in place; qc receives the
// link-transform cache of the last sub-step (valid when s1 == nsub).
template <typename T, int TASK, int CTRL>
PG_HD void env_step_sim(const Model<T>& M, const Scene<T>& S, T* q, T* qd, Obj<T>* ob, const float* action, const float* target_quat, Contacts<T>& C, int& sched_key,
                        T* target, T* qc, int s0 = 0, int s1 = 20, int nsub = 20) {
    constexpr int NOBJ = task_nobj(TASK);
    if (s0 == 0) env_set_action<T, TASK, CTRL>(M, q, qd, action, target_quat, target);
    // sticky: once an arm limit engaged, later sub-steps (and, through the key's KEY_FULL bit, the next segment / step) start with the
    // full sweep; it is dropped again after a segment in which no arm limit row carried impulse
    bool full_sweep = (sched_key & KEY_FULL) != 0, limits_active = false;
    int nsub_contact = 0; bool near = false;
    {
        for (int s = s0; s < s1; s++) {
            if (s == nsub - 1) {
#pragma unroll
                for (int d = 0; d < ND; d++) qc[d] = q[d];   // the link-transform cache is refreshed at the start of each sub-step
            }
            // watched arm-limit rows: a measured policy -- +25 % with joint control, -37..55 % with ee control (contact rows dominate there), so
            // it is enabled for joint control only.  Round 2 re-measured the alternatives (full sweep out of line, watched sweep for ee
            // control, a rolled local-memory fallback inside the one loop: 3-10x slower): profiles/r2_solver_structure_ab.
            env_substep<T, NOBJ, CTRL == CTRL_JOINTS>(M, S, q, qd, target, ob, C, full_sweep, limits_active);
            if (C.n > 0) nsub_contact++;
            near = near || C.near;
        }
        // scheduling key for the next launch (see perm_bucket): the contact picture of this launch's last sub-step
        const int ngen = C.n - C.nB - C.nA;                     // generic contacts (robot box <-> object, object <-> object): the most expensive rows
        sched_key = (C.n < 31 ? C.n : 31) | (NOBJ == 2 ? (ngen < 15 ? ngen : 15) << 10 : 0) | (C.nr > 0 ? KEY_ROBOT : 0) | ((near || nsub_contact > 0) ? KEY_NEAR : 0) | (C.capped ? KEY_CAPPED : 0) | (limits_active ? KEY_FULL : 0);
    }
}
// _get_obs + is_success + compute_reward of the step that just ended (core.py:283-288)
template <typename T, int TASK>
PG_HD void env_step_finish(const Model<T>& M, int reward_type, const T* q, const T* qd, const T* qc, const Obj<T>* ob, const double* goal, double thr,
                           float* obs, float* ag, float* dg, float& reward, unsigned char& success) {
    env_observe<T, TASK>(M, q, qd, qc, ob, goal, obs, ag, dg);
    step_reward<TASK>(reward_type, ag, goal, thr, reward, success);
}
// the whole step (host test build and small callers)
template <typename T, int TASK, int CTRL>
PG_HD void env_step(const Model<T>& M, const Scene<T>& S, int reward_type, T* q, T* qd, Obj<T>* ob, const double* goal, const float* action, const float* target_quat,
                    float* obs, float* ag, float* dg, float& reward, unsigned char& success, Contacts<T>& C, int& sched_key, T* target, int nsub = 20, double thr = -1.0) {
    T qc[ND];
    env_step_sim<T, TASK, CTRL>(M, S, q, qd, ob, action, target_quat, C, sched_key, target, qc, 0, nsub, nsub);
    env_step_finish<T, TASK>(M, reward_type, q, qd, qc, ob, goal, thr < 0.0 ? threshold_f64(TASK) : thr, obs, ag, dg, reward, success);
}

}  // namespace pg
