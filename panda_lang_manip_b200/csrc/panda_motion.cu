// panda_motion.cu -- the fork's scripted motion primitives (robots/panda_cartesian.py:47-68: move / grasp / release) for every env:
// one thread per env begins a primitive (move: fresh forward kinematics, then the plan rows) or turns the plan into the actions and
// EE target orientations of the next env step.  The math is panda_motion.cuh; pg_motion_step in panda_b200.cu runs the step kernel
// on the scratch rows written here.
#include <cuda_runtime.h>
#include "panda_kernels.cuh"
#include "panda_motion.cuh"

namespace pg {

extern long long g_launches;

template <typename T>
__device__ __forceinline__ void fresh_ee(const EnvDev<T>& E, int i, double* pos, double* quat) {
    T q[ND];
    for (int d = 0; d < ND; d++) q[d] = E.q[d * E.n + i];
    V3<T> p; T qt[4];
    ee_pose(E.M, q, p, qt);
    pos[0] = p.x; pos[1] = p.y; pos[2] = p.z;
    for (int k = 0; k < 4; k++) quat[k] = qt[k];
}

// move of the envs whose mask byte is set (NULL = all): goal [n,3], goal_quat [n,4] (x,y,z,w) float64
template <typename T>
__global__ void __launch_bounds__(BLOCK) motion_move_kernel(const __grid_constant__ EnvDev<T> E, const MotionPlan P, const double* goal, const double* goal_quat,
                                                             const unsigned char* mask) {
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= P.n || (mask && !mask[i])) return;
    const int n = P.n;
    double start[3], q0[4], delta[3], q0u[4], rv[3];
    fresh_ee(E, i, start, q0);
    const int cnt = move_plan(start, q0, goal + (size_t)i * 3, goal_quat + (size_t)i * 4, delta, q0u, rv);
    for (int k = 0; k < 3; k++) { P.f[(MP_START + k) * n + i] = start[k]; P.f[(MP_DELTA + k) * n + i] = delta[k]; P.f[(MP_ROTVEC + k) * n + i] = rv[k]; }
    for (int k = 0; k < 4; k++) P.f[(MP_Q0 + k) * n + i] = q0u[k];
    P.kind[i] = MOTION_MOVE; P.step[i] = 0; P.count[i] = cnt;
}

// grasp / release: `steps` steps with the finger action `finger`
__global__ void __launch_bounds__(BLOCK) motion_gripper_kernel(const MotionPlan P, double finger, int steps, const unsigned char* mask) {
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= P.n || (mask && !mask[i])) return;
    P.f[MP_FINGER * P.n + i] = finger;
    P.kind[i] = steps > 0 ? MOTION_GRIPPER : MOTION_IDLE; P.step[i] = 0; P.count[i] = steps;
}

// The actions [n, A] and target orientations [n, 4] of the next env step from the current joint state, then every active env's
// counter advances; remaining[i] = steps of the env's primitive still to take after this one (0: idle from the next step on).
template <typename T>
__global__ void __launch_bounds__(BLOCK) motion_step_kernel(const __grid_constant__ EnvDev<T> E, const MotionPlan P, int A, int* remaining) {
    const int i = blockIdx.x * BLOCK + threadIdx.x;
    if (i >= P.n) return;
    const int n = P.n;
    double ee[3], quat[4];
    fresh_ee(E, i, ee, quat);             // grasp, release and idle steps hold the current orientation
    float* a = P.act + (size_t)i * A;
    for (int k = 0; k < A; k++) a[k] = 0.0f;
    const int kind = P.kind[i], cnt = P.count[i], s = P.step[i] + 1;
    if (kind == MOTION_MOVE) {
        for (int k = 0; k < 3; k++) a[k] = (float)(waypoint(P.f[(MP_START + k) * n + i], P.f[(MP_DELTA + k) * n + i], cnt, s) - ee[k]);
        double q0[4], rv[3];
        for (int k = 0; k < 4; k++) q0[k] = P.f[(MP_Q0 + k) * n + i];
        for (int k = 0; k < 3; k++) rv[k] = P.f[(MP_ROTVEC + k) * n + i];
        slerp_at(q0, rv, cnt, s, quat);
    } else if (kind == MOTION_GRIPPER) {
        a[A - 1] = (float)P.f[MP_FINGER * n + i];
    }
    for (int k = 0; k < 4; k++) P.quat[(size_t)i * 4 + k] = (float)quat[k];
    if (kind != MOTION_IDLE) {
        P.step[i] = s;
        if (s >= cnt) P.kind[i] = MOTION_IDLE;
    }
    if (remaining) remaining[i] = kind == MOTION_IDLE ? 0 : cnt - s;
}

template <typename T> void launch_motion_move(const EnvDev<T>& E, const MotionPlan& P, const double* goal, const double* goal_quat, const unsigned char* mask, cudaStream_t st) {
    motion_move_kernel<T><<<(P.n + BLOCK - 1) / BLOCK, BLOCK, 0, st>>>(E, P, goal, goal_quat, mask);
    g_launches++;
}
void launch_motion_gripper(const MotionPlan& P, double finger, int steps, const unsigned char* mask, cudaStream_t st) {
    motion_gripper_kernel<<<(P.n + BLOCK - 1) / BLOCK, BLOCK, 0, st>>>(P, finger, steps, mask);
    g_launches++;
}
template <typename T> void launch_motion_step(const EnvDev<T>& E, const MotionPlan& P, int act_dim, int* remaining, cudaStream_t st) {
    motion_step_kernel<T><<<(P.n + BLOCK - 1) / BLOCK, BLOCK, 0, st>>>(E, P, act_dim, remaining);
    g_launches++;
}
template void launch_motion_move<float>(const EnvDev<float>&, const MotionPlan&, const double*, const double*, const unsigned char*, cudaStream_t);
template void launch_motion_move<double>(const EnvDev<double>&, const MotionPlan&, const double*, const double*, const unsigned char*, cudaStream_t);
template void launch_motion_step<float>(const EnvDev<float>&, const MotionPlan&, int, int*, cudaStream_t);
template void launch_motion_step<double>(const EnvDev<double>&, const MotionPlan&, int, int*, cudaStream_t);

}  // namespace pg
