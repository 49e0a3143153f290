// panda_motion.cuh -- per-env math of the fork's scripted motion primitives (robots/panda_cartesian.py: move / grasp / release),
// shared by the motion kernels (panda_motion.cu) and the host build of tests/hostcheck/motion.cpp.
//
// move(goal_pos, goal_quat) from the EE pose (start, q0) read when the primitive begins:
//   d = goal_pos - start;  n = 20 if |d| < 0.03, else floor(|d| / 0.015) + (|d| mod 0.015 > 1e-3), at least 1 (numpy // and %);
//   step i = 1..n: position target start + (d / n) * min(i, n), action = target - (EE position before the step), finger action 0;
//   orientation target = scipy Slerp([1, K], [q0, q1]) at clamp(i, 1, K), K = max(n, 2).
// The position arithmetic is float64 and never contracted into an FMA, so the targets are bit-identical to numpy's.
#pragma once
#include <math.h>
#include "panda_dyn.cuh"

namespace pg {

enum { MOTION_IDLE = 0, MOTION_MOVE = 1, MOTION_GRIPPER = 2 };

// Plan state of a batch of n envs: SoA rows of n entries each (row r of env i at [r * n + i]).
enum { MP_START = 0, MP_DELTA = 3, MP_Q0 = 6, MP_ROTVEC = 10, MP_FINGER = 13, MP_ROWS = 14 };   // float64 rows
struct MotionPlan {
    int n;
    double* f;          // [MP_ROWS][n]: start xyz, delta xyz, q0 xyzw, rotvec(q0^-1 q1) xyz, finger action
    int* kind;          // [n] MOTION_*
    int* step;          // [n] primitive steps taken
    int* count;         // [n] primitive length
    float* act;         // [n, act_dim] scratch: the actions of the next env step
    float* quat;        // [n, 4] scratch: the EE target orientations (x, y, z, w) of the next env step
};

// IEEE double product and sum, never fused (nvcc contracts a * b + c into an FMA by default; numpy rounds both)
PG_HD double mul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
PG_HD double add_rn(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// numpy's a // b and a % b for float64 (npy_divmod)
PG_HD void np_divmod(double a, double b, double& div, double& mod) {
    mod = fmod(a, b);
    double d = (a - mod) / b;
    if (mod != 0.0) {
        if ((b < 0) != (mod < 0)) { mod += b; d -= 1.0; }
    } else {
        mod = copysign(0.0, b);
    }
    if (d != 0.0) {
        div = floor(d);
        if (d - div > 0.5) div += 1.0;
    } else {
        div = copysign(0.0, a / b);
    }
}

// Panda.move's way-point count for the distance |goal - start| (panda_cartesian.py:32-40,50-53); a non-finite distance gives 1
PG_HD int waypoint_count(double dist) {
    if (dist < 0.03) return 20;
    double div, mod;
    np_divmod(dist, 0.015, div, mod);
    if (mod > 1e-3) div += 1.0;
    return div >= 1e6 ? 1000000 : (div >= 1.0 ? (int)div : 1);
}

// numpy.linalg.norm of a 3-vector, unfused
PG_HD double norm3_rn(const double* d) { return sqrt(add_rn(add_rn(mul_rn(d[0], d[0]), mul_rn(d[1], d[1])), mul_rn(d[2], d[2]))); }

// Hamilton product a * b, quaternions (x, y, z, w) -- scipy's _compose_quat
PG_HD void quat_mul(const double* a, const double* b, double* out) {
    const double x = a[3] * b[0] + b[3] * a[0] + (a[1] * b[2] - a[2] * b[1]);
    const double y = a[3] * b[1] + b[3] * a[1] + (a[2] * b[0] - a[0] * b[2]);
    const double z = a[3] * b[2] + b[3] * a[2] + (a[0] * b[1] - a[1] * b[0]);
    const double w = a[3] * b[3] - (a[0] * b[0] + a[1] * b[1] + a[2] * b[2]);
    out[0] = x; out[1] = y; out[2] = z; out[3] = w;
}

PG_HD void quat_normalise(const double* q, double* out) {
    const double s = 1.0 / sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
    for (int k = 0; k < 4; k++) out[k] = q[k] * s;
}

// Rotation.as_rotvec: the shortest arc (w >= 0), angle 2 atan2(|v|, w), scipy's series below 1e-3 rad
PG_HD void quat_to_rotvec(const double* q, double* rv) {
    const double sg = q[3] < 0 ? -1.0 : 1.0;
    const double x = sg * q[0], y = sg * q[1], z = sg * q[2], w = sg * q[3];
    const double angle = 2.0 * atan2(sqrt(x * x + y * y + z * z), w);
    const double a2 = angle * angle;
    const double scale = angle <= 1e-3 ? 2.0 + a2 / 12.0 + 7.0 * a2 * a2 / 2880.0 : angle / sin(angle / 2.0);
    rv[0] = scale * x; rv[1] = scale * y; rv[2] = scale * z;
}

// Rotation.from_rotvec
PG_HD void rotvec_to_quat(const double* rv, double* q) {
    const double angle = sqrt(rv[0] * rv[0] + rv[1] * rv[1] + rv[2] * rv[2]);
    const double a2 = angle * angle;
    const double scale = angle <= 1e-3 ? 0.5 - a2 / 48.0 + a2 * a2 / 3840.0 : sin(angle / 2.0) / angle;
    q[0] = scale * rv[0]; q[1] = scale * rv[1]; q[2] = scale * rv[2]; q[3] = cos(angle / 2.0);
}

// Begin a move: way-point count, per-step displacement, unit start orientation and the Slerp's rotation vector rotvec(q0^-1 q1).
// start / q0 are the EE pose at begin time, goal / goal_quat the primitive's arguments.
PG_HD int move_plan(const double* start, const double* q0, const double* goal, const double* goal_quat, double* delta, double* q0_unit, double* rotvec) {
    double d[3];
    for (int k = 0; k < 3; k++) d[k] = goal[k] - start[k];
    const int n = waypoint_count(norm3_rn(d));
    for (int k = 0; k < 3; k++) delta[k] = d[k] / (double)n;
    double q1[4], inv[4], rel[4];
    quat_normalise(q0, q0_unit);
    quat_normalise(goal_quat, q1);
    inv[0] = -q0_unit[0]; inv[1] = -q0_unit[1]; inv[2] = -q0_unit[2]; inv[3] = q0_unit[3];
    quat_mul(inv, q1, rel);
    quat_to_rotvec(rel, rotvec);
    return n;
}

// Position target of move step i (1-based) of n: start + delta * min(i, n), rounded as numpy rounds it
PG_HD double waypoint(double start, double delta, int n, int i) { return add_rn(start, mul_rn(delta, (double)(i < n ? i : n))); }

// Orientation target of move step i of n: Slerp([1, K], [q0, q1])(clamp(i, 1, K)) = q0 * exp(t rotvec), t = (clamp(i, 1, K) - 1) / (K - 1)
PG_HD void slerp_at(const double* q0, const double* rotvec, int n, int i, double* out) {
    const int K = n > 2 ? n : 2;
    const int c = i < 1 ? 1 : (i > K ? K : i);
    const double t = (double)(c - 1) / (double)(K - 1);
    const double rv[3] = {rotvec[0] * t, rotvec[1] * t, rotvec[2] * t};
    double e[4];
    rotvec_to_quat(rv, e);
    quat_mul(q0, e, out);
}

}  // namespace pg
