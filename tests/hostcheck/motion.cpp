// motion.cpp -- TEST-ONLY host compilation of the motion primitives' per-env math (panda_lang_manip_b200/csrc/panda_motion.cuh), so
// that the CPU test-suite can compare it with the facade's own static helpers Panda.get_waypoint / Panda.get_ori without a GPU
// (tests/test_hostcheck_motion.py builds it with -ffp-contract=off).  Nothing in the package loads it.
#include "../../panda_lang_manip_b200/csrc/panda_motion.cuh"
using namespace pg;

extern "C" {
// way-point count of a move from start to goal (3-vectors)
int hc_waypoint_count(const double* start, const double* goal) {
    double d[3] = {goal[0] - start[0], goal[1] - start[1], goal[2] - start[2]};
    return waypoint_count(norm3_rn(d));
}
// the n way-point positions of a move, out [n, 3] (n = hc_waypoint_count)
void hc_waypoints(const double* start, const double* goal, double* out) {
    const double q[4] = {0, 0, 0, 1};
    double delta[3], q0[4], rv[3];
    const int n = move_plan(start, q, goal, q, delta, q0, rv);
    for (int i = 1; i <= n; i++)
        for (int k = 0; k < 3; k++) out[(i - 1) * 3 + k] = waypoint(start[k], delta[k], n, i);
}
// the move's orientation target at step i of n from q0 to q1 (x, y, z, w)
void hc_slerp(const double* q0, const double* q1, int n, int i, double* out) {
    const double p[3] = {0, 0, 0};
    double delta[3], q0u[4], rv[3];
    move_plan(p, q0, p, q1, delta, q0u, rv);
    slerp_at(q0u, rv, n, i, out);
}
}
