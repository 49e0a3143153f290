// contact_report.cpp -- TEST-ONLY host compilation of the step kernel's contact-report decode (contact_report_row in
// panda_lang_manip_b200/csrc/panda_contact.cuh) after a whole env step of the kernel math, so that the CPU test-suite can compare the
// report with the oracle's without a GPU (tests/test_hostcheck_contact_report.py builds it).  Nothing in the package loads it.
#include "../../panda_lang_manip_b200/csrc/panda_model.h"
#include "../../panda_lang_manip_b200/csrc/panda_scene.h"
using namespace pg;

// state layout (doubles): q[9], qd[9], obj[2][13] = pos3 quat4 lin3 ang3, goal[6]; rows [max_contacts][REPORT_WORDS] in double
template <typename T, int TASK, int CTRL> static void step_report(const double* base, double* st, const float* action, double* rows, int* count) {
    Model<T> M = make_model<T>(base); Scene<T> S = make_scene<T>(TASK);
    constexpr int NOBJ = task_nobj(TASK);
    T q[ND], qd[ND], target[ND]; double goal[6]; Obj<T> ob[NOBJ > 0 ? NOBJ : 1];
    for (int i = 0; i < ND; i++) { q[i] = (T)st[i]; qd[i] = (T)st[9 + i]; }
    for (int o = 0; o < NOBJ; o++) { const double* p = st + 18 + 13 * o; ob[o].pos = mk<T>((T)p[0], (T)p[1], (T)p[2]); ob[o].qx = (T)p[3]; ob[o].qy = (T)p[4]; ob[o].qz = (T)p[5]; ob[o].qw = (T)p[6]; ob[o].lin = mk<T>((T)p[7], (T)p[8], (T)p[9]); ob[o].ang = mk<T>((T)p[10], (T)p[11], (T)p[12]); }
    for (int k = 0; k < 6; k++) goal[k] = st[44 + k];
    static T slab[solver_slots(2)];
    Contacts<T> C; C.st.base = slab; C.st.stride = 1; C.dropped = 0;
    float obs[40], ag[6], dg[6], rew; unsigned char succ; int key = 0;
    env_step<T, TASK, CTRL>(M, S, REWARD_SPARSE, q, qd, ob, goal, action, nullptr, obs, ag, dg, rew, succ, C, key, target);
    for (int c = 0; c < C.n; c++) contact_report_row(S, C, c, rows + c * REPORT_WORDS);
    *count = C.n;
    for (int i = 0; i < ND; i++) { st[i] = q[i]; st[9 + i] = qd[i]; }
    for (int o = 0; o < NOBJ; o++) { double* p = st + 18 + 13 * o; p[0] = ob[o].pos.x; p[1] = ob[o].pos.y; p[2] = ob[o].pos.z; p[3] = ob[o].qx; p[4] = ob[o].qy; p[5] = ob[o].qz; p[6] = ob[o].qw; p[7] = ob[o].lin.x; p[8] = ob[o].lin.y; p[9] = ob[o].lin.z; p[10] = ob[o].ang.x; p[11] = ob[o].ang.y; p[12] = ob[o].ang.z; }
}
template <typename T, int TASK> static void step_report_c(int ctrl, const double* base, double* st, const float* action, double* rows, int* count) {
    if (ctrl == CTRL_EE) step_report<T, TASK, CTRL_EE>(base, st, action, rows, count); else step_report<T, TASK, CTRL_JOINTS>(base, st, action, rows, count);
}
template <typename T> static void step_report_d(int task, int ctrl, const double* base, double* st, const float* action, double* rows, int* count) {
    switch (task) {
    case 0: step_report_c<T, 0>(ctrl, base, st, action, rows, count); break;
    case 1: step_report_c<T, 1>(ctrl, base, st, action, rows, count); break;
    case 2: step_report_c<T, 2>(ctrl, base, st, action, rows, count); break;
    case 3: step_report_c<T, 3>(ctrl, base, st, action, rows, count); break;
    case 4: step_report_c<T, 4>(ctrl, base, st, action, rows, count); break;
    default: step_report_c<T, 5>(ctrl, base, st, action, rows, count); break;
    }
}
extern "C" {
// one env step of the kernel math from state st (updated in place), then the report of its last sub-step: *count rows
void hc_env_step_contacts(int dbl, int task, int ctrl, const double* base, double* st, const float* action, double* rows, int* count) {
    if (dbl) step_report_d<double>(task, ctrl, base, st, action, rows, count); else step_report_d<float>(task, ctrl, base, st, action, rows, count);
}
}
