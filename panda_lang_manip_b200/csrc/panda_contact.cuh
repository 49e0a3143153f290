// panda_contact.cuh -- free rigid bodies, contact generation and the full constrained sub-step, one thread per env.
//
// Replaces what the reference obtains from pybullet's stepSimulation for the task scenes
// (reference panda_gym/pybullet.py:52-55; scenes: panda_gym/envs/tasks/{reach,push,slide,pick_and_place,stack,flip}.py
// _create_scene; friction: panda_gym/envs/robots/panda.py:47-50, slide.py:34-42).
//
// Contact model (defined by oracle/panda_oracle.c, "contact model"): vertices of one body against the signed-distance
// field of the other (table plane, box, z-cylinder; box <-> box object pairs: vertices against the other box's reference face plus
// edge against edge), speculative rows inside a 4 mm margin, two friction directions with an implicit cone, soft finger contacts,
// sequential impulses interleaved with the joint-limit and motor rows.
// Contact records (geometry + 3 x (1/D, rhs, impulse)) and the operational-space Jacobian live in shared memory, word-interleaved
// by thread; the robot part of a row is a wrench in the gripper's 8-dimensional operational space, the free-body part is
// recomputed from the contact geometry each sweep (see "contact storage" below).
#pragma once
#include "panda_dyn.cuh"

namespace pg {

constexpr int MAXOBJ = 2;

enum { SH_BOX = 0, SH_CYL = 1 };
template <typename T> struct Scene {
    int nobj;
    int shape[MAXOBJ];
    T half[MAXOBJ][3];          // box half extents, or (r, r, h/2)
    T mass[MAXOBJ], Ic[MAXOBJ][3], mu[MAXOBJ];
    T table_x0, table_x1, table_y0, table_y1;
    T rb_c[3][3], rb_h[3][3], rb_mu[3];   // robot collision boxes: hand (link 8), finger 1, finger 2 -- centre / half extents in the link frame
    T margin, margin_grasp, ground_z, table_mu;   // speculative margins: 4 mm; robot box <-> object 12 mm when the closest feature is a face (fingers close at up to 5 m/s)
    T soft_erp, soft_cfm;       // finger contact stiffness 30000 / damping 1000 -> erp, cfm/dt
};

template <typename T> struct Obj { V3<T> pos; T qx, qy, qz, qw; V3<T> lin, ang; };
template <typename T> struct Rot { V3<T> X, Y, Z; };   // columns
template <typename T> PG_HD Rot<T> quat_rot(T x, T y, T z, T w) {
    Rot<T> R;
    R.X = mk<T>(1 - 2 * (y * y + z * z), 2 * (x * y + w * z), 2 * (x * z - w * y));
    R.Y = mk<T>(2 * (x * y - w * z), 1 - 2 * (x * x + z * z), 2 * (y * z + w * x));
    R.Z = mk<T>(2 * (x * z + w * y), 2 * (y * z - w * x), 1 - 2 * (x * x + y * y));
    return R;
}
template <typename T> PG_HD V3<T> rot_mul(const Rot<T>& R, V3<T> u) { return R.X * u.x + R.Y * u.y + R.Z * u.z; }
template <typename T> PG_HD V3<T> rot_tmul(const Rot<T>& R, V3<T> u) { return mk<T>(dot(R.X, u), dot(R.Y, u), dot(R.Z, u)); }

// 0-link floating base of a btMultiBody: gravity, per-body damping, gyroscopic term; semi-implicit Euler on the velocity
template <typename T> PG_HD void obj_unconstrained(const Scene<T>& S, int o, Obj<T>& b, const Rot<T>& R) {
    const T k = Consts<T>::kdamp, dt = Consts<T>::dt;
    T kl = k + k * norm(b.lin), ka = k + k * norm(b.ang);
    V3<T> wl = rot_tmul(R, b.ang);
    V3<T> Iw = mk<T>(S.Ic[o][0] * wl.x, S.Ic[o][1] * wl.y, S.Ic[o][2] * wl.z);
    V3<T> g = cross(wl, Iw);
    V3<T> al = mk<T>(-(g.x + Iw.x * ka) / S.Ic[o][0], -(g.y + Iw.y * ka) / S.Ic[o][1], -(g.z + Iw.z * ka) / S.Ic[o][2]);
    b.ang = b.ang + rot_mul(R, al) * dt;
    b.lin.x += (-b.lin.x * kl) * dt; b.lin.y += (-b.lin.y * kl) * dt; b.lin.z += (-b.lin.z * kl - Consts<T>::g) * dt;
}
// stepPositionsMultiDof for the base: p += v dt, q <- exp(w dt) q
template <typename T> PG_HD void obj_integrate(Obj<T>& b) {
    const T dt = Consts<T>::dt;
    b.pos = b.pos + b.lin * dt;
    T fa = norm(b.ang);
    if (fa * dt > Consts<T>::pi / 4) fa = Consts<T>::pi / 4 / dt;
    T sc = fa < T(0.001) ? (T(0.5) * dt - dt * dt * dt * T(0.020833333333) * fa * fa) : sin(T(0.5) * fa * dt) / fa;
    T ax = b.ang.x * sc, ay = b.ang.y * sc, az = b.ang.z * sc, aw = cos(T(0.5) * fa * dt);
    T x = aw * b.qx + ax * b.qw + ay * b.qz - az * b.qy;
    T y = aw * b.qy - ax * b.qz + ay * b.qw + az * b.qx;
    T z = aw * b.qz + ax * b.qy - ay * b.qx + az * b.qw;
    T w = aw * b.qw - ax * b.qx - ay * b.qy - az * b.qz;
    T n = T(1) / sqrt(x * x + y * y + z * z + w * w);
    b.qx = x * n; b.qy = y * n; b.qz = z * n; b.qw = w * n;
}

template <typename T> PG_HD V3<T> box_vertex(const T* h, int k) { return mk<T>((k & 1) ? h[0] : -h[0], (k & 2) ? h[1] : -h[1], (k & 4) ? h[2] : -h[2]); }
template <typename T> PG_HD V3<T> obj_vertex(const Scene<T>& S, int o, int k) {
    if (S.shape[o] == SH_BOX) return box_vertex(S.half[o], k);
    const T c = S.half[o][0] * Consts<T>::k45;
    int a = k & 3;
    return mk<T>((a == 0 || a == 3) ? c : -c, (a < 2) ? c : -c, (k & 4) ? S.half[o][2] : -S.half[o][2]);
}
// edge e (0..11) of a box in the world: axis e / 4, the two other coordinates at -+ half by the bits of e; start point p, direction d (full length)
template <typename T> PG_HD T sdf_box(const T* h, V3<T> p, V3<T>& n, bool& face) {
    face = true;
    T dx = fabs(p.x) - h[0], dy = fabs(p.y) - h[1], dz = fabs(p.z) - h[2];
    if (dx <= 0 && dy <= 0 && dz <= 0) {
        int a = 0; T d = dx;
        if (dy > d) { a = 1; d = dy; }
        if (dz > d) { a = 2; d = dz; }
        n = mk<T>(T(0), T(0), T(0));
        if (a == 0) n.x = p.x >= 0 ? T(1) : T(-1); else if (a == 1) n.y = p.y >= 0 ? T(1) : T(-1); else n.z = p.z >= 0 ? T(1) : T(-1);
        return d;
    }
    T ox = dx > 0 ? dx : T(0), oy = dy > 0 ? dy : T(0), oz = dz > 0 ? dz : T(0);
    face = ((dx > 0) + (dy > 0) + (dz > 0)) == 1;
    T len = sqrt(ox * ox + oy * oy + oz * oz), inv = T(1) / len;
    n = mk<T>((p.x >= 0 ? ox : -ox) * inv, (p.y >= 0 ? oy : -oy) * inv, (p.z >= 0 ? oz : -oz) * inv);
    return len;
}
template <typename T> PG_HD T sdf_cyl(T r, T hz, V3<T> p, V3<T>& n, bool& face) {
    T rho = sqrt(p.x * p.x + p.y * p.y);
    T dr = rho - r, dz = fabs(p.z) - hz;
    T rx = rho > T(1e-12) ? p.x / rho : T(1), ry = rho > T(1e-12) ? p.y / rho : T(0), sz = p.z >= 0 ? T(1) : T(-1);
    face = !(dr > 0 && dz > 0);
    if (dr <= 0 && dz <= 0) { if (dr > dz) { n = mk<T>(rx, ry, T(0)); return dr; } n = mk<T>(T(0), T(0), sz); return dz; }
    T a = dr > 0 ? dr : T(0), b = dz > 0 ? dz : T(0), len = sqrt(a * a + b * b);
    n = mk<T>(rx * a / len, ry * a / len, sz * b / len);
    return len;
}
template <typename T> PG_HD void box_edge(const T* h, const Rot<T>& R, V3<T> pos, int e, V3<T>& p, V3<T>& d) {
    const int a = e >> 2, b1 = (a + 1) % 3, c1 = (a + 2) % 3;
    T l[3];
    l[a] = -h[a]; l[b1] = (e & 1) ? h[b1] : -h[b1]; l[c1] = (e & 2) ? h[c1] : -h[c1];
    p = rot_mul(R, mk<T>(l[0], l[1], l[2])) + pos;
    const V3<T> ax = a == 0 ? R.X : (a == 1 ? R.Y : R.Z);
    d = ax * (T(2) * h[a]);
}
template <typename T> PG_HD T obj_sdf(const Scene<T>& S, int o, V3<T> p, V3<T>& n, bool& face) {
    return S.shape[o] == SH_BOX ? sdf_box(S.half[o], p, n, face) : sdf_cyl(S.half[o][0], S.half[o][2], p, n, face);
}
template <typename T> PG_HD void plane_space(V3<T> n, V3<T>& p, V3<T>& q) {   // btPlaneSpace1
    if (fabs(n.z) > Consts<T>::k45) {
        T a = n.y * n.y + n.z * n.z, k = T(1) / sqrt(a);
        p = mk<T>(T(0), -n.z * k, n.y * k); q = mk<T>(a * k, -n.x * p.z, n.x * p.y);
    } else {
        T a = n.x * n.x + n.y * n.y, k = T(1) / sqrt(a);
        p = mk<T>(-n.y * k, n.x * k, T(0)); q = mk<T>(-n.z * p.y, n.z * p.x, a * k);
    }
}

// ---------------------------------------------------------------------------------------------- contact storage
// body codes: -1 static, 0..2 robot box (hand / finger 1 / finger 2), 3 + o object o
// Every robot collision box rides on link 6 (hand) or on a finger that slides on it, so a robot contact row never needs its
// 9-wide joint Jacobian: it is a wrench w (8 numbers: moment about the link-6 origin, force, the two finger-slide components)
// in the 8-dimensional operational space x = [omega6, v6, q7', q8'] = Jx q', and the solver works on that space's inverse
// inertia Lambda = Jx M^-1 Jx^T (8x8, registers).  A contact record is then pure geometry + 3 x (1/D, rhs, impulse): 17 words.
// Records and Jx live in shared memory, word-interleaved by thread (bank-conflict free).
constexpr int REC = 17;                 // words per contact record
constexpr int JX_SLOTS = 42;            // Jx: per arm joint j, angular (z_j) and linear (z_j x (O6 - p_j)) columns
// contacts per env and sub-step (later candidates are dropped; the oracle applies the same cap): robot-only scenes keep two
// 128-thread blocks per SM, scenes with objects take the whole SM's shared memory for one block
PG_HD constexpr int max_contacts(int nobj) { return nobj <= 1 ? 10 : 22; }
PG_HD constexpr int solver_slots(int nobj) { return JX_SLOTS + max_contacts(nobj) * REC; }
enum { C_P = 0, C_N = 3, C_INVD = 6, C_RHS = 9, C_APP = 12, C_MU = 15, C_CODE = 16 };

template <typename T> struct CStore {   // per-thread view of the shared-memory slab (host test build: a plain array, stride 1)
    T* base; int stride;
    PG_HD T& at(int slot) const { return base[slot * stride]; }
};
template <typename T> struct Contacts {
    CStore<T> st;
    int n, nr, cap;
    int dropped;                // candidates beyond the cap since the caller last zeroed it (counted, surfaced through pg_contact_overflows)
    int nB, nA;                 // contacts are collected in type order: [0, nB) object vertex on a plane, [nB, nB + nA) robot box on the table, then generic
    bool near;                  // the gripper is within 3 cm of the table or inside an object's broad-phase sphere (scheduling hint)
    bool capped;                // the last solve ran (nearly) all 50 sweeps (scheduling hint)
    PG_HD T& f(int c, int k) { return st.at(JX_SLOTS + c * REC + k); }
    PG_HD T& jx(int j, int a) { return st.at(6 * j + a); }
};
PG_HD constexpr int sidx(int a, int b) { return a <= b ? a * 8 - a * (a - 1) / 2 + (b - a) : b * 8 - b * (b - 1) / 2 + (a - b); }
template <typename T> struct OpSpace {
    T L[36];            // Lambda, symmetric 8x8 packed by sidx
    T v[8];             // Jx * qd (current operational-space velocity)
    V3<T> O6, hy;       // link-6 origin, hand y axis (finger slide direction) in the world
};

template <typename T, int NOBJ> struct World {
    Frame<T> F[7];              // arm link frames at the sub-step's q
    Rot<T> Rb; V3<T> cb[3];     // robot collision boxes in the world (all three share the hand's orientation)
    Rot<T> Ro[NOBJ > 0 ? NOBJ : 1];
    T Iinv[NOBJ > 0 ? NOBJ : 1][6];   // world inverse inertia (xx,xy,xz,yy,yz,zz)
};
template <typename T> PG_HD V3<T> sym6_mul(const T* I, V3<T> w) {
    return mk<T>(I[0] * w.x + I[1] * w.y + I[2] * w.z, I[1] * w.x + I[3] * w.y + I[4] * w.z, I[2] * w.x + I[4] * w.y + I[5] * w.z);
}

// geometry only: the rows are set up once the operational space is known
template <typename T>
PG_HD void add_contact(Contacts<T>& C, V3<T> P, V3<T> n, T dist, int A, int B, T mu, bool soft, bool table = false) {
    bool on_robot = (A >= 0 && A < 3) || (B >= 0 && B < 3);
    if (C.n >= C.cap) { C.dropped++; return; }
    int c = C.n++;
    if (on_robot) C.nr++;
    C.f(c, C_P) = P.x; C.f(c, C_P + 1) = P.y; C.f(c, C_P + 2) = P.z;
    C.f(c, C_N) = n.x; C.f(c, C_N + 1) = n.y; C.f(c, C_N + 2) = n.z;
    C.f(c, C_RHS) = dist;       // parked here until rows_setup
    C.f(c, C_MU) = mu;
    C.f(c, C_CODE) = (T)((A + 1) + 8 * (B + 1) + (soft ? 64 : 0) + (table ? 128 : 0));
}

template <typename T> PG_HD bool over_table(const Scene<T>& S, V3<T> p) { return p.x >= S.table_x0 && p.x <= S.table_x1 && p.y >= S.table_y0 && p.y <= S.table_y1; }

template <typename T, int NOBJ>
PG_HD void collect_contacts(const Scene<T>& S, const World<T, NOBJ>& W, const Obj<T>* ob, Contacts<T>& C) {
    C.n = 0; C.nr = 0; C.cap = max_contacts(NOBJ); C.near = false;
    const V3<T> up = mk<T>(T(0), T(0), T(1));
    // 1. object vertices against the table top / ground plane
#pragma unroll
    for (int o = 0; o < NOBJ; o++) {
        for (int k = 0; k < 8; k++) {
            V3<T> P = rot_mul(W.Ro[o], obj_vertex(S, o, k)) + ob[o].pos;
            T plane = (over_table(S, P) && P.z > T(-0.05)) ? T(0) : S.ground_z;
            T d = P.z - plane;
            if (d < S.margin) add_contact(C, P, up, d, 3 + o, -1, S.mu[o] * S.table_mu, false, true);
        }
    }
    C.nB = C.n;
    // 2. robot box vertices against the table top
#pragma unroll
    for (int b = 0; b < 3; b++) {
        T lowest = W.cb[b].z - (fabs(W.Rb.X.z) * S.rb_h[b][0] + fabs(W.Rb.Y.z) * S.rb_h[b][1] + fabs(W.Rb.Z.z) * S.rb_h[b][2]);
        C.near = C.near || lowest < T(0.03);
        if (lowest >= S.margin) continue;
        for (int k = 0; k < 8; k++) {
            // fingers: outer-face vertices only (against a plane the inner-face vertices of the pair are never the lowest points)
            if ((b == 1 && !(k & 2)) || (b == 2 && (k & 2))) continue;
            V3<T> P = rot_mul(W.Rb, box_vertex(S.rb_h[b], k)) + W.cb[b];
            if (over_table(S, P) && P.z < S.margin) add_contact(C, P, up, P.z, b, -1, S.rb_mu[b] * S.table_mu, b > 0, true);
        }
    }
    C.nA = C.n - C.nB;
    // 3. robot box <-> object, both directions
    if (NOBJ > 0) {
#pragma unroll
        for (int b = 0; b < 3; b++) {
            T rbr = sqrt(S.rb_h[b][0] * S.rb_h[b][0] + S.rb_h[b][1] * S.rb_h[b][1] + S.rb_h[b][2] * S.rb_h[b][2]);
#pragma unroll
            for (int o = 0; o < NOBJ; o++) {
                T orad = sqrt(S.half[o][0] * S.half[o][0] + S.half[o][1] * S.half[o][1] + S.half[o][2] * S.half[o][2]);
                if (norm(W.cb[b] - ob[o].pos) > rbr + orad + S.margin_grasp) continue;
                C.near = true;
                T mu = S.rb_mu[b] * S.mu[o];
                for (int k = 0; k < 8; k++) {
                    V3<T> P = rot_mul(W.Rb, box_vertex(S.rb_h[b], k)) + W.cb[b];
                    V3<T> nl, pl = rot_tmul(W.Ro[o], P - ob[o].pos);
                    bool face; T d = obj_sdf(S, o, pl, nl, face);
                    if (d < S.margin || (d < S.margin_grasp && face)) add_contact(C, P, rot_mul(W.Ro[o], nl), d, b, 3 + o, mu, b > 0);
                }
                for (int k = 0; k < 8; k++) {
                    V3<T> P = rot_mul(W.Ro[o], obj_vertex(S, o, k)) + ob[o].pos;
                    V3<T> nl, pl = rot_tmul(W.Rb, P - W.cb[b]);
                    bool face; T d = sdf_box(S.rb_h[b], pl, nl, face);
                    if (d < S.margin || (d < S.margin_grasp && face)) add_contact(C, P, rot_mul(W.Rb, nl), d, 3 + o, b, mu, b > 0);
                }
            }
        }
    }
    // 4. object <-> object
    if (NOBJ == 2) {
        T r0 = sqrt(S.half[0][0] * S.half[0][0] + S.half[0][1] * S.half[0][1] + S.half[0][2] * S.half[0][2]);
        T r1 = sqrt(S.half[1][0] * S.half[1][0] + S.half[1][1] * S.half[1][1] + S.half[1][2] * S.half[1][2]);
        if (norm(ob[0].pos - ob[NOBJ - 1].pos) <= r0 + r1 + S.margin) {
#pragma unroll
            for (int a = 0; a < 2; a++) {
                const int b = 1 - a;
                const int ia = NOBJ == 2 ? a : 0, ib = NOBJ == 2 ? b : 0;
                if (S.shape[a] == SH_BOX && S.shape[b] == SH_BOX) {
                    // 4a. box <-> box, vertices of A against B's REFERENCE FACE: the face axis of B along which the two boxes overlap least (the
                    // separating-axis choice of Bullet's box-box detector restricted to B's face normals); a vertex within the margin of that
                    // face's plane and inside the face's rectangle grown by the margin is a contact along the face normal.  B's signed-distance
                    // field alone cannot make this choice: a vertex of a cube stacked on a cube of the same size sits at a corner of the
                    // other's face, where the nearest face is a side face as often as the top (the oracle's "4a").
                    const Rot<T>& Ra = W.Ro[ia]; const Rot<T>& Rbm = W.Ro[ib];
                    const V3<T> cl = rot_tmul(Rbm, ob[ia].pos - ob[ib].pos);
                    const V3<T> Bx[3] = {Rbm.X, Rbm.Y, Rbm.Z}, Ax[3] = {Ra.X, Ra.Y, Ra.Z};
                    const T clv[3] = {cl.x, cl.y, cl.z};
                    T depth[3];
#pragma unroll
                    for (int k = 0; k < 3; k++) {
                        T proj = T(0);
#pragma unroll
                        for (int j = 0; j < 3; j++) proj += fabs(dot(Bx[k], Ax[j])) * S.half[a][j];
                        depth[k] = S.half[b][k] + proj - fabs(clv[k]);
                    }
                    int km = 0; if (depth[1] < depth[km]) km = 1; if (depth[2] < depth[km]) km = 2;
                    if (depth[km] < -S.margin) continue;            // separated along that axis
                    const T sg = clv[km] >= T(0) ? T(1) : T(-1);
                    const V3<T> nw = Bx[km] * sg;
                    const int i1 = (km + 1) % 3, i2 = (km + 2) % 3;
                    for (int k = 0; k < 8; k++) {
                        const V3<T> P = rot_mul(Ra, box_vertex(S.half[a], k)) + ob[ia].pos;
                        const V3<T> pl = rot_tmul(Rbm, P - ob[ib].pos);
                        const T plv[3] = {pl.x, pl.y, pl.z};
                        const T d = sg * plv[km] - S.half[b][km];
                        if (d < S.margin && d > T(-0.01) && fabs(plv[i1]) <= S.half[b][i1] + S.margin && fabs(plv[i2]) <= S.half[b][i2] + S.margin)
                            add_contact(C, P, nw, d, 3 + a, 3 + b, S.mu[a] * S.mu[b], false);
                    }
                    continue;
                }
                for (int k = 0; k < 8; k++) {
                    V3<T> P = rot_mul(W.Ro[(NOBJ == 2 ? a : 0)], obj_vertex(S, a, k)) + ob[(NOBJ == 2 ? a : 0)].pos;
                    V3<T> nl, pl = rot_tmul(W.Ro[(NOBJ == 2 ? b : 0)], P - ob[(NOBJ == 2 ? b : 0)].pos);
                    bool face; T d = obj_sdf(S, b, pl, nl, face);
                    if (d < S.margin) add_contact(C, P, rot_mul(W.Ro[(NOBJ == 2 ? b : 0)], nl), d, 3 + a, 3 + b, S.mu[a] * S.mu[b], false);
                }
            }
            // 4b. box <-> box, edge against edge: two boxes whose faces overlap with every vertex of either outside the other's face (a cube
            // lying rotated on a cube of the same size: tasks/stack.py:30-62) have no vertex-in-field contact.  Every pair of edges whose
            // mutual closest points are interior to both edges and closer than the margin is a contact along the edges' common
            // perpendicular, pointing from object 1 to object 0 (the oracle's "4b", same enumeration order).
            if (S.shape[0] == SH_BOX && S.shape[NOBJ - 1] == SH_BOX) {
                const V3<T> dc = ob[0].pos - ob[NOBJ - 1].pos;
#pragma unroll 1
                for (int ea = 0; ea < 12; ea++) {
                    V3<T> p1, d1; box_edge(S.half[0], W.Ro[0], ob[0].pos, ea, p1, d1);
#pragma unroll 1
                    for (int eb = 0; eb < 12; eb++) {
                        V3<T> p2, d2; box_edge(S.half[NOBJ - 1], W.Ro[NOBJ - 1], ob[NOBJ - 1].pos, eb, p2, d2);
                        const V3<T> r = p1 - p2;
                        const T A = dot(d1, d1), E = dot(d2, d2), B = dot(d1, d2), Cc = dot(d1, r), F = dot(d2, r), den = A * E - B * B;
                        if (den <= T(0.01) * A * E) continue;                      // (nearly) parallel edges
                        const T sa = (B * F - Cc * E) / den, tb = (A * F - B * Cc) / den;
                        if (sa <= T(0.02) || sa >= T(0.98) || tb <= T(0.02) || tb >= T(0.98)) continue;     // an end point is closest: a vertex contact's business
                        V3<T> n = cross(d1, d2) * (T(1) / sqrt(den));
                        if (dot(n, dc) < T(0)) n = n * T(-1);
                        const V3<T> pa = p1 + d1 * sa, pb = p2 + d2 * tb;
                        const T d = dot(pa - pb, n);
                        if (d < S.margin && d > T(-0.01)) add_contact(C, (pa + pb) * T(0.5), n, d, 3, 3 + NOBJ - 1, S.mu[0] * S.mu[NOBJ - 1], false);
                    }
                }
            }
        }
    }
}

// operational space of the gripper: Jx into the store, Lambda = Jx M^-1 Jx^T and v = Jx qd into registers
template <typename T, int NOBJ>
PG_HD void opspace_jx(const World<T, NOBJ>& W, Contacts<T>& C, OpSpace<T>& Op) {
    Op.O6 = W.F[6].p;
    Op.hy = (W.F[6].X + W.F[6].Y) * Consts<T>::k45;
#pragma unroll
    for (int j = 0; j < 7; j++) {
        V3<T> z = W.F[j].Z, l = cross(z, Op.O6 - W.F[j].p);
        C.jx(j, 0) = z.x; C.jx(j, 1) = z.y; C.jx(j, 2) = z.z; C.jx(j, 3) = l.x; C.jx(j, 4) = l.y; C.jx(j, 5) = l.z;
    }
}
template <typename T> PG_HD void opspace_lambda(const T (*Minv)[ND], const T* qd, Contacts<T>& C, OpSpace<T>& Op) {
#pragma unroll
    for (int a = 0; a < 6; a++) {
        T row[7], Y[ND], va = T(0);
#pragma unroll
        for (int j = 0; j < 7; j++) { row[j] = C.jx(j, a); va += row[j] * qd[j]; }
        Op.v[a] = va;
#pragma unroll
        for (int k = 0; k < ND; k++) {
            T t = T(0);
#pragma unroll
            for (int j = 0; j < 7; j++) t += row[j] * Minv[j][k];
            Y[k] = t;
        }
#pragma unroll
        for (int b = a; b < 6; b++) {
            T t = T(0);
#pragma unroll
            for (int k = 0; k < 7; k++) t += Y[k] * C.jx(k, b);
            Op.L[sidx(a, b)] = t;
        }
        Op.L[sidx(a, 6)] = Y[7]; Op.L[sidx(a, 7)] = Y[8];
    }
    Op.L[sidx(6, 6)] = Minv[7][7]; Op.L[sidx(6, 7)] = Minv[7][8]; Op.L[sidx(7, 7)] = Minv[8][8];
    Op.v[6] = qd[7]; Op.v[7] = qd[8];
}
template <typename T, int NOBJ>
PG_HD void opspace_setup(const World<T, NOBJ>& W, const T (*Minv)[ND], const T* qd, Contacts<T>& C, OpSpace<T>& Op) {
    opspace_jx<T, NOBJ>(W, C, Op);
    opspace_lambda<T>(Minv, qd, C, Op);
}

// per-contact decode shared by its three rows
enum { KIND_OBJ_PLANE = 0, KIND_ROBOT_TABLE = 1, KIND_GENERIC = 2 };
template <int K> struct KindTag { static constexpr int value = K; };
template <typename T, int NOBJ> struct ContactCtx {
    V3<T> P, n;
    int rb;                     // robot box (-1: none)
    T s;                        // +1: the robot is body A, -1: body B
    T sgo[NOBJ > 0 ? NOBJ : 1]; // sign of object o in this contact (0: not involved)
    bool soft;
    bool table;                 // robot box against the table plane: normal +z, tangents -y, +x (axis-aligned sparse wrenches)
};
template <typename T, int NOBJ> PG_HD ContactCtx<T, NOBJ> contact_ctx(Contacts<T>& C, int c) {
    ContactCtx<T, NOBJ> X;
    X.P = mk<T>(C.f(c, C_P), C.f(c, C_P + 1), C.f(c, C_P + 2));
    X.n = mk<T>(C.f(c, C_N), C.f(c, C_N + 1), C.f(c, C_N + 2));
    int code = (int)C.f(c, C_CODE);
    if (NOBJ == 0) {    // robot-only scene: every contact is a robot box on the table
        X.rb = (code & 7) - 1; X.s = T(1); X.soft = X.rb > 0; X.table = true;
        return X;
    }
    int A = (code & 7) - 1, B = ((code >> 3) & 7) - 1;
    X.soft = (code & 64) != 0; X.table = (code & 128) != 0;
    X.rb = (A >= 0 && A < 3) ? A : ((B >= 0 && B < 3) ? B : -1);
    X.s = (A >= 0 && A < 3) ? T(1) : T(-1);
#pragma unroll
    for (int o = 0; o < NOBJ; o++) X.sgo[o] = (A == 3 + o) ? T(1) : ((B == 3 + o) ? T(-1) : T(0));
    return X;
}

// ---------------------------------------------------------------------------------------------- contact report
// pybullet getContactPoints of the last sub-step, one row of REPORT_WORDS per contact (pg_step's contacts, include/panda_b200.h):
// point (3), normal on B pointing from B to A (3), normal force, lateral friction force 1 and its direction (1 + 3), force 2 and its
// direction (1 + 3), id_a + 32 id_b.  Forces are the solver's accumulated impulses / dt.  Body ids are the segmentation ids of
// pg_render: 1 plane, 2 table, 3 / 4 objects, 14 hand, 15 / 16 fingers.  The record's distance word holds the normal row's rhs by now,
// so the row has no contactDistance.
constexpr int REPORT_WORDS = 16;
PG_HD constexpr int report_body_id(int body) { return body < 3 ? 14 + body : body; }      // body codes 0..2 robot boxes, 3 + o objects
template <typename T, typename R> PG_HD void contact_report_row(const Scene<T>& S, Contacts<T>& C, int c, R* row) {
    const V3<T> P = mk<T>(C.f(c, C_P), C.f(c, C_P + 1), C.f(c, C_P + 2)), n = mk<T>(C.f(c, C_N), C.f(c, C_N + 1), C.f(c, C_N + 2));
    const int code = (int)C.f(c, C_CODE), A = (code & 7) - 1, B = ((code >> 3) & 7) - 1;
    V3<T> t1, t2;
    if (code & 128) { t1 = mk<T>(T(0), T(-1), T(0)); t2 = mk<T>(T(1), T(0), T(0)); }     // table kinds: the rows' axis-aligned tangents
    else plane_space(n, t1, t2);
    // static body B: robot boxes only touch the table top; an object vertex is on the table or the ground plane by collect_contacts' rule
    const int idb = B >= 0 ? report_body_id(B) : ((A < 3 || (over_table(S, P) && P.z > T(-0.05))) ? 2 : 1);
    const T k = Consts<T>::inv_dt;
    const T v[REPORT_WORDS] = {P.x, P.y, P.z, n.x, n.y, n.z, C.f(c, C_APP) * k, C.f(c, C_APP + 1) * k, t1.x, t1.y, t1.z, C.f(c, C_APP + 2) * k, t2.x, t2.y, t2.z,
                               T(report_body_id(A) + 32 * idb)};
#pragma unroll
    for (int w = 0; w < REPORT_WORDS; w++) row[w] = (R)v[w];
}
template <typename T, int NOBJ> PG_HD void robot_wrench(const OpSpace<T>& Op, const ContactCtx<T, NOBJ>& X, V3<T> d, T* w) {
    V3<T> m = cross(X.P - Op.O6, d);
    T fd = dot(Op.hy, d);
    w[0] = X.s * m.x; w[1] = X.s * m.y; w[2] = X.s * m.z; w[3] = X.s * d.x; w[4] = X.s * d.y; w[5] = X.s * d.z;
    w[6] = X.rb == 1 ? X.s * fd : T(0);
    w[7] = X.rb == 2 ? -X.s * fd : T(0);
}
template <typename T> PG_HD void lambda_mul(const OpSpace<T>& Op, const T* w, T* y) {
#pragma unroll
    for (int a = 0; a < 8; a++) {
        T t = T(0);
#pragma unroll
        for (int b = 0; b < 8; b++) t += Op.L[sidx(a, b)] * w[b];
        y[a] = t;
    }
}
// Sparse wrench of a robot-vs-table row: direction SG * e_AX, robot is body A.  Non-zeros: two moment components, one force
// component, one finger-slide component.
template <int AX, int SG, typename T, int NOBJ> struct AxisRow {
    static constexpr int I1 = (AX + 1) % 3, I2 = (AX + 2) % 3;     // r x e_AX = r[I2] e_I1 - r[I1] e_I2
    T m1, m2, f6, f7;
    PG_HD AxisRow(const OpSpace<T>& Op, const ContactCtx<T, NOBJ>& X) {
        V3<T> r = X.P - Op.O6;
        const T rr[3] = {r.x, r.y, r.z}, hh[3] = {Op.hy.x, Op.hy.y, Op.hy.z};
        m1 = T(SG) * rr[I2]; m2 = T(-SG) * rr[I1];
        T fd = T(SG) * hh[AX];
        f6 = X.rb == 1 ? fd : T(0); f7 = X.rb == 2 ? -fd : T(0);
    }
    PG_HD T jdv(const T* d8) const { return m1 * d8[I1] + m2 * d8[I2] + T(SG) * d8[3 + AX] + f6 * d8[6] + f7 * d8[7]; }
    PG_HD void lam(const OpSpace<T>& Op, T* y) const {
#pragma unroll
        for (int k = 0; k < 8; k++) y[k] = Op.L[sidx(k, I1)] * m1 + Op.L[sidx(k, I2)] * m2 + T(SG) * Op.L[sidx(k, 3 + AX)] + Op.L[sidx(k, 6)] * f6 + Op.L[sidx(k, 7)] * f7;
    }
    PG_HD void apply(const OpSpace<T>& Op, T di, T* d8, T* F8) const {
        T y[8]; lam(Op, y);
#pragma unroll
        for (int k = 0; k < 8; k++) d8[k] += y[k] * di;
        F8[I1] += m1 * di; F8[I2] += m2 * di; F8[3 + AX] += T(SG) * di; F8[6] += f6 * di; F8[7] += f7 * di;
    }
};
// Object-vs-plane row along SG * e_AX (the object is body A): J = [e; r x e], W = [e/m; Iinv (r x e)] with r x e_AX two-sparse.
template <int AX, int SG, typename T> struct ObjAxisRow {
    static constexpr int I1 = (AX + 1) % 3, I2 = (AX + 2) % 3;
    T m1, m2;
    PG_HD ObjAxisRow(V3<T> r) { const T rr[3] = {r.x, r.y, r.z}; m1 = T(SG) * rr[I2]; m2 = T(-SG) * rr[I1]; }
    PG_HD T jdv(V3<T> vl, V3<T> va) const { const T l[3] = {vl.x, vl.y, vl.z}, a[3] = {va.x, va.y, va.z}; return T(SG) * l[AX] + m1 * a[I1] + m2 * a[I2]; }
    PG_HD V3<T> wang(const T* I) const {        // Iinv (r x e): columns I1, I2 of the symmetric matrix
        const int c1[3] = {I1 == 0 ? 0 : (I1 == 1 ? 1 : 2), I1 == 0 ? 1 : (I1 == 1 ? 3 : 4), I1 == 0 ? 2 : (I1 == 1 ? 4 : 5)};
        const int c2[3] = {I2 == 0 ? 0 : (I2 == 1 ? 1 : 2), I2 == 0 ? 1 : (I2 == 1 ? 3 : 4), I2 == 0 ? 2 : (I2 == 1 ? 4 : 5)};
        return mk<T>(I[c1[0]] * m1 + I[c2[0]] * m2, I[c1[1]] * m1 + I[c2[1]] * m2, I[c1[2]] * m1 + I[c2[2]] * m2);
    }
    PG_HD void apply(const T* I, T inv_mass, T di, V3<T>& vl, V3<T>& va) const {
        const T dl = T(SG) * di * inv_mass;
        if (AX == 0) vl.x += dl; else if (AX == 1) vl.y += dl; else vl.z += dl;
        va = va + wang(I) * di;
    }
};
template <typename T> PG_HD T dot8(const T* a, const T* b) {
    T t = T(0);
#pragma unroll
    for (int i = 0; i < 8; i++) t += a[i] * b[i];
    return t;
}

// 1/D and rhs of the three rows of every contact (setupMultiBodyContactConstraint: speculative when separated, ERP when penetrating)
template <typename T, int NOBJ>
PG_HD void rows_setup(const Scene<T>& S, const World<T, NOBJ>& W, const OpSpace<T>& Op, const Obj<T>* ob, Contacts<T>& C) {
    for (int c = 0; c < C.n; c++) {
        ContactCtx<T, NOBJ> X = contact_ctx<T, NOBJ>(C, c);
        T dist = C.f(c, C_RHS);
        V3<T> t1, t2; plane_space(X.n, t1, t2);
        T erp = X.soft ? S.soft_erp : Consts<T>::erp, cfm = X.soft ? S.soft_cfm : T(0);
#pragma unroll
        for (int k = 0; k < 3; k++) {
            V3<T> d = k == 0 ? X.n : (k == 1 ? t1 : t2);
            T den = T(0), rel = T(0);
            if (NOBJ == 0 || (X.table && X.rb >= 0)) {
                T y[8];
                if (k == 0) { AxisRow<2, 1, T, NOBJ> r(Op, X); r.lam(Op, y); den += r.jdv(y); rel += r.jdv(Op.v); }
                else if (k == 1) { AxisRow<1, -1, T, NOBJ> r(Op, X); r.lam(Op, y); den += r.jdv(y); rel += r.jdv(Op.v); }
                else { AxisRow<0, 1, T, NOBJ> r(Op, X); r.lam(Op, y); den += r.jdv(y); rel += r.jdv(Op.v); }
            } else if (X.rb >= 0) { T w[8], y[8]; robot_wrench<T, NOBJ>(Op, X, d, w); lambda_mul(Op, w, y); den += dot8(w, y); rel += dot8(w, Op.v); }
#pragma unroll
            for (int o = 0; o < NOBJ; o++) {
                if (X.sgo[o] != T(0)) {
                    V3<T> r = X.P - ob[o].pos, rxd = cross(r, d);
                    den += T(1) / S.mass[o] + dot(rxd, sym6_mul(W.Iinv[o], rxd));
                    rel += X.sgo[o] * dot(d, ob[o].lin + cross(ob[o].ang, r));
                }
            }
            if (k == 0) {
                T inv = T(1) / (den + cfm);
                T pen = dist + T(1e-5), poserr = T(0), velerr = -rel;
                if (pen > 0) velerr -= pen * Consts<T>::inv_dt; else poserr = -pen * erp * Consts<T>::inv_dt;
                C.f(c, C_INVD) = inv; C.f(c, C_RHS) = (poserr + velerr) * inv;
            } else {
                T inv = T(1) / den;
                C.f(c, C_INVD + k) = inv; C.f(c, C_RHS + k) = -rel * inv;
            }
            C.f(c, C_APP + k) = T(0);
        }
    }
}

#ifdef PG_HOST_DEBUG
static long g_dbg_fallbacks = 0, g_dbg_full_starts = 0, g_dbg_sweeps = 0, g_dbg_solves = 0, g_dbg_contacts = 0;
static int g_dbg_trace[4096], g_dbg_ntrace = 0;
#endif
// Generic rows (robot box <-> object, object <-> object) work on the relative velocity change at the contact point, body A minus
// body B: u = s (v6 + w6 x r6 +- hy q'_finger) + sum_o sg_o (dv_o + dw_o x r_o).  J dv of a row along d is d . u (one u for the three
// rows of a contact), and an impulse vector f (normal: n di; friction: t1 d1 + t2 d2, solved from the same state) is applied
// with one Lambda product.
template <typename T, int NOBJ>
PG_HD V3<T> contact_dv(const OpSpace<T>& Op, const ContactCtx<T, NOBJ>& X, const T* d8, const V3<T>* dvl, const V3<T>* dva, const Obj<T>* ob) {
    V3<T> u = mk<T>(T(0), T(0), T(0));
    if (X.rb >= 0) {
        const T fs = X.rb == 1 ? d8[6] : (X.rb == 2 ? -d8[7] : T(0));
        u = (mk<T>(d8[3], d8[4], d8[5]) + cross(mk<T>(d8[0], d8[1], d8[2]), X.P - Op.O6) + Op.hy * fs) * X.s;
    }
#pragma unroll
    for (int o = 0; o < NOBJ; o++) if (X.sgo[o] != T(0)) u = u + (dvl[o] + cross(dva[o], X.P - ob[o].pos)) * X.sgo[o];
    return u;
}
template <typename T, int NOBJ>
PG_HD void contact_apply(const Scene<T>& S, const World<T, NOBJ>& W, const OpSpace<T>& Op, const ContactCtx<T, NOBJ>& X, V3<T> f,
                         T* d8, T* F8, V3<T>* dvl, V3<T>* dva, const Obj<T>* ob) {
    if (X.rb >= 0) {
        T w[8], y[8];
        robot_wrench<T, NOBJ>(Op, X, f, w);
        lambda_mul(Op, w, y);
#pragma unroll
        for (int i = 0; i < 8; i++) { F8[i] += w[i]; d8[i] += y[i]; }
    }
#pragma unroll
    for (int o = 0; o < NOBJ; o++) {
        if (X.sgo[o] != T(0)) {
            dvl[o] = dvl[o] + f * (X.sgo[o] / S.mass[o]);
            dva[o] = dva[o] + sym6_mul(W.Iinv[o], cross(X.P - ob[o].pos, f)) * X.sgo[o];
        }
    }
}

// ---------------------------------------------------------------------------------------------- full sub-step
// One 2 ms stepSimulation: unconstrained velocities, contact generation at the current poses, <= 50 sequential-impulse sweeps
// over [joint limits, motors] (direction alternating), contact normals, friction cones; exit when the largest squared
// velocity change of a sweep is <= 1e-7; semi-implicit Euler.
// The sequential-impulse loop.  FAST: the 14 arm limit rows are only watched; returns true if one of them would have engaged
// (the caller then restarts with FAST = false).  Two instantiations, so the hot loop carries only the rows it executes.
template <typename T, int NOBJ, bool FAST>
PG_HD bool pgs_solve(const T* max_imp, const Scene<T>& S, const World<T, NOBJ>& W, const OpSpace<T>& Op, const T (*Minv)[ND], JointRows<T>& R,
                     Contacts<T>& C, const Obj<T>* ob, const bool robot_contacts, T* dvq, V3<T>* dvl, V3<T>* dva) {
    const int nc = C.n;
    bool live = false;
    int it = 0;
    for (; it < 50; it++) {
        T res = T(0), watch = T(0);
        joint_rows_sweep<FAST>(max_imp, Minv, R, dvq, it, res, watch);
        if (FAST && watch > T(0)) { live = true; break; }
        if (nc > 0) {
            T d8[8], F8[8];
#pragma unroll
            for (int a = 0; a < 8; a++) { d8[a] = T(0); F8[a] = T(0); }
            if (robot_contacts) {       // operational-space velocity change so far: Jx dvq
#pragma unroll
                for (int j = 0; j < 7; j++) {
#pragma unroll
                    for (int a = 0; a < 6; a++) d8[a] += C.jx(j, a) * dvq[j];
                }
                d8[6] = dvq[7]; d8[7] = dvq[8];
            }
            // Typed passes: the three kinds of contact run different row code, and a warp pays for every kind present in any of its
            // lanes at a given contact index; looping kind by kind (collection order = kind order, so the row order is unchanged)
            // makes lanes meet in the same code even when their counts differ.
            const int eB = NOBJ > 0 ? C.nB : 0, eA = NOBJ > 0 ? C.nB + C.nA : nc;
            auto normal_row = [&](int c, auto kind) {
                constexpr int K = decltype(kind)::value;
                ContactCtx<T, NOBJ> X = contact_ctx<T, NOBJ>(C, c);
                T app = C.f(c, C_APP), inv = C.f(c, C_INVD), di = T(0);
                if constexpr (K == KIND_ROBOT_TABLE) {
                    AxisRow<2, 1, T, NOBJ> row(Op, X);
                    di = C.f(c, C_RHS) - app * (X.soft ? S.soft_cfm * inv : T(0)) - row.jdv(d8) * inv;
                    di = fmax(di, -app);              // accumulated normal impulse >= 0, on the change (short dependency chain)
                    C.f(c, C_APP) = app + di;
                    row.apply(Op, di, d8, F8);
                } else if constexpr (K == KIND_OBJ_PLANE) {       // object vertex on the table / ground plane
                    const int o = (NOBJ == 2 && X.sgo[NOBJ - 1] != T(0)) ? 1 : 0;
                    ObjAxisRow<2, 1, T> row(X.P - ob[o].pos);
                    di = C.f(c, C_RHS) - row.jdv(dvl[o], dva[o]) * inv;
                    di = fmax(di, -app);              // accumulated normal impulse >= 0, on the change (short dependency chain)
                    C.f(c, C_APP) = app + di;
                    row.apply(W.Iinv[o], T(1) / S.mass[o], di, dvl[o], dva[o]);
                } else {
                    T jd = dot(X.n, contact_dv<T, NOBJ>(Op, X, d8, dvl, dva, ob));
                    di = C.f(c, C_RHS) - app * (X.soft ? S.soft_cfm * inv : T(0)) - jd * inv;
                    di = fmax(di, -app);              // accumulated normal impulse >= 0, on the change (short dependency chain)
                    C.f(c, C_APP) = app + di;
                    contact_apply<T, NOBJ>(S, W, Op, X, X.n * di, d8, F8, dvl, dva, ob);
                }
                res = fmax(res, fabs(div_fast(di, inv)));
            };
            auto friction_rows = [&](int c, auto kind) {          // implicit friction cone over the two tangent rows
                constexpr int K = decltype(kind)::value;
                T napp = C.f(c, C_APP);
                if (napp <= T(0)) return;
                ContactCtx<T, NOBJ> X = contact_ctx<T, NOBJ>(C, c);
                T a1 = C.f(c, C_APP + 1), a2 = C.f(c, C_APP + 2), i1 = C.f(c, C_INVD + 1), i2 = C.f(c, C_INVD + 2);
                T lim = C.f(c, C_MU) * napp, d1 = T(0), d2 = T(0);
                if constexpr (K == KIND_OBJ_PLANE) {
                    const int o = (NOBJ == 2 && X.sgo[NOBJ - 1] != T(0)) ? 1 : 0;
                    V3<T> r = X.P - ob[o].pos;
                    ObjAxisRow<1, -1, T> r1(r); ObjAxisRow<0, 1, T> r2(r);
                    T s1 = a1 + C.f(c, C_RHS + 1) - r1.jdv(dvl[o], dva[o]) * i1, s2 = a2 + C.f(c, C_RHS + 2) - r2.jdv(dvl[o], dva[o]) * i2;
                    T len = sqrt(s1 * s1 + s2 * s2);
                    if (len > lim) { T f = div_fast(lim, len); s1 *= f; s2 *= f; }
                    d1 = s1 - a1; d2 = s2 - a2;
                    C.f(c, C_APP + 1) = s1; C.f(c, C_APP + 2) = s2;
                    const T im = T(1) / S.mass[o];
                    r1.apply(W.Iinv[o], im, d1, dvl[o], dva[o]); r2.apply(W.Iinv[o], im, d2, dvl[o], dva[o]);
                } else if constexpr (K == KIND_ROBOT_TABLE) {
                    AxisRow<1, -1, T, NOBJ> r1(Op, X); AxisRow<0, 1, T, NOBJ> r2(Op, X);
                    T s1 = a1 + C.f(c, C_RHS + 1) - r1.jdv(d8) * i1, s2 = a2 + C.f(c, C_RHS + 2) - r2.jdv(d8) * i2;
                    T len = sqrt(s1 * s1 + s2 * s2);
                    if (len > lim) { T f = div_fast(lim, len); s1 *= f; s2 *= f; }
                    d1 = s1 - a1; d2 = s2 - a2;
                    C.f(c, C_APP + 1) = s1; C.f(c, C_APP + 2) = s2;
                    {   // both tangent impulses act at once (the cone solved them from the same state): one Lambda product for the
                        // combined wrench  -d1 e_y + d2 e_x  at r
                        V3<T> r = X.P - Op.O6;
                        V3<T> fdir = mk<T>(d2, -d1, T(0));
                        V3<T> m = cross(r, fdir);
                        T fd = dot(Op.hy, fdir);
                        T w[8] = {m.x, m.y, m.z, fdir.x, fdir.y, T(0), X.rb == 1 ? fd : T(0), X.rb == 2 ? -fd : T(0)};
#pragma unroll
                        for (int k = 0; k < 8; k++) {
                            d8[k] += Op.L[sidx(k, 0)] * w[0] + Op.L[sidx(k, 1)] * w[1] + Op.L[sidx(k, 2)] * w[2] + Op.L[sidx(k, 3)] * w[3] + Op.L[sidx(k, 4)] * w[4]
                                   + Op.L[sidx(k, 6)] * w[6] + Op.L[sidx(k, 7)] * w[7];
                            F8[k] += w[k];
                        }
                    }
                } else {
                    V3<T> t1, t2; plane_space(X.n, t1, t2);
                    const V3<T> u = contact_dv<T, NOBJ>(Op, X, d8, dvl, dva, ob);
                    T j1 = dot(t1, u), j2 = dot(t2, u);
                    T s1 = a1 + C.f(c, C_RHS + 1) - j1 * i1, s2 = a2 + C.f(c, C_RHS + 2) - j2 * i2;
                    T len = sqrt(s1 * s1 + s2 * s2);
                    if (len > lim) { T f = div_fast(lim, len); s1 *= f; s2 *= f; }
                    d1 = s1 - a1; d2 = s2 - a2;
                    C.f(c, C_APP + 1) = s1; C.f(c, C_APP + 2) = s2;
                    contact_apply<T, NOBJ>(S, W, Op, X, t1 * d1 + t2 * d2, d8, F8, dvl, dva, ob);
                }
                res = fmax(res, fmax(fabs(div_fast(d1, i1)), fabs(div_fast(d2, i2))));
            };
            {
                int c = 0;
                if (NOBJ > 0) for (; c < eB; c++) normal_row(c, KindTag<KIND_OBJ_PLANE>{});
                for (; c < eA; c++) normal_row(c, KindTag<KIND_ROBOT_TABLE>{});
                if (NOBJ > 0) for (; c < nc; c++) normal_row(c, KindTag<KIND_GENERIC>{});
                c = 0;
                if (NOBJ > 0) for (; c < eB; c++) friction_rows(c, KindTag<KIND_OBJ_PLANE>{});
                for (; c < eA; c++) friction_rows(c, KindTag<KIND_ROBOT_TABLE>{});
                if (NOBJ > 0) for (; c < nc; c++) friction_rows(c, KindTag<KIND_GENERIC>{});
            }
            if (robot_contacts) {       // fold this sweep's contact wrench back into the joint velocities: dvq += M^-1 Jx^T F8
                T tau[ND];
#pragma unroll
                for (int j = 0; j < 7; j++) {
                    T t = T(0);
#pragma unroll
                    for (int a = 0; a < 6; a++) t += C.jx(j, a) * F8[a];
                    tau[j] = t;
                }
                tau[7] = F8[6]; tau[8] = F8[7];
#pragma unroll
                for (int i = 0; i < ND; i++) {
                    T t = T(0);
#pragma unroll
                    for (int j = 0; j < ND; j++) t += Minv[i][j] * tau[j];
                    dvq[i] += t;
                }
            }
        }
#ifdef PG_HOST_DEBUG
        g_dbg_sweeps++;
#endif
        if (res * res <= T(1e-7)) break;
    }
#ifdef PG_HOST_DEBUG
    g_dbg_solves++; g_dbg_contacts += nc;
    if (g_dbg_ntrace < 4096) g_dbg_trace[g_dbg_ntrace++] = it | (nc << 8) | (C.nr << 16);
#endif
    C.capped = it >= 49;
    return live;
}

// world frames of the arm links and of the robot's collision boxes from the joints' sines / cosines
template <typename T, int NOBJ>
PG_HD void world_robot(const Model<T>& M, const Scene<T>& S, const T* q, const T* sn, const T* cs, World<T, NOBJ>& W) {
    Frame<T> B; B.X = mk<T>(1, 0, 0); B.Y = mk<T>(0, 1, 0); B.Z = mk<T>(0, 0, 1); B.p = ld3(M.base);
    W.F[0] = fk_next<0>(M, B, sn[0], cs[0]); W.F[1] = fk_next<1>(M, W.F[0], sn[1], cs[1]); W.F[2] = fk_next<2>(M, W.F[1], sn[2], cs[2]);
    W.F[3] = fk_next<3>(M, W.F[2], sn[3], cs[3]); W.F[4] = fk_next<4>(M, W.F[3], sn[4], cs[4]); W.F[5] = fk_next<5>(M, W.F[4], sn[5], cs[5]);
    W.F[6] = fk_next<6>(M, W.F[5], sn[6], cs[6]);
    const T k = Consts<T>::k45;
    W.Rb.X = (W.F[6].X - W.F[6].Y) * k; W.Rb.Y = (W.F[6].X + W.F[6].Y) * k; W.Rb.Z = W.F[6].Z;
    V3<T> ph = W.F[6].p + W.F[6].Z * (M.hz - T(0.0584));   // hand frame origin
    V3<T> pf = W.F[6].p + W.F[6].Z * M.hz;
    W.cb[0] = ph + rot_mul(W.Rb, ld3(S.rb_c[0]));
    W.cb[1] = pf + W.Rb.Y * q[7] + rot_mul(W.Rb, ld3(S.rb_c[1]));
    W.cb[2] = pf - W.Rb.Y * q[8] + rot_mul(W.Rb, ld3(S.rb_c[2]));
}
// world inverse inertia of object o from its rotation W.Ro[o]
template <typename T, int NOBJ>
PG_HD void world_inertia(const Scene<T>& S, int o, World<T, NOBJ>& W) {
    const Rot<T>& R = W.Ro[o];
    T ix = T(1) / S.Ic[o][0], iy = T(1) / S.Ic[o][1], iz = T(1) / S.Ic[o][2];
    W.Iinv[o][0] = ix * R.X.x * R.X.x + iy * R.Y.x * R.Y.x + iz * R.Z.x * R.Z.x;
    W.Iinv[o][1] = ix * R.X.x * R.X.y + iy * R.Y.x * R.Y.y + iz * R.Z.x * R.Z.y;
    W.Iinv[o][2] = ix * R.X.x * R.X.z + iy * R.Y.x * R.Y.z + iz * R.Z.x * R.Z.z;
    W.Iinv[o][3] = ix * R.X.y * R.X.y + iy * R.Y.y * R.Y.y + iz * R.Z.y * R.Z.y;
    W.Iinv[o][4] = ix * R.X.y * R.X.z + iy * R.Y.y * R.Y.z + iz * R.Z.y * R.Z.z;
    W.Iinv[o][5] = ix * R.X.z * R.X.z + iy * R.Y.z * R.Y.z + iz * R.Z.z * R.Z.z;
}

// WATCH_LIMITS (joint control): the arm-limit rows are only watched, and the solve restarts inline with every row real when one would
// engage; !WATCH_LIMITS (ee control, bare worlds): every row real from the start.
template <typename T, int NOBJ, bool WATCH_LIMITS, bool GENERIC_MOTORS = false>
PG_HD void env_substep(const Model<T>& M, const Scene<T>& S, T* q, T* qd, const T* target, Obj<T>* ob, Contacts<T>& C, bool& full_sweep, bool& limits_active,
                       const T* mot = nullptr) {
    T sn[7], cs[7], Minv[ND][ND], qdd[ND];
    robot_dynamics(M, q, qd, sn, cs, Minv, qdd);
#pragma unroll
    for (int d = 0; d < ND; d++) qd[d] += qdd[d] * Consts<T>::dt;
    World<T, NOBJ> W;
    world_robot(M, S, q, sn, cs, W);
#pragma unroll
    for (int o = 0; o < NOBJ; o++) {
        W.Ro[o] = quat_rot(ob[o].qx, ob[o].qy, ob[o].qz, ob[o].qw);
        obj_unconstrained(S, o, ob[o], W.Ro[o]);
        world_inertia(S, o, W);
    }
    JointRows<T> R;
    joint_rows_setup<WATCH_LIMITS, GENERIC_MOTORS>(M, q, qd, target, Minv, R, mot);
    collect_contacts<T, NOBJ>(S, W, ob, C);
    OpSpace<T> Op;
    const bool robot_contacts = C.nr > 0;
    if (robot_contacts) opspace_setup<T, NOBJ>(W, Minv, qd, C, Op);
    rows_setup<T, NOBJ>(S, W, Op, ob, C);

    T dvq[ND];
    V3<T> dvl[NOBJ > 0 ? NOBJ : 1], dva[NOBJ > 0 ? NOBJ : 1];
#pragma unroll
    for (int d = 0; d < ND; d++) dvq[d] = T(0);
#pragma unroll
    for (int o = 0; o < NOBJ; o++) { dvl[o] = mk<T>(0, 0, 0); dva[o] = mk<T>(0, 0, 0); }
    // Arm limit rows are exact no-ops while they rest at zero impulse: the fast solve only watches them and, if one would engage,
    // the solve restarts from zero impulses with every row real (a watched row is an exact no-op: the result is the full sweep's, up to
    // FMA-contraction differences between the two loop instantiations).  Which of the two ran is a function of the env's own state,
    // never of the batch or the schedule.
    bool fast = WATCH_LIMITS && !full_sweep && !arm_limit_violated(M, q);
#ifdef PG_HOST_DEBUG
    if (!fast) g_dbg_full_starts++;
#endif
    bool live = false;
    if (fast) live = pgs_solve<T, NOBJ, true>(M.max_imp, S, W, Op, Minv, R, C, ob, robot_contacts, dvq, dvl, dva);
    if (!fast || live) {
        full_sweep = true;
#ifdef PG_HOST_DEBUG
        if (live) g_dbg_fallbacks++;
#endif
        if (live) {
#pragma unroll
            for (int d = 0; d < ND; d++) { dvq[d] = T(0); R.mot_app[d] = T(0); R.lim_app[2 * d] = T(0); R.lim_app[2 * d + 1] = T(0); }
#pragma unroll
            for (int o = 0; o < NOBJ; o++) { dvl[o] = mk<T>(0, 0, 0); dva[o] = mk<T>(0, 0, 0); }
            for (int c = 0; c < C.n; c++) { C.f(c, C_APP) = T(0); C.f(c, C_APP + 1) = T(0); C.f(c, C_APP + 2) = T(0); }
        }
        pgs_solve<T, NOBJ, false>(M.max_imp, S, W, Op, Minv, R, C, ob, robot_contacts, dvq, dvl, dva);
        bool any = false;
#pragma unroll
        for (int r = 0; r < 14; r++) any = any || R.lim_app[r] > T(0);
        limits_active = limits_active || any || live;
    }
#pragma unroll
    for (int d = 0; d < ND; d++) { qd[d] += dvq[d]; q[d] += qd[d] * Consts<T>::dt; }
#pragma unroll
    for (int o = 0; o < NOBJ; o++) { ob[o].lin = ob[o].lin + dvl[o]; ob[o].ang = ob[o].ang + dva[o]; obj_integrate(ob[o]); }
}


}  // namespace pg
