// panda_dyn.cuh -- per-environment Panda articulated dynamics, one thread per environment.
//
// Replaces, for the bodies panda_gym creates, what the reference obtains from pybullet's
// stepSimulation / calculateInverseKinematics / getLinkState
// (reference panda_gym/pybullet.py:52-55, :479-497, :351-400; panda_gym/envs/robots/panda.py:52-140).
//
// B200-first formulation (not Bullet's): the robot is a fixed kinematic tree known at compile time, so every
// loop over links is unrolled, the constant joint frames (roll = 0 / +-90 deg) become component permutations,
// and the forward dynamics is RNEA (bias forces) + CRBA (joint-space inertia, rigid 10-parameter composite
// inertias) + a 9x9 Cholesky factorisation held in registers.  The constraint solve (joint limits, position
// motors, contacts) needs M^-1 explicitly anyway, so the factorisation is shared between the unconstrained
// acceleration and the sequential-impulse sweep -- cheaper per env than ABA + 9 impulse responses, and
// mathematically identical (same q-ddot, same M^-1).
//
// Everything is templated on the scalar type: float is the product path, double exists for parity debugging.
#pragma once
#include <math.h>

#ifdef __CUDACC__
#define PG_HD __host__ __device__ __forceinline__
#else
#define PG_HD inline
#endif

namespace pg {

constexpr int ND = 9;           // 7 arm joints + 2 finger joints
constexpr int NPART = 10;       // damped rigid parts: 7 arm links, hand, 2 fingers

// ---------------------------------------------------------------------------------------------- model
template <typename T> struct Model {
    T base[3];
    T pT[7][3];                 // arm joint origin in the parent frame
    T m[9], h[9][3], Io[9][6];  // per dynamic body: mass, first moment, inertia about the body-frame origin (xx,xy,xz,yy,yz,zz)
    T dm[NPART], dc[NPART][3], dI[NPART][3];  // per damped part: mass, CoM in body coords, principal inertia (part axes)
    T lo[9], hi[9], max_imp[9]; // joint limits, motor impulse limit per sub-step (force * dt)
    T z7;                       // hand frame height above the link-6 origin (panda_joint8: 0.107)
    T hz;                       // finger joint frame height above the link-6 origin (0.107 + 0.0584)
    T eez;                      // grasp-target frame height above the link-6 origin (0.107 + 0.105)
    T fa[2];                    // finger slide direction sign in hand axes (+1, -1)
    T ee_scale, finger_scale;   // action scaling: 0.05 / 0.2 (panda.py:81,65); the fork's panda_cartesian.py:67,157 uses 1 / 1
};

template <typename T> struct Consts {
    static constexpr T dt = T(1.0 / 500.0);
    static constexpr T inv_dt = T(500.0);
    static constexpr T g = T(9.81);
    static constexpr T kdamp = T(0.04);          // btMultiBody linear/angular damping (SURVEY App. B.1)
    static constexpr T erp = T(0.2);
    static constexpr T k45 = T(0.70710678118654752440);
    static constexpr T pi = T(3.14159265358979323846);
};

// ---------------------------------------------------------------------------------------------- vectors
template <typename T> struct V3 { T x, y, z; };
template <typename T> PG_HD V3<T> mk(T x, T y, T z) { V3<T> r; r.x = x; r.y = y; r.z = z; return r; }
template <typename T> PG_HD V3<T> operator+(V3<T> a, V3<T> b) { return mk<T>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <typename T> PG_HD V3<T> operator-(V3<T> a, V3<T> b) { return mk<T>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <typename T> PG_HD V3<T> operator*(V3<T> a, T s) { return mk<T>(a.x * s, a.y * s, a.z * s); }
template <typename T> PG_HD T dot(V3<T> a, V3<T> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
template <typename T> PG_HD V3<T> cross(V3<T> a, V3<T> b) { return mk<T>(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
template <typename T> PG_HD T norm(V3<T> a) { return sqrt(dot(a, a)); }
template <typename T> PG_HD V3<T> ld3(const T* p) { return mk<T>(p[0], p[1], p[2]); }
template <typename T> struct SV { V3<T> a, l; };   // spatial vector: angular / linear part (motion) or moment / force

PG_HD void sincos_t(float a, float& s, float& c) {
#ifdef __CUDA_ARCH__
    sincosf(a, &s, &c);
#else
    s = sinf(a); c = cosf(a);
#endif
}
PG_HD void sincos_t(double a, double& s, double& c) { s = sin(a); c = cos(a); }
// quotient for the solver's convergence metric and cone scaling: the IEEE float division expands to a guarded sequence whose slow
// path is taken for zero numerators (the common case of an inactive row); the approximate form is one MUFU.RCP + multiply
PG_HD float div_fast(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fdividef(a, b);
#else
    return a / b;
#endif
}
PG_HD double div_fast(double a, double b) { return a / b; }

// constant part of the arm joint frames: roll about x by ROLL * 90 deg (SURVEY App. C)
PG_HD constexpr int roll_of(int i) { return i == 0 ? 0 : ((i == 1 || i == 4) ? -1 : 1); }
template <int ROLL, typename T> PG_HD V3<T> roll(V3<T> u) {   // Rx(ROLL*90) u
    if (ROLL == 1) return mk<T>(u.x, -u.z, u.y);
    if (ROLL == -1) return mk<T>(u.x, u.z, -u.y);
    return u;
}
template <int ROLL, typename T> PG_HD V3<T> to_parent(T s, T c, V3<T> u) { return roll<ROLL>(mk<T>(c * u.x - s * u.y, s * u.x + c * u.y, u.z)); }
template <int ROLL, typename T> PG_HD V3<T> to_child(T s, T c, V3<T> u) { V3<T> t = roll<-ROLL>(u); return mk<T>(c * t.x + s * t.y, c * t.y - s * t.x, t.z); }
// hand axes relative to link-6 axes: Rz(-45 deg)
template <typename T> PG_HD V3<T> hand_to_l6(V3<T> u) { const T k = Consts<T>::k45; return mk<T>(k * (u.x + u.y), k * (u.y - u.x), u.z); }
template <typename T> PG_HD V3<T> l6_to_hand(V3<T> u) { const T k = Consts<T>::k45; return mk<T>(k * (u.x - u.y), k * (u.x + u.y), u.z); }

// ---------------------------------------------------------------------------------------------- rigid inertia
template <typename T> struct RI { T m; V3<T> h; T xx, xy, xz, yy, yz, zz; };
template <typename T> PG_HD RI<T> body_inertia(const Model<T>& M, int b) {
    RI<T> r; r.m = M.m[b]; r.h = ld3(M.h[b]);
    r.xx = M.Io[b][0]; r.xy = M.Io[b][1]; r.xz = M.Io[b][2]; r.yy = M.Io[b][3]; r.yz = M.Io[b][4]; r.zz = M.Io[b][5];
    return r;
}
template <typename T> PG_HD V3<T> sym_mul(const RI<T>& I, V3<T> w) {
    return mk<T>(I.xx * w.x + I.xy * w.y + I.xz * w.z, I.xy * w.x + I.yy * w.y + I.yz * w.z, I.xz * w.x + I.yz * w.y + I.zz * w.z);
}
template <typename T> PG_HD SV<T> inertia_apply(const RI<T>& I, const SV<T>& v) {
    SV<T> f; f.a = sym_mul(I, v.a) + cross(I.h, v.l); f.l = v.l * I.m - cross(I.h, v.a); return f;
}
template <typename T> PG_HD SV<T> crf(const SV<T>& v, const SV<T>& f) { SV<T> r; r.a = cross(v.a, f.a) + cross(v.l, f.l); r.l = cross(v.a, f.l); return r; }
template <typename T> PG_HD void ri_add(RI<T>& a, const RI<T>& b) {
    a.m += b.m; a.h = a.h + b.h; a.xx += b.xx; a.xy += b.xy; a.xz += b.xz; a.yy += b.yy; a.yz += b.yz; a.zz += b.zz;
}
// express a rigid inertia given in a child frame (rotation Rz(angle) then roll, origin at r in parent coords) in the parent frame
template <int ROLL, typename T> PG_HD RI<T> ri_to_parent(T s, T c, V3<T> r, const RI<T>& in) {
    RI<T> o; o.m = in.m;
    V3<T> hR = to_parent<ROLL>(s, c, in.h);
    // Rz
    T cc = c * c, ss = s * s, cs = c * s;
    T xx = cc * in.xx - 2 * cs * in.xy + ss * in.yy;
    T yy = ss * in.xx + 2 * cs * in.xy + cc * in.yy;
    T xy = cs * (in.xx - in.yy) + (cc - ss) * in.xy;
    T xz = c * in.xz - s * in.yz;
    T yz = s * in.xz + c * in.yz;
    T zz = in.zz;
    // roll
    if (ROLL == 1) { T t; t = xy; xy = -xz; xz = t; t = yy; yy = zz; zz = t; yz = -yz; }
    else if (ROLL == -1) { T t; t = xy; xy = xz; xz = -t; t = yy; yy = zz; zz = t; yz = -yz; }
    // shift of the reference point by r
    T e = dot(r, hR), rr = dot(r, r), m = in.m;
    o.h = hR + r * m;
    o.xx = xx + m * (rr - r.x * r.x) + 2 * e - 2 * r.x * hR.x;
    o.yy = yy + m * (rr - r.y * r.y) + 2 * e - 2 * r.y * hR.y;
    o.zz = zz + m * (rr - r.z * r.z) + 2 * e - 2 * r.z * hR.z;
    o.xy = xy - m * r.x * r.y - r.x * hR.y - hR.x * r.y;
    o.xz = xz - m * r.x * r.z - r.x * hR.z - hR.x * r.z;
    o.yz = yz - m * r.y * r.z - r.y * hR.z - hR.y * r.z;
    return o;
}
// Bullet's per-link damping: force m v_c (k + k|v_c|) at the CoM, moment I w (k + k|w|); returns the bias-force contribution
template <typename T> PG_HD SV<T> damping(const Model<T>& M, int part, const SV<T>& v, bool hand_axes) {
    const T k = Consts<T>::kdamp;
    V3<T> c = ld3(M.dc[part]);
    V3<T> vc = v.l + cross(v.a, c);
    V3<T> fl = vc * (M.dm[part] * (k + k * norm(vc)));
    T ka = k + k * norm(v.a);
    V3<T> w = hand_axes ? l6_to_hand(v.a) : v.a;
    V3<T> fa = mk<T>(M.dI[part][0] * w.x * ka, M.dI[part][1] * w.y * ka, M.dI[part][2] * w.z * ka);
    if (hand_axes) fa = hand_to_l6(fa);
    SV<T> f; f.a = cross(c, fl) + fa; f.l = fl; return f;
}

// ---------------------------------------------------------------------------------------------- forward pass (RNEA, zero q-ddot)
template <int I, typename T> PG_HD void fwd_arm_link(const Model<T>& M, T s, T c, T qd, const SV<T>& vp, const SV<T>& ap, SV<T>& v, SV<T>& a, SV<T>& f) {
    constexpr int R = roll_of(I);
    V3<T> r = ld3(M.pT[I]);
    v.a = to_child<R>(s, c, vp.a); v.a.z += qd;
    v.l = to_child<R>(s, c, vp.l - cross(r, vp.a));
    a.a = to_child<R>(s, c, ap.a) + mk<T>(v.a.y * qd, -v.a.x * qd, T(0));
    a.l = to_child<R>(s, c, ap.l - cross(r, ap.a)) + mk<T>(v.l.y * qd, -v.l.x * qd, T(0));
    RI<T> In = body_inertia(M, I);
    SV<T> Ia = inertia_apply(In, a), Iv = inertia_apply(In, v), g = crf(v, Iv), d = damping(M, I, v, false);
    f.a = Ia.a + g.a + d.a; f.l = Ia.l + g.l + d.l;
    if (I == 6) { SV<T> dh = damping(M, 7, v, true); f.a = f.a + dh.a; f.l = f.l + dh.l; }
}
template <typename T> PG_HD V3<T> finger_origin(const Model<T>& M, int fi, T q) { const T k = Consts<T>::k45; T d = M.fa[fi] * k * q; return mk<T>(d, d, M.hz); }
template <typename T> PG_HD void fwd_finger(const Model<T>& M, int fi, T q, T qd, const SV<T>& v6, const SV<T>& a6, SV<T>& v, SV<T>& f) {
    V3<T> r = finger_origin(M, fi, q);
    T sq = M.fa[fi] * qd;
    v.a = l6_to_hand(v6.a);
    v.l = l6_to_hand(v6.l - cross(r, v6.a)); v.l.y += sq;
    SV<T> a;
    a.a = l6_to_hand(a6.a);
    a.l = l6_to_hand(a6.l - cross(r, a6.a)) + cross(v.a, mk<T>(T(0), sq, T(0)));
    RI<T> In = body_inertia(M, 7 + fi);
    SV<T> Ia = inertia_apply(In, a), Iv = inertia_apply(In, v), g = crf(v, Iv), d = damping(M, 8 + fi, v, false);
    f.a = Ia.a + g.a + d.a; f.l = Ia.l + g.l + d.l;
}

// walk a spatial force (moment n, force f, frame I) up to the root, recording the z-moment seen by every ancestor joint
template <int I, typename T> struct WalkUp {
    static PG_HD void run(const Model<T>& M, const T* sn, const T* cs, V3<T> n, V3<T> f, T* col) {
        constexpr int R = roll_of(I);
        V3<T> fp = to_parent<R>(sn[I], cs[I], f);
        V3<T> np = to_parent<R>(sn[I], cs[I], n) + cross(ld3(M.pT[I]), fp);
        col[I - 1] = np.z;
        WalkUp<I - 1, T>::run(M, sn, cs, np, fp, col);
    }
};
template <typename T> struct WalkUp<0, T> { static PG_HD void run(const Model<T>&, const T*, const T*, V3<T>, V3<T>, T*) {} };

// backward step for arm link I: joint bias, mass-matrix column, accumulate composite inertia / force into the parent
template <int I, typename T> PG_HD void bwd_arm_link(const Model<T>& M, const T* sn, const T* cs, RI<T>* Ic, SV<T>* f, T (*A)[ND], T* bias) {
    constexpr int R = roll_of(I);
    bias[I] = f[I].a.z;
    A[I][I] = Ic[I].zz;
    // F = Ic * [z; 0]
    V3<T> n = mk<T>(Ic[I].xz, Ic[I].yz, Ic[I].zz), fz = mk<T>(-Ic[I].h.y, Ic[I].h.x, T(0));
    T col[ND];
    WalkUp<I, T>::run(M, sn, cs, n, fz, col);
#pragma unroll
    for (int k = 0; k < I; k++) { A[k][I] = col[k]; A[I][k] = col[k]; }
    if (I > 0) {
        V3<T> r = ld3(M.pT[I]);
        ri_add(Ic[I > 0 ? I - 1 : 0], ri_to_parent<R>(sn[I], cs[I], r, Ic[I]));
        V3<T> fp = to_parent<R>(sn[I], cs[I], f[I].l);
        V3<T> np = to_parent<R>(sn[I], cs[I], f[I].a) + cross(r, fp);
        f[I > 0 ? I - 1 : 0].a = f[I > 0 ? I - 1 : 0].a + np; f[I > 0 ? I - 1 : 0].l = f[I > 0 ? I - 1 : 0].l + fp;
    }
}

// ---------------------------------------------------------------------------------------------- forward dynamics + M^-1
// In: q, qd.  Out: qdd (unconstrained joint accelerations), Minv (dense symmetric 9x9), sn/cs of the arm joints.
template <typename T> PG_HD void robot_dynamics_sc(const Model<T>& M, const T* q, const T* qd, const T* sn, const T* cs, T (*Minv)[ND], T* qdd);
template <typename T> PG_HD void robot_dynamics(const Model<T>& M, const T* q, const T* qd, T* sn, T* cs, T (*Minv)[ND], T* qdd) {
#pragma unroll
    for (int i = 0; i < 7; i++) sincos_t(q[i], sn[i], cs[i]);
    robot_dynamics_sc(M, q, qd, sn, cs, Minv, qdd);
}
// the same with the arm joints' sines / cosines supplied by the caller (the split sub-step computes the world frames and collects the
// contacts from them before it decides whether to run the dynamics at all)
template <typename T> PG_HD void robot_dynamics_sc(const Model<T>& M, const T* q, const T* qd, const T* sn, const T* cs, T (*Minv)[ND], T* qdd) {
    SV<T> f[ND];
    RI<T> Ic[ND];
    {
        SV<T> v0, a0, v, a, vn, an;
        v0.a = mk<T>(0, 0, 0); v0.l = mk<T>(0, 0, 0); a0.a = mk<T>(0, 0, 0); a0.l = mk<T>(T(0), T(0), Consts<T>::g);
        fwd_arm_link<0>(M, sn[0], cs[0], qd[0], v0, a0, v, a, f[0]);
        fwd_arm_link<1>(M, sn[1], cs[1], qd[1], v, a, vn, an, f[1]);
        fwd_arm_link<2>(M, sn[2], cs[2], qd[2], vn, an, v, a, f[2]);
        fwd_arm_link<3>(M, sn[3], cs[3], qd[3], v, a, vn, an, f[3]);
        fwd_arm_link<4>(M, sn[4], cs[4], qd[4], vn, an, v, a, f[4]);
        fwd_arm_link<5>(M, sn[5], cs[5], qd[5], v, a, vn, an, f[5]);
        fwd_arm_link<6>(M, sn[6], cs[6], qd[6], vn, an, v, a, f[6]);
        SV<T> vf;
        fwd_finger(M, 0, q[7], qd[7], v, a, vf, f[7]);
        fwd_finger(M, 1, q[8], qd[8], v, a, vf, f[8]);
    }
#pragma unroll
    for (int b = 0; b < ND; b++) Ic[b] = body_inertia(M, b);
    T A[ND][ND], bias[ND];
    // fingers: prismatic along +-y of the hand axes
#pragma unroll
    for (int fi = 0; fi < 2; fi++) {
        const int b = 7 + fi;
        T sg = M.fa[fi];
        V3<T> ax = mk<T>(T(0), sg, T(0));
        bias[b] = sg * f[b].l.y;
        A[b][b] = Ic[b].m;
        A[7][8] = T(0); A[8][7] = T(0);
        V3<T> r = finger_origin(M, fi, q[b]);
        // F = Ic * [0; ax] -> link-6 frame
        V3<T> n = cross(Ic[b].h, ax), fl = ax * Ic[b].m;
        V3<T> f6 = hand_to_l6(fl), n6 = hand_to_l6(n) + cross(r, f6);
        T col[ND];
        col[6] = n6.z;
        WalkUp<6, T>::run(M, sn, cs, n6, f6, col);
#pragma unroll
        for (int k = 0; k < 7; k++) { A[k][b] = col[k]; A[b][k] = col[k]; }
        // composite inertia and force into link 6
        const T k45 = Consts<T>::k45;
        ri_add(Ic[6], ri_to_parent<0>(-k45, k45, r, Ic[b]));
        V3<T> fp = hand_to_l6(f[b].l), np = hand_to_l6(f[b].a) + cross(r, fp);
        f[6].a = f[6].a + np; f[6].l = f[6].l + fp;
    }
    bwd_arm_link<6>(M, sn, cs, Ic, f, A, bias);
    bwd_arm_link<5>(M, sn, cs, Ic, f, A, bias);
    bwd_arm_link<4>(M, sn, cs, Ic, f, A, bias);
    bwd_arm_link<3>(M, sn, cs, Ic, f, A, bias);
    bwd_arm_link<2>(M, sn, cs, Ic, f, A, bias);
    bwd_arm_link<1>(M, sn, cs, Ic, f, A, bias);
    bwd_arm_link<0>(M, sn, cs, Ic, f, A, bias);

    // Cholesky A = L L^T (lower, in place), Linv, Minv = Linv^T Linv
    T Li[ND][ND];
#pragma unroll
    for (int j = 0; j < ND; j++) {
        T d = A[j][j];
#pragma unroll
        for (int k = 0; k < j; k++) d -= A[j][k] * A[j][k];
        T inv = T(1) / sqrt(d);
        A[j][j] = d * inv;
        Li[j][j] = inv;
#pragma unroll
        for (int i = j + 1; i < ND; i++) {
            T t = A[i][j];
#pragma unroll
            for (int k = 0; k < j; k++) t -= A[i][k] * A[j][k];
            A[i][j] = t * inv;
        }
    }
#pragma unroll
    for (int j = 0; j < ND; j++) {
#pragma unroll
        for (int i = j + 1; i < ND; i++) {
            T t = T(0);
#pragma unroll
            for (int k = j; k < i; k++) t += A[i][k] * Li[k][j];
            Li[i][j] = -t * Li[i][i];
        }
    }
#pragma unroll
    for (int i = 0; i < ND; i++) {
#pragma unroll
        for (int j = 0; j <= i; j++) {
            T t = T(0);
#pragma unroll
            for (int k = i; k < ND; k++) t += Li[k][i] * Li[k][j];
            Minv[i][j] = t; Minv[j][i] = t;
        }
    }
#pragma unroll
    for (int i = 0; i < ND; i++) {
        T t = T(0);
#pragma unroll
        for (int j = 0; j < ND; j++) t -= Minv[i][j] * bias[j];
        qdd[i] = t;
    }
}

// ---------------------------------------------------------------------------------------------- world-frame kinematics
template <typename T> struct Frame { V3<T> X, Y, Z, p; };   // columns of the world<-link rotation, origin
template <int I, typename T> PG_HD Frame<T> fk_next(const Model<T>& M, const Frame<T>& P, T s, T c) {
    constexpr int R = roll_of(I);
    Frame<T> F;
    V3<T> r = ld3(M.pT[I]);
    F.p = P.p + P.X * r.x + P.Y * r.y + P.Z * r.z;
    V3<T> Yp, Zp;
    if (R == 1) { Yp = P.Z; Zp = P.Y * T(-1); } else if (R == -1) { Yp = P.Z * T(-1); Zp = P.Y; } else { Yp = P.Y; Zp = P.Z; }
    F.X = P.X * c + Yp * s; F.Y = Yp * c - P.X * s; F.Z = Zp;
    return F;
}
// frames of the 7 arm links for joint vector q
template <typename T> PG_HD void fk_arm(const Model<T>& M, const T* q, Frame<T>* F) {
    Frame<T> B; B.X = mk<T>(1, 0, 0); B.Y = mk<T>(0, 1, 0); B.Z = mk<T>(0, 0, 1); B.p = ld3(M.base);
    T s, c;
    sincos_t(q[0], s, c); F[0] = fk_next<0>(M, B, s, c);
    sincos_t(q[1], s, c); F[1] = fk_next<1>(M, F[0], s, c);
    sincos_t(q[2], s, c); F[2] = fk_next<2>(M, F[1], s, c);
    sincos_t(q[3], s, c); F[3] = fk_next<3>(M, F[2], s, c);
    sincos_t(q[4], s, c); F[4] = fk_next<4>(M, F[3], s, c);
    sincos_t(q[5], s, c); F[5] = fk_next<5>(M, F[4], s, c);
    sincos_t(q[6], s, c); F[6] = fk_next<6>(M, F[5], s, c);
}
// link-6 spatial velocity (link-6 coordinates) for (q, qd)
template <int I, typename T> PG_HD SV<T> vel_next(const Model<T>& M, const SV<T>& vp, T q, T qd) {
    constexpr int R = roll_of(I);
    T s, c; sincos_t(q, s, c);
    SV<T> v; V3<T> r = ld3(M.pT[I]);
    v.a = to_child<R>(s, c, vp.a); v.a.z += qd;
    v.l = to_child<R>(s, c, vp.l - cross(r, vp.a));
    return v;
}
template <typename T> PG_HD SV<T> link6_velocity(const Model<T>& M, const T* q, const T* qd) {
    SV<T> v; v.a = mk<T>(0, 0, 0); v.l = mk<T>(0, 0, 0);
    v = vel_next<0>(M, v, q[0], qd[0]); v = vel_next<1>(M, v, q[1], qd[1]); v = vel_next<2>(M, v, q[2], qd[2]);
    v = vel_next<3>(M, v, q[3], qd[3]); v = vel_next<4>(M, v, q[4], qd[4]); v = vel_next<5>(M, v, q[5], qd[5]);
    v = vel_next<6>(M, v, q[6], qd[6]);
    return v;
}
// End-effector (link 11) observation as getLinkState returns it (SURVEY App. B.5): position from the cached transforms
// FK(qc), velocity = link-local velocity from the fresh (q, qd) rotated by the cached basis.
template <typename T> PG_HD void ee_observe(const Model<T>& M, const T* q, const T* qd, const T* qc, V3<T>& pos, V3<T>& vel) {
    Frame<T> F[7]; fk_arm(M, qc, F);
    pos = F[6].p + F[6].Z * M.eez;
    SV<T> v6 = link6_velocity(M, q, qd);
    V3<T> vl = v6.l + cross(v6.a, mk<T>(T(0), T(0), M.eez));
    vel = F[6].X * vl.x + F[6].Y * vl.y + F[6].Z * vl.z;
}

// ---------------------------------------------------------------------------------------------- inverse kinematics
// pybullet calculateInverseKinematics on link 11 without limits (SURVEY App. B.2): 20 damped-least-squares iterations from the
// current q, damping 0.5 on the diagonal, step clamp 45 deg, exit test on the position error only.  Solved in the 6x6
// (J J^T + 0.5 I) form, which is identical to the 9x9 (J^T J + 0.5 I) form.  tq = target quaternion (x,y,z,w), unit.
template <typename T> PG_HD void rot_to_quat(const Frame<T>& F, T* q) {
    T R0 = F.X.x, R1 = F.Y.x, R2 = F.Z.x, R3 = F.X.y, R4 = F.Y.y, R5 = F.Z.y, R6 = F.X.z, R7 = F.Y.z, R8 = F.Z.z;
    T tr = R0 + R4 + R8;
    if (tr > 0) { T s = sqrt(tr + T(1)) * 2; q[3] = T(0.25) * s; q[0] = (R7 - R5) / s; q[1] = (R2 - R6) / s; q[2] = (R3 - R1) / s; }
    else if (R0 > R4 && R0 > R8) { T s = sqrt(T(1) + R0 - R4 - R8) * 2; q[3] = (R7 - R5) / s; q[0] = T(0.25) * s; q[1] = (R1 + R3) / s; q[2] = (R2 + R6) / s; }
    else if (R4 > R8) { T s = sqrt(T(1) + R4 - R0 - R8) * 2; q[3] = (R2 - R6) / s; q[0] = (R1 + R3) / s; q[1] = T(0.25) * s; q[2] = (R5 + R7) / s; }
    else { T s = sqrt(T(1) + R8 - R0 - R4) * 2; q[3] = (R3 - R1) / s; q[0] = (R2 + R6) / s; q[1] = (R5 + R7) / s; q[2] = T(0.25) * s; }
}
// End-effector (link 11) pose from joint vector q, as getLinkState(computeForwardKinematics=1) returns it: the link-11 origin sits on
// the link-6 z axis, its axes are the link-6 axes rotated by -45 deg about z.  quat = (x, y, z, w).
template <typename T> PG_HD void ee_pose(const Model<T>& M, const T* q, V3<T>& pos, T* quat) {
    Frame<T> F[7]; fk_arm(M, q, F);
    Frame<T> Ee; const T k = Consts<T>::k45;
    Ee.p = F[6].p + F[6].Z * M.eez; Ee.X = (F[6].X - F[6].Y) * k; Ee.Y = (F[6].X + F[6].Y) * k; Ee.Z = F[6].Z;
    pos = Ee.p;
    rot_to_quat(Ee, quat);
}
template <typename T> PG_HD void ik_ee(const Model<T>& M, const T* q0, V3<T> target, const T* tq, T* qout) {
    T q[7];
#pragma unroll
    for (int i = 0; i < 7; i++) q[i] = q0[i];
    T diff = T(1e30);
    for (int it = 0; it < 20 && diff > T(1e-4); it++) {
        Frame<T> F[7]; fk_arm(M, q, F);
        // link 11 frame: origin on the link-6 z axis, axes = link-6 axes rotated by -45 deg about z
        Frame<T> E; const T k = Consts<T>::k45;
        E.p = F[6].p + F[6].Z * M.eez; E.X = (F[6].X - F[6].Y) * k; E.Y = (F[6].X + F[6].Y) * k; E.Z = F[6].Z;
        V3<T> ep = target - E.p;
        diff = norm(ep);
        T qr[4]; rot_to_quat(E, qr);
        // dq = tq * conj(qr)
        T ax = -qr[0], ay = -qr[1], az = -qr[2], aw = qr[3];
        T dx = tq[3] * ax + tq[0] * aw + tq[1] * az - tq[2] * ay;
        T dy = tq[3] * ay - tq[0] * az + tq[1] * aw + tq[2] * ax;
        T dz = tq[3] * az + tq[0] * ay - tq[1] * ax + tq[2] * aw;
        T dw = tq[3] * aw - tq[0] * ax - tq[1] * ay - tq[2] * az;
        // rotation vector: angle * axis, angle = 2 atan2(|v|, w) wrapped to (-pi, pi]  (robust form of 2 acos(w))
        T vn = sqrt(dx * dx + dy * dy + dz * dz);
        T ang = 2 * atan2(vn, dw);
        if (ang > Consts<T>::pi) ang -= 2 * Consts<T>::pi;
        T sc = vn > T(1e-12) ? ang / vn : T(0);
        T e[6] = {ep.x, ep.y, ep.z, dx * sc, dy * sc, dz * sc};
        // J columns
        T J[6][7];
#pragma unroll
        for (int j = 0; j < 7; j++) {
            V3<T> z = F[j].Z, l = cross(z, E.p - F[j].p);
            J[0][j] = l.x; J[1][j] = l.y; J[2][j] = l.z; J[3][j] = z.x; J[4][j] = z.y; J[5][j] = z.z;
        }
        T A[6][6];
#pragma unroll
        for (int a = 0; a < 6; a++)
#pragma unroll
            for (int b = 0; b <= a; b++) {
                T t = (a == b) ? T(0.5) : T(0);
#pragma unroll
                for (int j = 0; j < 7; j++) t += J[a][j] * J[b][j];
                A[a][b] = t;
            }
        // Cholesky solve A y = e
        T y[6];
#pragma unroll
        for (int j = 0; j < 6; j++) {
            T d = A[j][j];
#pragma unroll
            for (int kk = 0; kk < j; kk++) d -= A[j][kk] * A[j][kk];
            T inv = T(1) / sqrt(d);
            A[j][j] = inv;   // store the reciprocal of the diagonal
#pragma unroll
            for (int i = j + 1; i < 6; i++) {
                T t = A[i][j];
#pragma unroll
                for (int kk = 0; kk < j; kk++) t -= A[i][kk] * A[j][kk];
                A[i][j] = t * inv;
            }
        }
#pragma unroll
        for (int i = 0; i < 6; i++) { T t = e[i];
#pragma unroll
            for (int kk = 0; kk < i; kk++) t -= A[i][kk] * y[kk];
            y[i] = t * A[i][i]; }
#pragma unroll
        for (int i = 5; i >= 0; i--) { T t = y[i];
#pragma unroll
            for (int kk = i + 1; kk < 6; kk++) t -= A[kk][i] * y[kk];
            y[i] = t * A[i][i]; }
        T dth[7], mx = T(0);
#pragma unroll
        for (int j = 0; j < 7; j++) { T t = T(0);
#pragma unroll
            for (int a = 0; a < 6; a++) t += J[a][j] * y[a];
            dth[j] = t; mx = fmax(mx, fabs(t)); }
        const T lim = Consts<T>::pi / 4;
        T scl = mx > lim ? lim / mx : T(1);
#pragma unroll
        for (int j = 0; j < 7; j++) q[j] += dth[j] * scl;
    }
#pragma unroll
    for (int i = 0; i < 7; i++) qout[i] = q[i];
}

// ---------------------------------------------------------------------------------------------- any-link kinematics
// What getLinkState / calculateInverseKinematics see for an arbitrary link index 0..11 (reference panda_gym/pybullet.py:351-400,
// :479-497; link table: SURVEY App. C).  Links 0..6 are the arm links, 7 = panda_link8 (fixed, +0.107 z), 8 = hand (yaw -45 deg),
// 9 / 10 = fingers (prismatic along +-y of the hand), 11 = grasp target (+0.105 z of the hand).
template <typename T> PG_HD Frame<T> link_frame_from(const Model<T>& M, const Frame<T>* F, const T* q, int link) {
    if (link <= 6) return F[link];
    Frame<T> L = F[6];
    L.p = F[6].p + F[6].Z * M.z7;
    if (link == 7) return L;
    const T k = Consts<T>::k45;
    L.X = (F[6].X - F[6].Y) * k; L.Y = (F[6].X + F[6].Y) * k;
    if (link == 9) L.p = F[6].p + F[6].Z * M.hz + L.Y * q[7];
    else if (link == 10) L.p = F[6].p + F[6].Z * M.hz - L.Y * q[8];
    else if (link == 11) L.p = F[6].p + F[6].Z * M.eez;
    return L;
}
// centre of mass of a link in its own frame (getLinkState[0] is the CoM frame; massless links: the frame origin)
template <typename T> PG_HD V3<T> link_com(const Model<T>& M, int link) {
    if (link <= 6) return ld3(M.dc[link]);
    if (link == 8) return mk<T>(M.dc[7][0], M.dc[7][1], M.dc[7][2] - M.z7);
    if (link == 9) return ld3(M.dc[8]);
    if (link == 10) return ld3(M.dc[9]);
    return mk<T>(T(0), T(0), T(0));
}
// spatial velocity of arm link `link` (<= 6) in its own coordinates at its frame origin
template <typename T> PG_HD SV<T> arm_link_velocity(const Model<T>& M, const T* q, const T* qd, int link) {
    SV<T> v; v.a = mk<T>(0, 0, 0); v.l = mk<T>(0, 0, 0);
    v = vel_next<0>(M, v, q[0], qd[0]); if (link == 0) return v;
    v = vel_next<1>(M, v, q[1], qd[1]); if (link == 1) return v;
    v = vel_next<2>(M, v, q[2], qd[2]); if (link == 2) return v;
    v = vel_next<3>(M, v, q[3], qd[3]); if (link == 3) return v;
    v = vel_next<4>(M, v, q[4], qd[4]); if (link == 4) return v;
    v = vel_next<5>(M, v, q[5], qd[5]); if (link == 5) return v;
    return vel_next<6>(M, v, q[6], qd[6]);
}
// getLinkState(link, computeLinkVelocity=1) without computeForwardKinematics (SURVEY App. B.5): pose of the CoM frame from the
// cached transforms FK(qc); velocity = link-local velocity from the fresh (q, qd), rotated to the world by the cached basis.
template <typename T> PG_HD void link_state(const Model<T>& M, int link, const T* q, const T* qd, const T* qc, V3<T>& pos, T* quat, V3<T>& lin, V3<T>& ang) {
    Frame<T> F[7]; fk_arm(M, qc, F);
    Frame<T> L = link_frame_from(M, F, qc, link);
    V3<T> c = link_com(M, link);
    pos = L.p + L.X * c.x + L.Y * c.y + L.Z * c.z;
    rot_to_quat(L, quat);
    if (link <= 6) {
        SV<T> v = arm_link_velocity(M, q, qd, link);
        V3<T> vc = v.l + cross(v.a, c);
        lin = L.X * vc.x + L.Y * vc.y + L.Z * vc.z; ang = L.X * v.a.x + L.Y * v.a.y + L.Z * v.a.z;
    } else {
        // links riding on link 6: velocity in hand axes at the link's CoM (fresh q for the finger offsets), rotated by the cached hand basis
        SV<T> v6 = arm_link_velocity(M, q, qd, 6);
        V3<T> w = l6_to_hand(v6.a);
        T oz = link == 7 || link == 8 ? M.z7 : (link == 11 ? M.eez : M.hz);
        T oy = link == 9 ? q[7] : (link == 10 ? -q[8] : T(0));
        V3<T> r = mk<T>(c.x, oy + c.y, oz + c.z);                      // CoM relative to the link-6 origin, hand axes
        V3<T> vl = l6_to_hand(v6.l) + cross(w, r);
        if (link == 9) vl.y += qd[7]; else if (link == 10) vl.y -= qd[8];
        Frame<T> H = link_frame_from(M, F, qc, 8);
        lin = H.X * vl.x + H.Y * vl.y + H.Z * vl.z; ang = H.X * w.x + H.Y * w.y + H.Z * w.z;
    }
}
// calculateInverseKinematics for an arbitrary link (the facade's PyBullet.inverse_kinematics; ik_ee below is the env path's fixed
// link-11 instance): the same 20 DLS iterations on the URDF frame origin of `link`, all 9 dofs (finger columns are the slide
// directions for links 9 / 10, zero otherwise), no joint-limit clamping.  tq = unit target quaternion (x,y,z,w).
template <typename T> PG_HD void ik_link(const Model<T>& M, int link, const T* q0, V3<T> target, const T* tq, T* qout) {
    T q[ND];
#pragma unroll
    for (int i = 0; i < ND; i++) q[i] = q0[i];
    T diff = T(1e30);
    for (int it = 0; it < 20 && diff > T(1e-4); it++) {
        Frame<T> F[7]; fk_arm(M, q, F);
        Frame<T> E = link_frame_from(M, F, q, link);
        V3<T> ep = target - E.p;
        diff = norm(ep);
        T qr[4]; rot_to_quat(E, qr);
        T ax = -qr[0], ay = -qr[1], az = -qr[2], aw = qr[3];
        T dx = tq[3] * ax + tq[0] * aw + tq[1] * az - tq[2] * ay;
        T dy = tq[3] * ay - tq[0] * az + tq[1] * aw + tq[2] * ax;
        T dz = tq[3] * az + tq[0] * ay - tq[1] * ax + tq[2] * aw;
        T dw = tq[3] * aw - tq[0] * ax - tq[1] * ay - tq[2] * az;
        T vn = sqrt(dx * dx + dy * dy + dz * dz);
        T ang = 2 * atan2(vn, dw);
        if (ang > Consts<T>::pi) ang -= 2 * Consts<T>::pi;
        T sc = vn > T(1e-12) ? ang / vn : T(0);
        T e[6] = {ep.x, ep.y, ep.z, dx * sc, dy * sc, dz * sc};
        T J[6][ND];
        for (int j = 0; j < ND; j++) {
            V3<T> l = mk<T>(T(0), T(0), T(0)), a = l;
            if (j < 7) { if (j <= link) { a = F[j].Z; l = cross(a, E.p - F[j].p); } }
            else if (link == j + 2) l = E.Y * M.fa[j - 7];
            J[0][j] = l.x; J[1][j] = l.y; J[2][j] = l.z; J[3][j] = a.x; J[4][j] = a.y; J[5][j] = a.z;
        }
        T A[6][6], y[6];
        for (int a = 0; a < 6; a++)
            for (int b = 0; b <= a; b++) { T t = (a == b) ? T(0.5) : T(0); for (int j = 0; j < ND; j++) t += J[a][j] * J[b][j]; A[a][b] = t; }
        for (int j = 0; j < 6; j++) {       // Cholesky (reciprocal diagonal), forward / backward substitution
            T d = A[j][j]; for (int kk = 0; kk < j; kk++) d -= A[j][kk] * A[j][kk];
            T inv = T(1) / sqrt(d); A[j][j] = inv;
            for (int i = j + 1; i < 6; i++) { T t = A[i][j]; for (int kk = 0; kk < j; kk++) t -= A[i][kk] * A[j][kk]; A[i][j] = t * inv; }
        }
        for (int i = 0; i < 6; i++) { T t = e[i]; for (int kk = 0; kk < i; kk++) t -= A[i][kk] * y[kk]; y[i] = t * A[i][i]; }
        for (int i = 5; i >= 0; i--) { T t = y[i]; for (int kk = i + 1; kk < 6; kk++) t -= A[kk][i] * y[kk]; y[i] = t * A[i][i]; }
        T dth[ND], mx = T(0);
        for (int j = 0; j < ND; j++) { T t = T(0); for (int a = 0; a < 6; a++) t += J[a][j] * y[a]; dth[j] = t; mx = fmax(mx, fabs(t)); }
        const T lim = Consts<T>::pi / 4;
        T scl = mx > lim ? lim / mx : T(1);
        for (int j = 0; j < ND; j++) q[j] += dth[j] * scl;
    }
#pragma unroll
    for (int i = 0; i < ND; i++) qout[i] = q[i];
}

// ---------------------------------------------------------------------------------------------- joint-space constraint rows
// btMultiBodyJointLimitConstraint (2 rows per joint, link order) then btMultiBodyJointMotor (SURVEY App. B.3).  A joint-space
// row's Jacobian is +-e_d, so its impulse response is a column of Minv.
template <typename T> struct JointRows {
    T lim_rhs[2 * ND], lim_app[2 * ND];
    T mot_rhs[ND], mot_app[ND];
    T invD[ND];
};
// Keeps a value in its register: without it the compiler rematerialises the 27 row right-hand sides from q, qd and the targets
// inside every sweep (~5 extra instructions per row and sweep, seen in the SASS of the sweep loop).
PG_HD void pin(float& x) {
#ifdef __CUDA_ARCH__
    asm volatile("" : "+f"(x));
#endif
}
PG_HD void pin(double& x) {
#ifdef __CUDA_ARCH__
    asm volatile("" : "+d"(x));
#endif
}
// `mot` (generic motors, the bare world's setJointMotorControlArray state): [0..8] position gain kp, [9..17] velocity gain kd,
// [18..26] target velocity; NULL = the env path's POSITION_CONTROL defaults (kp 0.1, kd 1, target velocity 0).
template <bool PIN = false, bool GENERIC = false, typename T> PG_HD void joint_rows_setup(const Model<T>& M, const T* q, const T* qd, const T* target, const T (*Minv)[ND], JointRows<T>& R, const T* mot = nullptr) {
    const T inv_dt = Consts<T>::inv_dt;
#pragma unroll
    for (int d = 0; d < ND; d++) {
        T invD = T(1) / Minv[d][d];
        R.invD[d] = invD;
        T pen_lo = q[d] - M.lo[d], pen_hi = M.hi[d] - q[d];
        // speculative when inside the range (velocityError = -penetration/dt), ERP push-out plus velocity removal when violated
        T v_lo = pen_lo > 0 ? -pen_lo * inv_dt : (-pen_lo * Consts<T>::erp * inv_dt - qd[d]);
        T v_hi = pen_hi > 0 ? -pen_hi * inv_dt : (-pen_hi * Consts<T>::erp * inv_dt + qd[d]);
        R.lim_rhs[2 * d] = v_lo * invD; R.lim_rhs[2 * d + 1] = v_hi * invD;
        R.lim_app[2 * d] = T(0); R.lim_app[2 * d + 1] = T(0);
        // POSITION_CONTROL, kp = 0.1, kd = 1, target velocity 0: desired velocity 0.1 (q* - q)/dt
        T vt = T(0.1) * (target[d] - q[d]) * inv_dt;
        if (GENERIC) vt = mot[d] * (target[d] - q[d]) * inv_dt + qd[d] + mot[9 + d] * (mot[18 + d] - qd[d]);   // btMultiBodyJointMotor: kp (q* - q)/dt + v + kd (v* - v)
        R.mot_rhs[d] = (vt - qd[d]) * invD; R.mot_app[d] = T(0);
        if (PIN) { pin(R.lim_rhs[2 * d]); pin(R.lim_rhs[2 * d + 1]); pin(R.mot_rhs[d]); }   // measured: +10 % with the watched-limit sweep, -2 % with the full one
    }
}
// Both limit rows of joint D, side FIRST then the other.  The same values as two single rows: the joint's own velocity is updated
// after each row (the second row reads it), the other eight joints get the two impulse changes at once -- at most one row of a
// pair carries impulse, the other's change is exactly zero, so the sum is that one change.  Saves 8 FMAs per joint and sweep.
template <int D, int FIRST, typename T> PG_HD void limit_pair(const T (*Minv)[ND], JointRows<T>& R, T* dv, T& res) {
    T w = T(0);
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int side = h == 0 ? FIRST : 1 - FIRST;
        const T sg = side == 0 ? T(1) : T(-1);
        // clamp of the accumulated impulse to [0, 100], written on the impulse change: di = clamp(di0, -app, 100 - app).  The bounds do
        // not depend on this row's J.dv, so the chain from dv[D] to the next row's dv is FFMA -> min/max -> FFMA.
        const T app = R.lim_app[2 * D + side];
        const T di = fmin(fmax(R.lim_rhs[2 * D + side] - sg * dv[D] * R.invD[D], -app), T(100) - app);
        R.lim_app[2 * D + side] = app + di;
        const T wi = sg * di;
        dv[D] += Minv[D][D] * wi;
        w += wi;
        res = fmax(res, fabs(di * Minv[D][D]));
    }
#pragma unroll
    for (int k = 0; k < ND; k++) if (k != D) dv[k] += Minv[k][D] * w;
}
template <int D, typename T> PG_HD void motor_row(const T* max_imp, const T (*Minv)[ND], JointRows<T>& R, T* dv, T& res) {
    const T app = R.mot_app[D], mx = max_imp[D];
    const T di = fmin(fmax(R.mot_rhs[D] - dv[D] * R.invD[D], -mx - app), mx - app);     // |accumulated impulse| <= max force * dt, on the change
    R.mot_app[D] = app + di;
#pragma unroll
    for (int k = 0; k < ND; k++) dv[k] += Minv[k][D] * di;
    res = fmax(res, fabs(di * Minv[D][D]));
}
// An arm limit row that rests at zero impulse and whose update would stay clamped at zero is an exact no-op, and that is the
// state of the 14 arm limit rows in almost every sweep.  The FAST sweep therefore only *watches* them (same expression as the
// real row, 3 instructions instead of 29) and raises `live` if one would have engaged; the caller then redoes the solve with
// the full sweep.  Finger limit rows (the blocked gripper sits on its lower limit, an open one on the upper) stay real rows.
// `watch` accumulates the largest "accumulated impulse this row would reach" over the watched rows of a sweep (their applied impulse is
// exactly 0 while they are only watched, so it is just rhs - J dv / D); the sweep's caller tests watch > 0 once.
template <int D, int SIDE, typename T> PG_HD void limit_watch(const JointRows<T>& R, const T* dv, T& watch) {
    const T sg = SIDE == 0 ? T(1) : T(-1);
    watch = fmax(watch, R.lim_rhs[2 * D + SIDE] - sg * dv[D] * R.invD[D]);
}
template <int D, bool FAST, typename T> struct RowsFwd {
    static PG_HD void lim(const T (*Mi)[ND], JointRows<T>& R, T* dv, T& res, T& live) {
        RowsFwd<D - 1, FAST, T>::lim(Mi, R, dv, res, live);
        if (FAST && D < 7) { limit_watch<D, 0>(R, dv, live); limit_watch<D, 1>(R, dv, live); }
        else limit_pair<D, 0>(Mi, R, dv, res);
    }
    static PG_HD void mot(const T* M, const T (*Mi)[ND], JointRows<T>& R, T* dv, T& res) { RowsFwd<D - 1, FAST, T>::mot(M, Mi, R, dv, res); motor_row<D>(M, Mi, R, dv, res); }
};
template <bool FAST, typename T> struct RowsFwd<-1, FAST, T> {
    static PG_HD void lim(const T (*)[ND], JointRows<T>&, T*, T&, T&) {}
    static PG_HD void mot(const T*, const T (*)[ND], JointRows<T>&, T*, T&) {}
};
template <int D, bool FAST, typename T> struct RowsRev {
    static PG_HD void lim(const T (*Mi)[ND], JointRows<T>& R, T* dv, T& res, T& live) {
        if (FAST && D < 7) { limit_watch<D, 1>(R, dv, live); limit_watch<D, 0>(R, dv, live); }
        else limit_pair<D, 1>(Mi, R, dv, res);
        RowsRev<D - 1, FAST, T>::lim(Mi, R, dv, res, live);
    }
    static PG_HD void mot(const T* M, const T (*Mi)[ND], JointRows<T>& R, T* dv, T& res) { motor_row<D>(M, Mi, R, dv, res); RowsRev<D - 1, FAST, T>::mot(M, Mi, R, dv, res); }
};
template <bool FAST, typename T> struct RowsRev<-1, FAST, T> {
    static PG_HD void lim(const T (*)[ND], JointRows<T>&, T*, T&, T&) {}
    static PG_HD void mot(const T*, const T (*)[ND], JointRows<T>&, T*, T&) {}
};
// one sweep over the non-contact rows; Bullet alternates the direction with the iteration parity.  `res` accumulates the largest
// |velocity change| of the sweep (the exit test squares it: max of squares == square of the max magnitude, rounding is monotone);
// `watch` > 0 afterwards means a watched arm-limit row would have engaged.
template <bool FAST, typename T> PG_HD void joint_rows_sweep(const T* max_imp, const T (*Minv)[ND], JointRows<T>& R, T* dv, int it, T& res, T& live) {
    if (it & 1) { RowsFwd<ND - 1, FAST, T>::lim(Minv, R, dv, res, live); RowsFwd<ND - 1, FAST, T>::mot(max_imp, Minv, R, dv, res); }
    else { RowsRev<ND - 1, FAST, T>::mot(max_imp, Minv, R, dv, res); RowsRev<ND - 1, FAST, T>::lim(Minv, R, dv, res, live); }
}
template <bool FAST, typename T> PG_HD void joint_rows_sweep(const Model<T>& M, const T (*Minv)[ND], JointRows<T>& R, T* dv, int it, T& res, T& live) {
    joint_rows_sweep<FAST>(M.max_imp, Minv, R, dv, it, res, live);
}
// true when an arm joint sits on or beyond a limit at set-up: its row is live from the start, use the full sweep
template <typename T> PG_HD bool arm_limit_violated(const Model<T>& M, const T* q) {
    bool v = false;
#pragma unroll
    for (int d = 0; d < 7; d++) v = v || !(q[d] - M.lo[d] > T(0)) || !(M.hi[d] - q[d] > T(0));
    return v;
}

// ---------------------------------------------------------------------------------------------- robot-only sub-step (Reach)
// One 2 ms stepSimulation for a robot with no contacts: unconstrained acceleration, limits + motors PGS (<= 50 sweeps,
// exit when the largest squared velocity change of a sweep is <= 1e-7), semi-implicit Euler.
template <typename T> PG_HD void robot_substep(const Model<T>& M, T* q, T* qd, const T* target) {
    T sn[7], cs[7], Minv[ND][ND], qdd[ND];
    robot_dynamics(M, q, qd, sn, cs, Minv, qdd);
#pragma unroll
    for (int d = 0; d < ND; d++) qd[d] += qdd[d] * Consts<T>::dt;
    JointRows<T> R;
    joint_rows_setup(M, q, qd, target, Minv, R);
    T dv[ND];
#pragma unroll
    for (int d = 0; d < ND; d++) dv[d] = T(0);
    for (int it = 0; it < 50; it++) {
        T res = T(0), watch = T(0);
        joint_rows_sweep<false>(M, Minv, R, dv, it, res, watch);
        if (res * res <= T(1e-7)) break;
    }
#pragma unroll
    for (int d = 0; d < ND; d++) { qd[d] += dv[d]; q[d] += qd[d] * Consts<T>::dt; }
}

}  // namespace pg
