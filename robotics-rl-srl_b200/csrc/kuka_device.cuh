// Kuka button-push physics, device side (sm_100a), one thread per environment.
//
// One call of kuka_physics_step() == Kuka.applyAction's IK + 12 motor set-points
// (environments/kuka_gym/kuka.py:142-187) followed by one p.stepSimulation()
// (environments/kuka_gym/kuka_button_gym_env.py:351) of the reference, restated as (DESIGN.md):
//
//   FK in the world frame  ->  sphere contacts (flags + rows)  ->  DLS inverse kinematics
//   -> composite-rigid-body mass matrix M(q) and recursive Newton-Euler bias in WORLD coordinates
//      about the world origin (sub-tree wrenches and composite inertias accumulate by plain sums)
//   -> Cholesky M = L L^T, A = M^-1 = L^-T L^-1 held in REGISTERS (78 unique entries)
//   -> 150 projected Gauss-Seidel sweeps over [motor | limit | contact | friction] rows; the 12 motor
//      rows have unit Jacobians, so a row is  v += A[:,i] * delta  (12 FMAs, no memory traffic)
//   -> semi-implicit Euler.
//
// The formulation is deliberately different from the CPU oracle (ABA + per-row impulse responses in
// double precision); the two must agree to fp32 tolerance.
#pragma once
#include <math.h>
#include <stdint.h>
#include "kuka_params.cuh"
#include "philox.cuh"
#include "kuka_coop.cuh"

#define KK_DEV __device__ __forceinline__
// Code-shape switches (measured on B200, see DESIGN.md "Kernel code shape"): per-body passes as rolled loops over
// thread-local arrays (small code, LDL latency) or fully unrolled register code (large code, instruction-fetch bound).
#ifndef KK_ROLL_IK
#define KK_ROLL_IK 0
#endif
#ifndef KK_ROLL_DYN
#define KK_ROLL_DYN 0
#endif
// Sweeps per loop iteration (2 lets ptxas rotate the lam registers instead of copying them, but doubles the loop body beyond the ~6 KB L0
// instruction cache: measured slower in both rounds).  Packed FP32 (FFMA2, `fma.rn.f32x2`) was tried in both rounds and is NOT used: on
// B200 an FFMA2 issues at HALF the rate of an FFMA (scripts/microbench/fma_issue.cu: 2.29 vs 1.09 cycles per instruction from one warp
// per scheduler), so packing the row update buys nothing (profiles/r02_fma_issue_microbench.txt).
#ifndef KK_SWEEP_UNROLL
#define KK_SWEEP_UNROLL 1
#endif
// a second copy of the sweep loop without the contact watch, taken when no lane of the warp has a contact row to watch
#ifndef KK_SWEEP_TIGHT
#define KK_SWEEP_TIGHT 1
#endif
// sweeps per iteration of the tight loop
#ifndef KK_TIGHT_UNROLL
#define KK_TIGHT_UNROLL 1
#endif
// Measured and dropped (profiles/r02_ab_kuka_sweep.txt): folding the previous row's contribution into the impulse update ("deferred" form:
// shorter loop-carried path, one more FFMA per row -- 5.15 ms against 5.07 ms, the saturating form is already issue-bound), and the
// unscaled sweep with FMNMX clamps (round 1's form).

#if defined(KK_TIMING)      // diagnostic build: first sweep in which no motor row moved (a fixed point of the fast loop)
#define KK_PROBE_D(d) kk_probe_any |= ((d) != 0.f);
#define KK_PROBE_SWEEP() { ++kk_probe_sweep; if (!kk_probe_any && !kk_probe_conv) kk_probe_conv = kk_probe_sweep; kk_probe_any = false; }
#else
#define KK_PROBE_D(d)
#define KK_PROBE_SWEEP()
#endif
struct f3 { float x, y, z; };
struct alignas(16) kk_f4 { float x, y, z, w; };   // one 128-bit load (host-compilable stand-in for float4)
KK_DEV f3 mk3(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
KK_DEV f3 operator+(f3 a, f3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
KK_DEV f3 operator-(f3 a, f3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
KK_DEV f3 operator*(float s, f3 a) { return mk3(s * a.x, s * a.y, s * a.z); }
KK_DEV float dot3(f3 a, f3 b) { return fmaf(a.x, b.x, fmaf(a.y, b.y, a.z * b.z)); }
KK_DEV f3 cross3(f3 a, f3 b) { return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
KK_DEV float norm3(f3 a) { return sqrtf(dot3(a, a)); }
// symmetric 3x3 (xx xy xz yy yz zz) times vector
KK_DEV f3 symv(const float* I, f3 v) {
    return mk3(I[0] * v.x + I[1] * v.y + I[2] * v.z, I[1] * v.x + I[3] * v.y + I[4] * v.z, I[2] * v.x + I[4] * v.y + I[5] * v.z);
}

// parent of each body: chain 0..7, fingers 8->9 and 10->11 hanging off the gripper base (7)
#define KK_PAR(i) ((i) == 0 ? -1 : (i) == 10 ? 7 : (i) - 1)

// ---- per-env dynamic state, register resident across the steps of a fused rollout ----
struct KukaEnv {
    float q[KK_NB], qd[KK_NB];
    float qb, qdb;           // button glider
    float ee[3];             // commanded end-effector position (kuka.py:73,134-139)
    float bbx, bby, bbz;     // button base origin (z moves only in the moving-button variant)
    float bspeed;            // signed button speed (moving-button variant)
    double by64;             // moving button: target y carried in float64 exactly like the reference's numpy accumulation,
                             // so the bounce at |y| > 0.3 happens on the same step (a 1-ulp matter after 300 additions of 0.001)
    float tgt[3];            // button_pos: target frozen at reset (:273-274)
    float grip[3], eepos[3]; // link states after the last step
    int counter, n_contacts, n_outside, terminated;
    int cbutton, ctable;     // manifold flags of the last stepSimulation
    uint32_t episode, total_steps;
    float ep_ret; int ep_len;
    // ---- Kuka2ButtonGymEnv only (kuka_2button_gym_env.py): second button body + goal bookkeeping ----
    float qb2, qdb2;         // second button glider
    float bb2x, bb2y;        // second button base origin (z = P.btn_base[2]: both rest on the table)
    int n_contacts2;         // n_contacts[1]; n_contacts above is n_contacts[0]
    int goal_id;             // which button is the next one to press (:43)
    int cany0, cany1;        // manifold flags: contact with ANY link of button 1 / 2 (getContactPoints without a link index, :165)
};

struct KukaKin {             // kinematics of the current configuration
    f3 a[KK_NB];             // joint axes, world
    f3 p[KK_NB];             // joint frame origins, world
    f3 c[KK_NB];             // centres of mass, world
    f3 pv[KK_NB];            // p x a: linear part of the joint motion vector about the world origin
    float Iw[KK_NB][6];      // rotational inertia about the COM, world axes
    float R6[9];             // rotation of the IK link (body 6)
};

struct KukaContacts {        // contact rows of this step (rare; lives in local memory)
    int n;
    int body[KK_MAXC], shape[KK_MAXC];
    float dist[KK_MAXC];
    f3 nrm[KK_MAXC], pt[KK_MAXC];
};

// sphere vs upright finite cylinder (axis +z through (cx, cy), z in [z0, z1], radius R)
KK_DEV void sphere_cylinder(f3 s, float r, float cx, float cy, float z0, float z1, float R, float& dist, f3& n) {
    const float dx = s.x - cx, dy = s.y - cy;
    const float rho = sqrtf(dx * dx + dy * dy);
    const f3 radial = rho > 1e-12f ? mk3(dx / rho, dy / rho, 0.f) : mk3(1.f, 0.f, 0.f);
    float d;
    if (s.z >= z1 || s.z <= z0) {
        const float zf = s.z >= z1 ? z1 : z0;
        if (rho <= R) { d = fabsf(s.z - zf); n = mk3(0.f, 0.f, s.z >= z1 ? 1.f : -1.f); }
        else { const f3 vec = mk3(dx - radial.x * R, dy - radial.y * R, s.z - zf); d = norm3(vec); n = (1.0f / d) * vec; }
    } else if (rho > R) {
        d = rho - R; n = radial;
    } else {
        const float d_top = z1 - s.z, d_side = R - rho;
        if (d_top <= d_side) { d = -d_top; n = mk3(0.f, 0.f, 1.f); } else { d = -d_side; n = radial; }
    }
    dist = d - r;
}

// Forward kinematics + link states + collision detection against table / button disc / button stack.
//
// CODE-SIZE NOTE (measured, profiles/): this kernel runs ONE warp per scheduler, and everything outside the PGS sweep
// executes once per step.  Fully unrolled, that once-per-step code was ~9000 SASS instructions (145 KB) that each warp
// streamed from L2 every step -- 58% of all stall samples were `no_inst` (instruction fetch).  The per-body passes are
// therefore ROLLED loops over the 12 bodies with their arrays in thread-local memory: a few hundred instructions that
// stay resident in the instruction caches.
template <bool WITH_CONTACTS, bool TWOB>
KK_DEV void kuka_fk(const KukaParams& P, KukaEnv& e, KukaKin& k, KukaContacts& ct) {
    float R[9], R7[9];
    float Rall[WITH_CONTACTS ? KK_NB : 1][9];  // per-body rotations for the sphere loop (local memory)
    float ql[KK_NB];
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) ql[i] = e.q[i];
    f3 p = mk3(P.base[0], P.base[1], P.base[2]), p7 = p;
    R[0] = 1.f; R[1] = 0.f; R[2] = 0.f; R[3] = 0.f; R[4] = 1.f; R[5] = 0.f; R[6] = 0.f; R[7] = 0.f; R[8] = 1.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) R7[t] = R[t];
    int cbutton = 0, ctable = 0, cany0 = 0, cany1 = 0;
    float zmin_body = 1e30f;
    if (WITH_CONTACTS) ct.n = 0;
    const float bz = e.bbz;
    const float disc0 = bz + P.glider_z + e.qb + P.disc_z0, disc1 = bz + P.glider_z + e.qb + P.disc_z1;
    const float b2z = P.btn_base[2];
    const float disc20 = b2z + P.glider_z + e.qb2 + P.disc_z0, disc21 = b2z + P.glider_z + e.qb2 + P.disc_z1;
    float zmax_shapes = fmaxf(disc1, fmaxf(bz + P.stack_top, P.table_z));
    if (TWOB) zmax_shapes = fmaxf(zmax_shapes, fmaxf(disc21, b2z + P.stack_top));
#pragma unroll 1
    for (int i = 0; i < KK_NB; ++i) {
        if (i == 10) {  // second finger restarts from the gripper base
#pragma unroll
            for (int t = 0; t < 9; ++t) R[t] = R7[t];
            p = p7;
        }
        // child frame: p_i = p_parent + R_parent * origin ; R_i = R_parent * rot * Rodrigues(axis, q)
        const float ox = P.org[i][0], oy = P.org[i][1], oz = P.org[i][2];
        p = mk3(p.x + R[0] * ox + R[1] * oy + R[2] * oz, p.y + R[3] * ox + R[4] * oy + R[5] * oz, p.z + R[6] * ox + R[7] * oy + R[8] * oz);
        float s, c;
        sincosf(ql[i], &s, &c);
        const float t = 1.f - c, ax = P.axis[i][0], ay = P.axis[i][1], az = P.axis[i][2];
        const float Q[9] = {c + t * ax * ax, t * ax * ay - s * az, t * ax * az + s * ay,
                            t * ax * ay + s * az, c + t * ay * ay, t * ay * az - s * ax,
                            t * ax * az - s * ay, t * ay * az + s * ax, c + t * az * az};
        float B[9], Rn[9];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int cc = 0; cc < 3; ++cc)
                B[3 * r + cc] = P.rot[i][3 * r] * Q[cc] + P.rot[i][3 * r + 1] * Q[3 + cc] + P.rot[i][3 * r + 2] * Q[6 + cc];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int cc = 0; cc < 3; ++cc)
                Rn[3 * r + cc] = R[3 * r] * B[cc] + R[3 * r + 1] * B[3 + cc] + R[3 * r + 2] * B[6 + cc];
#pragma unroll
        for (int t2 = 0; t2 < 9; ++t2) R[t2] = Rn[t2];
        const f3 ai = mk3(R[0] * ax + R[1] * ay + R[2] * az, R[3] * ax + R[4] * ay + R[5] * az, R[6] * ax + R[7] * ay + R[8] * az);
        const float mx = P.com[i][0], my = P.com[i][1], mz = P.com[i][2];
        k.p[i] = p;
        k.a[i] = ai;
        k.pv[i] = cross3(p, ai);
        k.c[i] = mk3(p.x + R[0] * mx + R[1] * my + R[2] * mz, p.y + R[3] * mx + R[4] * my + R[5] * mz, p.z + R[6] * mx + R[7] * my + R[8] * mz);
        {   // Iw = R Ic R^T
            const float I0 = P.Ic[i][0], I1 = P.Ic[i][1], I2 = P.Ic[i][2], I3 = P.Ic[i][3], I4 = P.Ic[i][4], I5 = P.Ic[i][5];
            float T[9];
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                T[3 * r + 0] = R[3 * r] * I0 + R[3 * r + 1] * I1 + R[3 * r + 2] * I2;
                T[3 * r + 1] = R[3 * r] * I1 + R[3 * r + 1] * I3 + R[3 * r + 2] * I4;
                T[3 * r + 2] = R[3 * r] * I2 + R[3 * r + 1] * I4 + R[3 * r + 2] * I5;
            }
            k.Iw[i][0] = T[0] * R[0] + T[1] * R[1] + T[2] * R[2];
            k.Iw[i][1] = T[0] * R[3] + T[1] * R[4] + T[2] * R[5];
            k.Iw[i][2] = T[0] * R[6] + T[1] * R[7] + T[2] * R[8];
            k.Iw[i][3] = T[3] * R[3] + T[4] * R[4] + T[5] * R[5];
            k.Iw[i][4] = T[3] * R[6] + T[4] * R[7] + T[5] * R[8];
            k.Iw[i][5] = T[6] * R[6] + T[7] * R[7] + T[8] * R[8];
        }
        if (i == 6) {
#pragma unroll
            for (int t2 = 0; t2 < 9; ++t2) k.R6[t2] = R[t2];
        }
        if (i == 7) {
#pragma unroll
            for (int t2 = 0; t2 < 9; ++t2) R7[t2] = R[t2];
            p7 = p;
        }
        if (WITH_CONTACTS) {
#pragma unroll
            for (int t2 = 0; t2 < 9; ++t2) Rall[i][t2] = R[t2];
            if (i >= P.sph_min_body) zmin_body = fminf(zmin_body, p.z);
        }
    }
    // Collision detection: ONE copy of the sphere-vs-shape code, runtime loop over the spheres.  The whole loop is skipped
    // while the lowest sphere-carrying body frame is more than (reach + margin) above every shape -- most of an episode
    // (this loop was 10 % of the kernel's stall samples before the test, profiles/r01).
    if (WITH_CONTACTS && zmin_body - P.sph_reach - zmax_shapes <= P.cdist) {
#pragma unroll 1
        for (int sidx = 0; sidx < P.nsph; ++sidx) {
            const int b = P.sph_body[sidx];
            const float* Rb = Rall[b];
            const f3 pb = k.p[b];
            const float r = P.sph_r[sidx];
            const float scz = pb.z + Rb[6] * P.sph_c[sidx][0] + Rb[7] * P.sph_c[sidx][1] + Rb[8] * P.sph_c[sidx][2];
            if (scz - r - zmax_shapes > P.cdist) continue;  // cheap reject on z alone: well above every shape
            const f3 sc = mk3(pb.x + Rb[0] * P.sph_c[sidx][0] + Rb[1] * P.sph_c[sidx][1] + Rb[2] * P.sph_c[sidx][2],
                              pb.y + Rb[3] * P.sph_c[sidx][0] + Rb[4] * P.sph_c[sidx][1] + Rb[5] * P.sph_c[sidx][2], scz);
#pragma unroll 1
            for (int shape = 0; shape < (TWOB ? 5 : 3); ++shape) {   // 0 table, 1 / 2 disc / stack of button 1, 3 / 4 of button 2
                float dist; f3 nn;
                if (shape == 0) {
                    if (sc.x < P.txmin || sc.x > P.txmax || sc.y < P.tymin || sc.y > P.tymax) continue;
                    dist = sc.z - P.table_z - r; nn = mk3(0.f, 0.f, 1.f);
                } else if (!TWOB || shape < 3) {
                    const float z0 = shape == 1 ? disc0 : bz, z1 = shape == 1 ? disc1 : bz + P.stack_top;
                    sphere_cylinder(sc, r, e.bbx, e.bby, z0, z1, shape == 1 ? P.disc_r : P.stack_r, dist, nn);
                } else {
                    const float z0 = shape == 3 ? disc20 : b2z, z1 = shape == 3 ? disc21 : b2z + P.stack_top;
                    sphere_cylinder(sc, r, e.bb2x, e.bb2y, z0, z1, shape == 3 ? P.disc_r : P.stack_r, dist, nn);
                }
                if (dist > P.cdist) continue;
                if (shape == 0) ctable = 1;
                if (shape == 1) cbutton = 1;
                if (TWOB) { if (shape == 1 || shape == 2) cany0 = 1; if (shape >= 3) cany1 = 1; }
                if (ct.n < P.max_contacts && ct.n < KK_MAXC) {
                    const int n = ct.n;
                    ct.body[n] = b; ct.shape[n] = shape; ct.dist[n] = dist; ct.nrm[n] = nn;
                    ct.pt[n] = sc - r * nn;
                    ct.n = n + 1;
                }
            }
        }
    }
    if (WITH_CONTACTS) { e.cbutton = cbutton; e.ctable = ctable; if (TWOB) { e.cany0 = cany0; e.cany1 = cany1; } }
    e.grip[0] = k.c[8].x; e.grip[1] = k.c[8].y; e.grip[2] = k.c[8].z;   // getLinkState(kuka, 8)[0]: COM of link 8
    e.eepos[0] = k.p[6].x; e.eepos[1] = k.p[6].y; e.eepos[2] = k.p[6].z;
}

// (x, y, z, w) of a rotation matrix, branch on the largest diagonal term
KK_DEV void quat_from_matrix(const float* R, float* q) {
    const float tr = R[0] + R[4] + R[8];
    if (tr > 0.f) {
        const float s = sqrtf(tr + 1.0f) * 2.f;
        q[3] = 0.25f * s; q[0] = (R[7] - R[5]) / s; q[1] = (R[2] - R[6]) / s; q[2] = (R[3] - R[1]) / s;
    } else if (R[0] > R[4] && R[0] > R[8]) {
        const float s = sqrtf(1.0f + R[0] - R[4] - R[8]) * 2.f;
        q[3] = (R[7] - R[5]) / s; q[0] = 0.25f * s; q[1] = (R[1] + R[3]) / s; q[2] = (R[2] + R[6]) / s;
    } else if (R[4] > R[8]) {
        const float s = sqrtf(1.0f + R[4] - R[0] - R[8]) * 2.f;
        q[3] = (R[2] - R[6]) / s; q[0] = (R[1] + R[3]) / s; q[1] = 0.25f * s; q[2] = (R[5] + R[7]) / s;
    } else {
        const float s = sqrtf(1.0f + R[8] - R[0] - R[4]) * 2.f;
        q[3] = (R[3] - R[1]) / s; q[0] = (R[2] + R[6]) / s; q[1] = (R[5] + R[7]) / s; q[2] = 0.25f * s;
    }
}

#if KK_ROLL_IK
// One damped-least-squares IK iteration at the current joint state (pybullet 1.8.6 / BussIK DLS):
// dtheta = (J^T J + lambda I)^-1 J^T e over the 7 arm joints.  The 7x7 normal equations are formed and
// solved in float64: they square the Jacobian's condition number, which float32 cannot afford.
// Rolled loops over thread-local arrays (see the code-size note above kuka_fk).
KK_DEV void kuka_ik(const KukaParams& P, const KukaEnv& e, const KukaKin& k, float* q_ik) {
    constexpr int n = 7;
    float J[n][6];
    const f3 pe = k.p[6];
#pragma unroll 1
    for (int j = 0; j < n; ++j) {
        const f3 aj = k.a[j];
        const f3 l = cross3(aj, pe - k.p[j]);
        J[j][0] = l.x; J[j][1] = l.y; J[j][2] = l.z; J[j][3] = aj.x; J[j][4] = aj.y; J[j][5] = aj.z;
    }
    float err[6];
    err[0] = e.ee[0] - pe.x; err[1] = e.ee[1] - pe.y; err[2] = e.ee[2] - pe.z;
    float qc[4];
    quat_from_matrix(k.R6, qc);
    const float cx = -qc[0], cy = -qc[1], cz = -qc[2], cw = qc[3];
    const float dx = P.ikq[3] * cx + P.ikq[0] * cw + P.ikq[1] * cz - P.ikq[2] * cy;
    const float dy = P.ikq[3] * cy - P.ikq[0] * cz + P.ikq[1] * cw + P.ikq[2] * cx;
    const float dz = P.ikq[3] * cz + P.ikq[0] * cy - P.ikq[1] * cx + P.ikq[2] * cw;
    const float dw = P.ikq[3] * cw - P.ikq[0] * cx - P.ikq[1] * cy - P.ikq[2] * cz;
    const float vn = sqrtf(dx * dx + dy * dy + dz * dz);
    // angle = 2 atan2(|v|, w) (== btQuaternion::getAngle, but well conditioned for small angles in fp32)
    float angle = 2.0f * atan2f(vn, dw);
    if (angle > 3.14159265358979f) angle -= 6.28318530717959f;
    if (vn > 1e-12f) { const float sc = angle / vn; err[3] = sc * dx; err[4] = sc * dy; err[5] = sc * dz; }
    else { err[3] = err[4] = err[5] = 0.f; }
    double A[n][n], b[n];
#pragma unroll 1
    for (int i = 0; i < n; ++i) {
#pragma unroll 1
        for (int j = 0; j <= i; ++j) {
            double acc = 0.0;
#pragma unroll
            for (int r = 0; r < 6; ++r) acc = fma((double)J[i][r], (double)J[j][r], acc);
            A[i][j] = acc;
        }
        A[i][i] += P.ik_damp;
        double acc = 0.0;
#pragma unroll
        for (int r = 0; r < 6; ++r) acc = fma((double)J[i][r], (double)err[r], acc);
        b[i] = acc;
    }
    // Cholesky A = L L^T (A is SPD thanks to the damping), forward/back substitution
#pragma unroll 1
    for (int j = 0; j < n; ++j) {
        double d = A[j][j];
        for (int kk = 0; kk < j; ++kk) d -= A[j][kk] * A[j][kk];
        const double inv = rsqrt(d);
        A[j][j] = inv;  // store 1 / L_jj
#pragma unroll 1
        for (int i = j + 1; i < n; ++i) {
            double acc = A[i][j];
            for (int kk = 0; kk < j; ++kk) acc -= A[i][kk] * A[j][kk];
            A[i][j] = acc * inv;
        }
    }
#pragma unroll 1
    for (int i = 0; i < n; ++i) {
        double acc = b[i];
        for (int kk = 0; kk < i; ++kk) acc -= A[i][kk] * b[kk];
        b[i] = acc * A[i][i];
    }
#pragma unroll 1
    for (int i = n - 1; i >= 0; --i) {
        double acc = b[i];
        for (int kk = i + 1; kk < n; ++kk) acc -= A[kk][i] * b[kk];
        b[i] = acc * A[i][i];
    }
    double mx = 0.0;
#pragma unroll
    for (int i = 0; i < n; ++i) mx = fmax(mx, fabs(b[i]));
    const double max_angle = 0.78539816339744830962;  // BussIK MaxAngleDLS = 45 degrees
    const double scale = mx > max_angle ? max_angle / mx : 1.0;
#pragma unroll
    for (int i = 0; i < n; ++i) q_ik[i] = e.q[i] + (float)(scale * b[i]);
}

#else
// One damped-least-squares IK iteration at the current joint state (pybullet 1.8.6 / BussIK DLS):
// dtheta = (J^T J + lambda I)^-1 J^T e over the 7 arm joints.  The 7x7 normal equations are formed and
// solved in float64: they square the Jacobian's condition number, which float32 cannot afford.
KK_DEV void kuka_ik(const KukaParams& P, const KukaEnv& e, const KukaKin& k, float* q_ik) {
    constexpr int n = 7;
    float J[6][n];
#pragma unroll
    for (int j = 0; j < n; ++j) {
        const f3 l = cross3(k.a[j], k.p[6] - k.p[j]);
        J[0][j] = l.x; J[1][j] = l.y; J[2][j] = l.z; J[3][j] = k.a[j].x; J[4][j] = k.a[j].y; J[5][j] = k.a[j].z;
    }
    float err[6];
    err[0] = e.ee[0] - k.p[6].x; err[1] = e.ee[1] - k.p[6].y; err[2] = e.ee[2] - k.p[6].z;
    float qc[4];
    quat_from_matrix(k.R6, qc);
    const float cx = -qc[0], cy = -qc[1], cz = -qc[2], cw = qc[3];
    const float dx = P.ikq[3] * cx + P.ikq[0] * cw + P.ikq[1] * cz - P.ikq[2] * cy;
    const float dy = P.ikq[3] * cy - P.ikq[0] * cz + P.ikq[1] * cw + P.ikq[2] * cx;
    const float dz = P.ikq[3] * cz + P.ikq[0] * cy - P.ikq[1] * cx + P.ikq[2] * cw;
    const float dw = P.ikq[3] * cw - P.ikq[0] * cx - P.ikq[1] * cy - P.ikq[2] * cz;
    const float vn = sqrtf(dx * dx + dy * dy + dz * dz);
    // angle = 2 atan2(|v|, w) (== btQuaternion::getAngle, but well conditioned for small angles in fp32)
    float angle = 2.0f * atan2f(vn, dw);
    if (angle > 3.14159265358979f) angle -= 6.28318530717959f;
    if (vn > 1e-12f) { const float s = angle / vn; err[3] = s * dx; err[4] = s * dy; err[5] = s * dz; }
    else { err[3] = err[4] = err[5] = 0.f; }
    double A[n][n], b[n];
#pragma unroll
    for (int i = 0; i < n; ++i) {
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double s = 0.0;
#pragma unroll
            for (int r = 0; r < 6; ++r) s = fma((double)J[r][i], (double)J[r][j], s);
            A[i][j] = s;
        }
        A[i][i] += P.ik_damp;
        double s = 0.0;
#pragma unroll
        for (int r = 0; r < 6; ++r) s = fma((double)J[r][i], (double)err[r], s);
        b[i] = s;
    }
    // Cholesky A = L L^T (A is SPD thanks to the damping), forward/back substitution
#pragma unroll
    for (int j = 0; j < n; ++j) {
        double d = A[j][j];
#pragma unroll
        for (int kk = 0; kk < j; ++kk) d -= A[j][kk] * A[j][kk];
        const double inv = rsqrt(d);
        A[j][j] = inv;  // store 1 / L_jj
#pragma unroll
        for (int i = j + 1; i < n; ++i) {
            double s = A[i][j];
#pragma unroll
            for (int kk = 0; kk < j; ++kk) s -= A[i][kk] * A[j][kk];
            A[i][j] = s * inv;
        }
    }
#pragma unroll
    for (int i = 0; i < n; ++i) {
        double s = b[i];
#pragma unroll
        for (int kk = 0; kk < i; ++kk) s -= A[i][kk] * b[kk];
        b[i] = s * A[i][i];
    }
#pragma unroll
    for (int i = n - 1; i >= 0; --i) {
        double s = b[i];
#pragma unroll
        for (int kk = i + 1; kk < n; ++kk) s -= A[kk][i] * b[kk];
        b[i] = s * A[i][i];
    }
    double mx = 0.0;
#pragma unroll
    for (int i = 0; i < n; ++i) mx = fmax(mx, fabs(b[i]));
    const double max_angle = 0.78539816339744830962;  // BussIK MaxAngleDLS = 45 degrees
    const double scale = mx > max_angle ? max_angle / mx : 1.0;
#pragma unroll
    for (int i = 0; i < n; ++i) q_ik[i] = e.q[i] + (float)(scale * b[i]);
}

#endif
#if KK_ROLL_DYN
// Mass matrix (lower triangle, M[i][j], j <= i) by the composite-rigid-body algorithm and bias torques
// (gravity, velocity products, Bullet link damping) by recursive Newton-Euler, both in world coordinates
// about the world origin: sub-tree quantities accumulate by plain addition.  Rolled per-body loops.
KK_DEV void kuka_dynamics(const KukaParams& P, const KukaEnv& e, const KukaKin& k, float (&M)[KK_NB][KK_NB], float* bias) {
    float qdl[KK_NB];
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) qdl[i] = e.qd[i];
    f3 nn[KK_NB], ff[KK_NB];          // body wrenches about the origin, then sub-tree sums
    float cm[KK_NB]; f3 ch[KK_NB]; float cI[KK_NB][6];  // composite mass, first moment, inertia about the origin
    // ---- RNEA forward pass + body wrenches (running parent state; the second finger restarts from body 7) ----
    f3 w = mk3(0.f, 0.f, 0.f), vO = w, aw = w, av = mk3(0.f, 0.f, -P.gz);  // gravity as a fictitious base acceleration
    f3 w7 = w, vO7 = w, aw7 = w, av7 = av;
#pragma unroll 1
    for (int i = 0; i < KK_NB; ++i) {
        if (i == 10) { w = w7; vO = vO7; aw = aw7; av = av7; }
        const float qd = qdl[i];
        const f3 ai = k.a[i], pvi = k.pv[i];
        const f3 awn = aw + qd * cross3(w, ai);
        const f3 avn = av + qd * (cross3(w, pvi) + cross3(vO, ai));
        w = w + qd * ai;
        vO = vO + qd * pvi;
        aw = awn; av = avn;
        if (i == 7) { w7 = w; vO7 = vO; aw7 = aw; av7 = av; }
        // spatial inertia about the origin: m, h = m c, I_O = Iw + m (|c|^2 1 - c c^T)
        const float m = P.mass[i];
        const f3 c = k.c[i];
        const f3 h = m * c;
        float Iw[6], IO[6];
#pragma unroll
        for (int t = 0; t < 6; ++t) Iw[t] = k.Iw[i][t];
        IO[0] = Iw[0] + m * (c.y * c.y + c.z * c.z);
        IO[1] = Iw[1] - m * c.x * c.y;
        IO[2] = Iw[2] - m * c.x * c.z;
        IO[3] = Iw[3] + m * (c.x * c.x + c.z * c.z);
        IO[4] = Iw[4] - m * c.y * c.z;
        IO[5] = Iw[5] + m * (c.x * c.x + c.y * c.y);
        cm[i] = m; ch[i] = h;
#pragma unroll
        for (int t = 0; t < 6; ++t) cI[i][t] = IO[t];
        const f3 Lv = symv(IO, w) + cross3(h, vO);
        const f3 Pv = m * vO + cross3(w, h);
        const f3 La = symv(IO, aw) + cross3(h, av);
        const f3 Pa = m * av + cross3(aw, h);
        f3 n = La + cross3(w, Lv) + cross3(vO, Pv);
        f3 f = Pa + cross3(w, Pv);
        // btMultiBody link damping (linear/angular 0.04, K1 = K2): resisting wrench added to the bias
        const f3 vc = vO + cross3(w, c);
        const f3 F = (P.kl * m * (1.0f + norm3(vc))) * vc;
        const f3 T = (P.ka * (1.0f + norm3(w))) * symv(Iw, w);
        nn[i] = n + T + cross3(c, F);
        ff[i] = f + F;
    }
    // ---- backward pass: bias_i = s_i . (wrench of the sub-tree); CRBA: M_ij = s_i . (I^c_j s_j), i ancestor-or-self of j ----
#pragma unroll 1
    for (int j = KK_NB - 1; j >= 0; --j) {
        const f3 aj = k.a[j], pvj = k.pv[j];
        const f3 nj = nn[j], fj = ff[j];
        bias[j] = dot3(aj, nj) + dot3(pvj, fj);
        const float mj = cm[j]; const f3 hj = ch[j];
        float Ij[6];
#pragma unroll
        for (int t = 0; t < 6; ++t) Ij[t] = cI[j][t];
        const f3 Pm = mj * pvj + cross3(aj, hj);              // linear momentum of the composite under unit joint rate
        const f3 Lm = symv(Ij, aj) + cross3(hj, pvj);         // angular momentum about the origin
        for (int i = 0; i <= j; ++i) M[j][i] = 0.f;
        for (int i = j; i >= 0; i = KK_PAR(i)) M[j][i] = dot3(k.a[i], Lm) + dot3(k.pv[i], Pm);
        const int pa = KK_PAR(j);
        if (pa >= 0) {
            nn[pa] = nn[pa] + nj; ff[pa] = ff[pa] + fj;
            cm[pa] += mj; ch[pa] = ch[pa] + hj;
#pragma unroll
            for (int t = 0; t < 6; ++t) cI[pa][t] += Ij[t];
        }
    }
}

#else
// Mass matrix (lower triangle, m[i][j], j <= i) by the composite-rigid-body algorithm and bias torques
// (gravity, velocity products, Bullet link damping) by recursive Newton-Euler, both in world coordinates
// about the world origin: sub-tree quantities accumulate by plain addition.
KK_DEV void kuka_dynamics(const KukaParams& P, const KukaEnv& e, const KukaKin& k, float (&M)[KK_NB][KK_NB], float* bias) {
    f3 pv[KK_NB];  // linear part of the joint motion vector about the origin: p x a
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) pv[i] = cross3(k.p[i], k.a[i]);

    // ---- RNEA forward pass + body wrenches ----
    f3 w[KK_NB], vO[KK_NB], aw[KK_NB], av[KK_NB], nn[KK_NB], ff[KK_NB];
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) {
        const int pa = KK_PAR(i);
        const f3 wp = pa < 0 ? mk3(0.f, 0.f, 0.f) : w[pa];
        const f3 vp = pa < 0 ? mk3(0.f, 0.f, 0.f) : vO[pa];
        const f3 awp = pa < 0 ? mk3(0.f, 0.f, 0.f) : aw[pa];
        const f3 avp = pa < 0 ? mk3(0.f, 0.f, -P.gz) : av[pa];  // gravity as a fictitious base acceleration
        const float qd = e.qd[i];
        w[i] = wp + qd * k.a[i];
        vO[i] = vp + qd * pv[i];
        aw[i] = awp + qd * cross3(wp, k.a[i]);
        av[i] = avp + qd * (cross3(wp, pv[i]) + cross3(vp, k.a[i]));
        // spatial inertia about the origin: m, h = m c, I_O = Iw + m (|c|^2 1 - c c^T)
        const float m = P.mass[i];
        const f3 c = k.c[i];
        const f3 h = m * c;
        float IO[6];
        IO[0] = k.Iw[i][0] + m * (c.y * c.y + c.z * c.z);
        IO[1] = k.Iw[i][1] - m * c.x * c.y;
        IO[2] = k.Iw[i][2] - m * c.x * c.z;
        IO[3] = k.Iw[i][3] + m * (c.x * c.x + c.z * c.z);
        IO[4] = k.Iw[i][4] - m * c.y * c.z;
        IO[5] = k.Iw[i][5] + m * (c.x * c.x + c.y * c.y);
        const f3 Lv = symv(IO, w[i]) + cross3(h, vO[i]);
        const f3 Pv = m * vO[i] + cross3(w[i], h);
        const f3 La = symv(IO, aw[i]) + cross3(h, av[i]);
        const f3 Pa = m * av[i] + cross3(aw[i], h);
        f3 n = La + cross3(w[i], Lv) + cross3(vO[i], Pv);
        f3 f = Pa + cross3(w[i], Pv);
        // btMultiBody link damping (linear/angular 0.04, K1 = K2): resisting wrench added to the bias
        const f3 vc = vO[i] + cross3(w[i], c);
        const f3 F = (P.kl * m * (1.0f + norm3(vc))) * vc;
        const f3 T = (P.ka * (1.0f + norm3(w[i]))) * symv(k.Iw[i], w[i]);
        n = n + T + cross3(c, F);
        f = f + F;
        nn[i] = n; ff[i] = f;
    }
    // ---- RNEA backward pass: bias_i = s_i . (wrench of the sub-tree) ----
#pragma unroll
    for (int i = KK_NB - 1; i >= 0; --i) {
        bias[i] = dot3(k.a[i], nn[i]) + dot3(pv[i], ff[i]);
        const int pa = KK_PAR(i);
        if (pa >= 0) { nn[pa] = nn[pa] + nn[i]; ff[pa] = ff[pa] + ff[i]; }
    }
    // ---- CRBA: composite inertias from the leaves, M_ij = s_i . (I^c_j s_j) for i ancestor-or-self of j ----
    float cm[KK_NB]; f3 ch[KK_NB]; float cI[KK_NB][6];
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) {
        const float m = P.mass[i];
        const f3 c = k.c[i];
        cm[i] = m; ch[i] = m * c;
        cI[i][0] = k.Iw[i][0] + m * (c.y * c.y + c.z * c.z);
        cI[i][1] = k.Iw[i][1] - m * c.x * c.y;
        cI[i][2] = k.Iw[i][2] - m * c.x * c.z;
        cI[i][3] = k.Iw[i][3] + m * (c.x * c.x + c.z * c.z);
        cI[i][4] = k.Iw[i][4] - m * c.y * c.z;
        cI[i][5] = k.Iw[i][5] + m * (c.x * c.x + c.y * c.y);
    }
#pragma unroll
    for (int j = KK_NB - 1; j >= 0; --j) {
        const f3 Pm = cm[j] * pv[j] + cross3(k.a[j], ch[j]);             // linear momentum of the composite
        const f3 Lm = symv(cI[j], k.a[j]) + cross3(ch[j], pv[j]);        // angular momentum about the origin
#pragma unroll
        for (int i = 0; i < KK_NB; ++i) {
            // i ancestor-or-self of j  (chain 0..7 precedes everything; 8 -> 9; 10 -> 11)
            const bool anc = (i == j) || (i <= 7 && i < j) || (i == 8 && j == 9) || (i == 10 && j == 11);
            if (i <= j) {
                if (anc) M[j][i] = dot3(k.a[i], Lm) + dot3(pv[i], Pm);
                else M[j][i] = 0.f;
            }
        }
        const int pa = KK_PAR(j);
        if (pa >= 0) {
            cm[pa] += cm[j]; ch[pa] = ch[pa] + ch[j];
#pragma unroll
            for (int t = 0; t < 6; ++t) cI[pa][t] += cI[j][t];
        }
    }
}

#endif
// In-place: M (lower) -> A = M^-1 (lower triangle valid), via Cholesky and triangular inverse.
// Every loop has a constant trip count and skips the indices outside the triangle with an `if` that folds once the enclosing loops are
// unrolled.  With bounds that depend on an outer index (i = j + 1 .. n) the compiler unrolls the inner loops before the outer ones, cannot
// unroll them fully, and M drops to a 576-byte local-memory array (a local load / store per entry in the once-per-step code).
KK_DEV void kuka_spd_inverse(float (&M)[KK_NB][KK_NB]) {
    constexpr int n = KK_NB;
    float dinv[n];
#pragma unroll
    for (int j = 0; j < n; ++j) {
        float d = M[j][j];
#pragma unroll
        for (int kk = 0; kk < n; ++kk)
            if (kk < j) d = fmaf(-M[j][kk], M[j][kk], d);
        const float inv = rsqrtf(d);
        dinv[j] = inv;
        M[j][j] = d * inv;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            if (i <= j) continue;
            float s = M[i][j];
#pragma unroll
            for (int kk = 0; kk < n; ++kk)
                if (kk < j) s = fmaf(-M[i][kk], M[j][kk], s);
            M[i][j] = s * inv;
        }
    }
    // X = L^-1 (lower), in place column by column
#pragma unroll
    for (int j = 0; j < n; ++j) {
        M[j][j] = dinv[j];
#pragma unroll
        for (int i = 0; i < n; ++i) {
            if (i <= j) continue;
            float s = 0.f;
#pragma unroll
            for (int kk = 0; kk < n; ++kk)
                if (kk >= j && kk < i) s = fmaf(M[i][kk], M[kk][j], s);
            M[i][j] = -s * dinv[i];
        }
    }
    // A = X^T X : A[i][j] = sum_{k >= i} X[k][i] X[k][j]   (i >= j); rows ascending keeps inputs intact
#pragma unroll
    for (int i = 0; i < n; ++i) {
#pragma unroll
        for (int j = 0; j < n; ++j) {
            if (j > i) continue;
            float s = 0.f;
#pragma unroll
            for (int kk = 0; kk < n; ++kk)
                if (kk >= i) s = fmaf(M[kk][i], M[kk][j], s);
            M[i][j] = s;
        }
    }
}

#define KK_A(i, j) ((i) >= (j) ? A[i][j] : A[j][i])

// One applyAction + stepSimulation.  `k`/`ct` hold the kinematics / contacts of the CURRENT configuration
// (computed by the caller with kuka_fk<true>); on return q, qd, qb, qdb are advanced by one time step.
// JOINTS: use_inverse_kinematics = False (action_joints): the 7 arm set-points are given (`q_joints`), no IK (kuka.py:158-161).
// TWOB: Kuka2ButtonGymEnv -- a second button glider (DoF KK_NB + 1) with the same motor / limit rows, right after the first.
// COOP: the env is a group of 4 lanes (kuka_coop.cuh): kinematics, contact manifold, mass-matrix inverse, bias and contact rows come from
// the group's scratch area `sc` (k / ct are unused); every lane of the group runs the row set-up and the sweeps on identical values.
struct KkNoScratch { float dummy; KK_DEV float& operator[](int) const { return const_cast<float&>(dummy); } };
template <bool JOINTS, bool TWOB, bool COOP = false, class SC = KkNoScratch>
KK_DEV void kuka_physics_step(const KukaParams& P, KukaEnv& e, const KukaKin& k, const KukaContacts& ct, bool button_armed, const float* q_joints,
                              const SC& sc = SC(), int u = 0, unsigned gmask = 0u, int nc_coop = 0, unsigned* dbg = nullptr) {
    constexpr int ND = TWOB ? KK_NB + 2 : KK_NB + 1;
    // ---- applyAction: IK + motor set-points (kuka.py:142-187) ----
    float q_ik[7];
    if (JOINTS) {
#pragma unroll
        for (int j = 0; j < 7; ++j) q_ik[j] = q_joints[j];
    } else if constexpr (COOP) {
        KukaKin kk7;            // what the IK reads: axes and origins of the 7 arm joints, rotation of link 6 (static indices: registers)
#pragma unroll
        for (int j = 0; j < 7; ++j) {
            kk7.a[j] = mk3(sc[j * KC_BS + KB_A], sc[j * KC_BS + KB_A + 1], sc[j * KC_BS + KB_A + 2]);
            kk7.p[j] = mk3(sc[j * KC_BS + KB_P], sc[j * KC_BS + KB_P + 1], sc[j * KC_BS + KB_P + 2]);
        }
#pragma unroll
        for (int t = 0; t < 9; ++t) kk7.R6[t] = sc[6 * KC_BS + KB_R + t];
        kuka_ik(P, e, kk7, q_ik);
    } else kuka_ik(P, e, k, q_ik);
    // ---- dynamics ----
    float A[KK_NB][KK_NB], bias[KK_NB];
    if constexpr (COOP) {
#if defined(__CUDACC__)
        __syncwarp(gmask);      // every lane has read link 6's rotation: the wrench phase reuses its storage
        kc_dynamics(sc, P, e.qd, u, gmask);
#endif
#pragma unroll
        for (int i = 0; i < KK_NB; ++i)
#pragma unroll
            for (int j = 0; j <= i; ++j) A[i][j] = sc[KC_OFF_MA + i * KC_MS + j];
        // Cholesky + M^-1 in registers, by every lane: dealt to the 4 lanes through shared memory it was three times slower (12 dependent
        // pivot steps of load -> rsqrt -> scale -> store -> barrier; measured on B200, profiles/r02_kuka_coop_by_function.txt)
        kuka_spd_inverse(A);
        // the bias stays in the scratch area until the inverse is done: the Cholesky does not need it
#pragma unroll
        for (int i = 0; i < KK_NB; ++i) bias[i] = sc[KC_OFF_BIAS + i];
    } else {
#if KK_ROLL_DYN
    {
        float Mloc[KK_NB][KK_NB], bloc[KK_NB];  // thread-local (dynamically indexed by the rolled loops)
        kuka_dynamics(P, e, k, Mloc, bloc);
#pragma unroll
        for (int i = 0; i < KK_NB; ++i) {       // -> registers (static indices only from here on)
            bias[i] = bloc[i];
#pragma unroll
            for (int j = 0; j <= i; ++j) A[i][j] = Mloc[i][j];
        }
    }
#else
    kuka_dynamics(P, e, k, A, bias);
#endif
    kuka_spd_inverse(A);
    }
    float v[ND];
    {
        float rhs[KK_NB];
#pragma unroll
        for (int i = 0; i < KK_NB; ++i) rhs[i] = -P.damping[i] * e.qd[i] - bias[i];
#pragma unroll
        for (int i = 0; i < KK_NB; ++i) {
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < KK_NB; ++j) s = fmaf(KK_A(i, j), rhs[j], s);
            v[i] = fmaf(P.dt, s, e.qd[i]);
        }
        const float vb = e.qdb;
        v[KK_NB] = fmaf(P.dt, P.gz - P.kl * vb * (1.0f + fabsf(vb)), vb);
        if (TWOB) { const float vb2 = e.qdb2; v[ND - 1] = fmaf(P.dt, P.gz - P.kl * vb2 * (1.0f + fabsf(vb2)), vb2); }
    }
    // ---- motor rows: target velocity, impulse bound (btMultiBodyJointMotor) ----
    float tgt[KK_NB], lam[KK_NB], invd[KK_NB];
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) {
        const float qdes = (P.tmode[i] == 0 && i < 7) ? q_ik[i < 7 ? i : 0] : 0.f;
        float t = fmaf(P.kp_dt[i], qdes - e.q[i], v[i]) - P.kd[i] * v[i];
        if (P.maxvel[i] > 0.f) t = fminf(fmaxf(t, -P.maxvel[i]), P.maxvel[i]);
        tgt[i] = t; lam[i] = 0.f; invd[i] = 1.0f / A[i][i];
    }
    float b_tgt, b_hi, b_lam = 0.f;
    if (button_armed) { b_tgt = fmaf(P.btn_kp_dt, P.btn_target - e.qb, v[KK_NB]) - P.btn_kd * v[KK_NB]; b_hi = P.btn_maximp; }
    else { b_tgt = 0.f; b_hi = P.btn_idle_imp; }
    const float b_invd = 1.0f / P.btn_minv;
    float b2_tgt = 0.f, b2_lam = 0.f;   // second button motor: same command as the first (kuka_2button_gym_env.py:137-138)
    if (TWOB && button_armed) b2_tgt = fmaf(P.btn_kp_dt, P.btn_target - e.qb2, v[ND - 1]) - P.btn_kd * v[ND - 1];
    // ---- limit rows (active while the joint is on / beyond the limit) ----
    const bool bl_lo = (e.qb - P.gl_lo) <= P.lim_eps, bl_hi = (P.gl_hi - e.qb) <= P.lim_eps;
    const float bl_lo_t = -P.erp * (e.qb - P.gl_lo) * P.inv_dt, bl_hi_t = -P.erp * (P.gl_hi - e.qb) * P.inv_dt;
    float bl_lo_lam = 0.f, bl_hi_lam = 0.f;
    const bool b2l_lo = TWOB && (e.qb2 - P.gl_lo) <= P.lim_eps, b2l_hi = TWOB && (P.gl_hi - e.qb2) <= P.lim_eps;
    const float b2l_lo_t = TWOB ? -P.erp * (e.qb2 - P.gl_lo) * P.inv_dt : 0.f, b2l_hi_t = TWOB ? -P.erp * (P.gl_hi - e.qb2) * P.inv_dt : 0.f;
    float b2l_lo_lam = 0.f, b2l_hi_lam = 0.f;
    unsigned lim_lo_mask = 0u, lim_hi_mask = 0u;
    float lim_lam_lo[KK_NB], lim_lam_hi[KK_NB];
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) {
        if ((e.q[i] - P.lower[i]) <= P.lim_eps) lim_lo_mask |= 1u << i;
        if ((P.upper[i] - e.q[i]) <= P.lim_eps) lim_hi_mask |= 1u << i;
        lim_lam_lo[i] = 0.f; lim_lam_hi[i] = 0.f;
    }
    // ---- the SCALED system the sweeps run on (round 2): impulses as lam' = (lam + max_imp) / sigma in [0, 1] with sigma = 2 max_imp, residuals
    //      as v'_j = sigma_j (v_j - target_j), M^-1 as sigma_i sigma_j A_ij (symmetric: 78 registers).  The projection of a motor impulse onto
    //      [-max_imp, +max_imp] is then the .SAT modifier of the FFMA that produces it: the loop-carried path of a row is FFMA.SAT -> FADD (8
    //      cycles) instead of FFMA -> FMNMX -> FMNMX -> FADD (18).  The button DoF (KK_NB, and ND - 1 of the second button) stay unscaled. ----
    float cs[KK_NB];
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) {
        cs[i] = invd[i] * P.sat_isig2[i];                  // 1 / (sigma_i^2 A_ii)
        v[i] = (v[i] - tgt[i]) * P.sat_sig[i];
        lam[i] = 0.5f;                                     // lam = 0
    }
    // ---- contact rows: J, W = M^-1 J^T (unscaled A), 1/D, target; two friction rows each.  Stored for the scaled system:
    //      J'_j = J_j / sigma_j and W'_j = sigma_j W_j on the 12 arm DoF, target' = target - J . tgt.  One row = KK_ROWW words: J'[0..13],
    //      1/D, target', W'[16..29] -- 16-byte groups, so that a row is eight 128-bit loads from the scratch area (COOP) or local memory. ----
    const int nc = COOP ? nc_coop : ct.n;
    alignas(16) float cR[COOP ? 1 : 3 * KK_MAXC][KK_ROWW];
    float c_lam[3 * KK_MAXC];
    if constexpr (COOP) {
        if (nc > 0) {           // rows dealt to the 4 lanes, through the scratch area
#if defined(__CUDACC__)
            __syncwarp(gmask);
            kc_ph_rows<TWOB, true>(sc, P, A, nc, u, tgt);
            __syncwarp(gmask);
#endif
            for (int r = 0; r < 3 * nc; ++r) c_lam[r] = 0.f;
        }
    } else
    if (nc > 0) {
        for (int r = 0; r < 3 * nc; ++r) {
            const int c = r < nc ? r : (r - nc) >> 1;
            f3 dir = ct.nrm[c];
            if (r >= nc) {  // btPlaneSpace1 tangents
                const f3 n = ct.nrm[c];
                f3 t1, t2;
                if (fabsf(n.z) > 0.70710678f) {
                    const float a = n.y * n.y + n.z * n.z, kk = rsqrtf(a);
                    t1 = mk3(0.f, -n.z * kk, n.y * kk); t2 = mk3(a * kk, -n.x * t1.z, n.x * t1.y);
                } else {
                    const float a = n.x * n.x + n.y * n.y, kk = rsqrtf(a);
                    t1 = mk3(-n.y * kk, n.x * kk, 0.f); t2 = mk3(-n.z * t1.y, n.z * t1.x, a * kk);
                }
                dir = ((r - nc) & 1) ? t2 : t1;
            }
            const int body = ct.body[c];
            float J[KK_NB];
#pragma unroll
            for (int j = 0; j < KK_NB; ++j) {
                const bool anc = (j == body) || (j <= 7 && j < body) || (j == 8 && body == 9) || (j == 10 && body == 11);
                J[j] = anc ? dot3(dir, cross3(k.a[j], ct.pt[c] - k.p[j])) : 0.f;
            }
            float* row = cR[COOP ? 0 : r];
            float D = 0.f, off = 0.f;
#pragma unroll
            for (int i = 0; i < KK_NB; ++i) {
                float w = 0.f;
#pragma unroll
                for (int j = 0; j < KK_NB; ++j) w = fmaf(KK_A(i, j), J[j], w);
                D = fmaf(J[i], w, D); off = fmaf(J[i], tgt[i], off);
                row[KK_ROW_J + i] = J[i] * P.sat_isig[i];
                row[KK_ROW_W + i] = w * P.sat_sig[i];
            }
            const float jb = ct.shape[c] == 1 ? -dir.z : 0.f, jb2 = TWOB && ct.shape[c] == 3 ? -dir.z : 0.f;
            row[KK_ROW_J + KK_NB] = jb; row[KK_ROW_W + KK_NB] = jb * P.btn_minv;
            row[KK_ROW_J + KK_NB + 1] = jb2; row[KK_ROW_W + KK_NB + 1] = jb2 * P.btn_minv;
            D = fmaf(jb, jb * P.btn_minv, D);
            if (TWOB) D = fmaf(jb2, jb2 * P.btn_minv, D);
            row[KK_ROW_INVD] = 1.0f / D;
            c_lam[r] = 0.f;
            const float pen = ct.dist[c];
            row[KK_ROW_TGT] = (r < nc ? (pen > 0.f ? -pen * P.inv_dt : -P.erp * pen * P.inv_dt) : 0.f) - off;
        }
    }
    // the scaled matrix (after the rows: W = M^-1 J^T uses the unscaled one)
#pragma unroll
    for (int i = 0; i < KK_NB; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) A[i][j] *= P.sat_ss[i * (i + 1) / 2 + j];
    // J' . v of one stored row: four independent partial sums (the loop-carried path of a contact row is 4 FFMA + 2 FADD, not 14 FFMA)
#define KK_ROW_PTR(r) (COOP ? &sc[KC_OFF_ROWS + (r) * KC_RS] : cR[COOP ? 0 : (r)])
#define KK_ROW_LOAD4(dst, ptr, base)                                                                                   \
    _Pragma("unroll")                                                                                                  \
    for (int q4 = 0; q4 < 4; ++q4) {                                                                                   \
        const kk_f4 t4 = *reinterpret_cast<const kk_f4*>((ptr) + (base) + 4 * q4);                                   \
        dst[4 * q4] = t4.x; dst[4 * q4 + 1] = t4.y; dst[4 * q4 + 2] = t4.z; dst[4 * q4 + 3] = t4.w;                    \
    }
#define KK_ROW_DOT(Jr, out)                                                                                            \
    {                                                                                                                  \
        float p0 = Jr[0] * v[0], p1 = Jr[1] * v[1], p2 = Jr[2] * v[2], p3 = Jr[3] * v[3];                              \
        p0 = fmaf(Jr[4], v[4], p0); p1 = fmaf(Jr[5], v[5], p1); p2 = fmaf(Jr[6], v[6], p2); p3 = fmaf(Jr[7], v[7], p3); \
        p0 = fmaf(Jr[8], v[8], p0); p1 = fmaf(Jr[9], v[9], p1); p2 = fmaf(Jr[10], v[10], p2); p3 = fmaf(Jr[11], v[11], p3); \
        p0 = fmaf(Jr[12], v[12], p0);                                                                                  \
        if (TWOB) p1 = fmaf(Jr[13], v[ND - 1], p1);                                                                    \
        out = (p0 + p1) + (p2 + p3);                                                                                   \
    }
    // ---- projected Gauss-Seidel: row order = motors (button first), limits (button first), contact normals, friction ----
    // Button rows are made branch-free: an inactive limit row gets the bound [0, 0] (an exact no-op).
    const float bl_lo_hi = bl_lo ? P.lim_maximp : 0.f, bl_hi_hi = bl_hi ? P.lim_maximp : 0.f;
    const float b2l_lo_hi = b2l_lo ? P.lim_maximp : 0.f, b2l_hi_hi = b2l_hi ? P.lim_maximp : 0.f;
    // the second button's rows (motor; lower / upper limit): an independent 1-DoF chain like the first one's
#define KK_BUTTON2_MOTOR()                                                                                             \
    if (TWOB) {                                                                                                        \
        const float s2 = fminf(fmaxf(fmaf(b2_tgt - v[ND - 1], b_invd, b2_lam), -b_hi), b_hi);                          \
        v[ND - 1] = fmaf(P.btn_minv, s2 - b2_lam, v[ND - 1]); b2_lam = s2;                                             \
    }
#define KK_BUTTON2_LIMITS()                                                                                            \
    if (TWOB) {                                                                                                        \
        float s2 = fminf(fmaxf(fmaf(b2l_lo_t - v[ND - 1], b_invd, b2l_lo_lam), 0.f), b2l_lo_hi);                       \
        v[ND - 1] = fmaf(P.btn_minv, s2 - b2l_lo_lam, v[ND - 1]); b2l_lo_lam = s2;                                     \
        s2 = fminf(fmaxf(fmaf(b2l_hi_t + v[ND - 1], b_invd, b2l_hi_lam), 0.f), b2l_hi_hi);                             \
        v[ND - 1] = fmaf(-P.btn_minv, s2 - b2l_hi_lam, v[ND - 1]); b2l_hi_lam = s2;                                    \
    }
    // one arm motor row of the scaled system + its update of the 12 residuals
#define KK_MOTOR_ROWS()                                                                                                \
    _Pragma("unroll")                                                                                                  \
    for (int i = 0; i < KK_NB; ++i) {                                                                                  \
        const float s = __saturatef(fmaf(-cs[i], v[i], lam[i]));                                                       \
        const float d = s - lam[i];                                                                                    \
        lam[i] += d;            /* in place: no register rename, no MOV at the loop end; equals s whenever s - lam is exact */ \
        KK_PROBE_D(d)                                                                                                  \
        _Pragma("unroll")                                                                                              \
        for (int j = 0; j < KK_NB; ++j) v[j] = fmaf(KK_A(j, i), d, v[j]);                                              \
    }
    // the same with the contact watch folded in: J'_c . v' of the (up to 4) watched normal rows is carried incrementally -- a motor row's step d
    // moves it by W'_ci d (W' = A' J'^T: the column the general loop would apply) -- as 4 independent FFMA per row off the loop-carried path,
    // fed by one 128-bit load of the watch matrix; recomputing the 14-term dot per contact after every sweep cost ~100 cycles per contact and
    // sweep on the single resident warp (profiles/r02_lockstep_slot_timing_before.txt: 66 / 75 / 82 / 90 us per step with 1 / 2 / 3 / 4 contacts, 49 without)
#define KK_MOTOR_ROWS_WATCH()                                                                                          \
    _Pragma("unroll")                                                                                                  \
    for (int i = 0; i < KK_NB; ++i) {                                                                                  \
        const kk_f4 w4 = *reinterpret_cast<const kk_f4*>(wt + 4 * i);                                                  \
        const float s = __saturatef(fmaf(-cs[i], v[i], lam[i]));                                                       \
        const float d = s - lam[i];                                                                                    \
        lam[i] += d;                                                                                                   \
        KK_PROBE_D(d)                                                                                                  \
        _Pragma("unroll")                                                                                              \
        for (int j = 0; j < KK_NB; ++j) v[j] = fmaf(KK_A(j, i), d, v[j]);                                              \
        wjv[0] = fmaf(w4.x, d, wjv[0]); wjv[1] = fmaf(w4.y, d, wjv[1]); wjv[2] = fmaf(w4.z, d, wjv[2]); wjv[3] = fmaf(w4.w, d, wjv[3]); \
    }
    int it0 = 0;                 // first sweep the general loop still has to do
#if defined(KK_TIMING)
    bool kk_probe_any = false; int kk_probe_sweep = 0, kk_probe_conv = 0;
#endif
    bool resume_mid_sweep = false;  // the fast loop already ran the motor + button rows of sweep it0
    if ((lim_lo_mask | lim_hi_mask) == 0u) {
        // FAST LOOP (no arm joint on a limit): straight-line sweep, registers only.  Contact rows of the manifold are
        // WATCHED: while every normal row is separating (lam = 0 and J v >= target) it and its friction rows are exact
        // no-ops; the first time one would activate, the solve continues in the general loop from that very row.
        // loop invariants of the button rows in vector registers (opaque copies: no uniform-register / constant-bank reloads inside the sweep)
        float bminv, nbminv, lo_hi, hi_hi, lo_t, hi_t;
        asm volatile("mov.f32 %0, %1;" : "=f"(bminv) : "f"(P.btn_minv));
        asm volatile("mov.f32 %0, %1;" : "=f"(nbminv) : "f"(-P.btn_minv));
        asm volatile("mov.f32 %0, %1;" : "=f"(lo_hi) : "f"(bl_lo_hi));
        asm volatile("mov.f32 %0, %1;" : "=f"(hi_hi) : "f"(bl_hi_hi));
        asm volatile("mov.f32 %0, %1;" : "=f"(lo_t) : "f"(bl_lo_t));
        asm volatile("mov.f32 %0, %1;" : "=f"(hi_t) : "f"(bl_hi_t));
        bool act = false;        // a watched contact row would activate in sweep `it - 1`
        bool more = true;
        int it = 0;
        // one sweep over the button rows and the 12 motor rows
#define KK_SWEEP_BUTTONS()                                                                                               \
                {   /* button motor + the two limit rows (an independent 1-DoF chain, fills issue slots) */              \
                    float s = fminf(fmaxf(fmaf(b_tgt - v[KK_NB], b_invd, b_lam), -b_hi), b_hi);                          \
                    v[KK_NB] = fmaf(bminv, s - b_lam, v[KK_NB]); b_lam = s;                                              \
                    s = fminf(fmaxf(fmaf(lo_t - v[KK_NB], b_invd, bl_lo_lam), 0.f), lo_hi);                              \
                    v[KK_NB] = fmaf(bminv, s - bl_lo_lam, v[KK_NB]); bl_lo_lam = s;                                      \
                    s = fminf(fmaxf(fmaf(hi_t + v[KK_NB], b_invd, bl_hi_lam), 0.f), hi_hi);                              \
                    v[KK_NB] = fmaf(nbminv, s - bl_hi_lam, v[KK_NB]); bl_hi_lam = s;                                     \
                }                                                                                                        \
                KK_BUTTON2_MOTOR() KK_BUTTON2_LIMITS()
        if (P.iters > 0) {
            int left = P.iters;
            asm volatile("mov.u32 %0, %0;" : "+r"(left));
#if defined(__CUDA_ARCH__) && KK_SWEEP_TIGHT
            // 93 % of the warp-sweeps watch no contact in ANY lane (profiles/r02): those run a loop that is nothing but the rows and one
            // back edge.  Warp-uniform choice: no divergence.
            const bool quiet = __all_sync(__activemask(), nc == 0);
#else
            const bool quiet = false;
#endif
            if (quiet) {
                constexpr int tight_unroll = KK_TIGHT_UNROLL;
#pragma unroll tight_unroll
                do { KK_SWEEP_BUTTONS() KK_MOTOR_ROWS() KK_PROBE_SWEEP() } while (--left > 0);
                it = P.iters;
            } else if constexpr (!COOP) {
                // one thread per env (32 envs per warp, batches >= 16 384): nearly every warp holds SOME env with a candidate contact, and every
                // lane pays for what one lane does -- so the watched rows are re-tested with their 14-term dot after each sweep by the lanes that
                // have any (the incremental form below made every lane carry four rows: 405 -> 246 M env-steps/s at 32 768 envs)
                constexpr int sweep_unroll = KK_SWEEP_UNROLL;
#pragma unroll sweep_unroll
                do {
                    KK_SWEEP_BUTTONS()
                    KK_MOTOR_ROWS()
                    KK_PROBE_SWEEP()
                    ++it;
                    more = --left > 0;
                    if (nc > 0) {
#pragma unroll 1
                        for (int c = 0; c < nc; ++c) {
                            const float* row = KK_ROW_PTR(c);
                            float Jr[16], jv;
                            KK_ROW_LOAD4(Jr, row, KK_ROW_J)
                            KK_ROW_DOT(Jr, jv)
                            act = act | (Jr[KK_ROW_TGT] - jv > 0.f);
                        }
                        if (act) more = false;
                    }
                } while (more);
            } else {
                // four lanes per env (<= 8 envs per warp): watched normal rows c < nc (slots c >= nc: zero column, threshold -inf -- they never
                // fire): arm part of J' . v' carried in wjv, the button DoF added when the row is tested
                const float* wt = &sc[KC_OFF_WT];
                float wjv[4], wthr[4], wjb[4], wjb2[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    wjv[c] = 0.f; wthr[c] = -1e30f; wjb[c] = 0.f; wjb2[c] = 0.f;
                    if (c < nc) {
                        const float* row = KK_ROW_PTR(c);
                        float Jr[16];
                        KK_ROW_LOAD4(Jr, row, KK_ROW_J)
                        float p0 = Jr[0] * v[0], p1 = Jr[1] * v[1], p2 = Jr[2] * v[2], p3 = Jr[3] * v[3];
                        p0 = fmaf(Jr[4], v[4], p0); p1 = fmaf(Jr[5], v[5], p1); p2 = fmaf(Jr[6], v[6], p2); p3 = fmaf(Jr[7], v[7], p3);
                        p0 = fmaf(Jr[8], v[8], p0); p1 = fmaf(Jr[9], v[9], p1); p2 = fmaf(Jr[10], v[10], p2); p3 = fmaf(Jr[11], v[11], p3);
                        wjv[c] = (p0 + p1) + (p2 + p3);
                        wthr[c] = Jr[KK_ROW_TGT]; wjb[c] = Jr[KK_NB]; wjb2[c] = Jr[KK_NB + 1];
                    }
                }
                if (nc == 0) {           // a quiet env in a warp that watches: its watch matrix was not written this step
#pragma unroll
                    for (int i = 0; i < KK_NB; ++i) sc[KC_OFF_WT + 4 * i + u] = 0.f;
#if defined(__CUDACC__)
                    __syncwarp(gmask);
#endif
                }
                constexpr int sweep_unroll = KK_SWEEP_UNROLL;
#pragma unroll sweep_unroll
                do {
                    KK_SWEEP_BUTTONS()
                    KK_MOTOR_ROWS_WATCH()
                    KK_PROBE_SWEEP()
                    ++it;
                    more = --left > 0;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float jv = fmaf(wjb[c], v[KK_NB], wjv[c]);
                        if (TWOB) jv = fmaf(wjb2[c], v[ND - 1], jv);
                        act = act | (wthr[c] - jv > 0.f);
                    }
                    if (act) more = false;
                } while (more);
            }
        }
#undef KK_SWEEP_BUTTONS
        if (act) { it0 = it - 1; resume_mid_sweep = true; } else it0 = it;
#ifdef KK_TIMING
        if (dbg && nc > 0) *dbg |= 1u;
#endif
    }
#ifdef KK_TIMING
    if (dbg) *dbg |= ((unsigned)kk_probe_conv & 255u) << 24;
    if (dbg) { *dbg |= ((unsigned)nc & 15u) << 2; if (lim_lo_mask | lim_hi_mask) *dbg |= 64u; if (it0 < P.iters) *dbg |= 2u | ((unsigned)(P.iters - it0) & 255u) << 8; }
#endif
    if (it0 < P.iters) {
        // GENERAL LOOP (a joint on its limit and / or an active contact): same row order, same scaled system.
#pragma unroll 1
        for (int it = it0; it < P.iters; ++it) {
            if (!resume_mid_sweep) {
            {   // button motor
                const float s = fminf(fmaxf(fmaf(b_tgt - v[KK_NB], b_invd, b_lam), -b_hi), b_hi);
                v[KK_NB] = fmaf(P.btn_minv, s - b_lam, v[KK_NB]); b_lam = s;
            }
            KK_BUTTON2_MOTOR()
            KK_MOTOR_ROWS()
            {   // button limits
                float s = fminf(fmaxf(fmaf(bl_lo_t - v[KK_NB], b_invd, bl_lo_lam), 0.f), bl_lo_hi);
                v[KK_NB] = fmaf(P.btn_minv, s - bl_lo_lam, v[KK_NB]); bl_lo_lam = s;
                s = fminf(fmaxf(fmaf(bl_hi_t + v[KK_NB], b_invd, bl_hi_lam), 0.f), bl_hi_hi);
                v[KK_NB] = fmaf(-P.btn_minv, s - bl_hi_lam, v[KK_NB]); bl_hi_lam = s;
            }
            KK_BUTTON2_LIMITS()
            }
            resume_mid_sweep = false;
            if (lim_lo_mask | lim_hi_mask) {
                // arm joint limits, J = +-e_i.  In the scaled variables v_i = v'_i / sigma_i + tgt_i, and an impulse step d moves the residuals
                // by sigma_j A_ji d = A'_ji (d / sigma_i).
#pragma unroll
                for (int i = 0; i < KK_NB; ++i) {
                    if (lim_lo_mask & (1u << i)) {  // J = +e_i
                        const float t = -P.erp * (e.q[i] - P.lower[i]) * P.inv_dt;
                        const float s = fminf(fmaxf(fmaf(-invd[i] * P.sat_isig[i], v[i], fmaf(t - tgt[i], invd[i], lim_lam_lo[i])), 0.f), P.lim_maximp);
                        const float d = (s - lim_lam_lo[i]) * P.sat_isig[i]; lim_lam_lo[i] = s;
#pragma unroll
                        for (int j = 0; j < KK_NB; ++j) v[j] = fmaf(KK_A(j, i), d, v[j]);
                    }
                    if (lim_hi_mask & (1u << i)) {  // J = -e_i
                        const float t = -P.erp * (P.upper[i] - e.q[i]) * P.inv_dt;
                        const float s = fminf(fmaxf(fmaf(invd[i] * P.sat_isig[i], v[i], fmaf(t + tgt[i], invd[i], lim_lam_hi[i])), 0.f), P.lim_maximp);
                        const float d = (s - lim_lam_hi[i]) * P.sat_isig[i]; lim_lam_hi[i] = s;
#pragma unroll
                        for (int j = 0; j < KK_NB; ++j) v[j] = fmaf(-KK_A(j, i), d, v[j]);
                    }
                }
            }
#pragma unroll 1
            for (int r = 0; r < 3 * nc; ++r) {
                float lo = 0.f, hi = 1e10f;
                if (r >= nc) {
                    hi = P.mu * c_lam[(r - nc) >> 1]; lo = -hi;
                    if (hi == 0.f && c_lam[r] == 0.f) continue;  // friction under a zero normal impulse: bounds [0, 0], an exact no-op
                }
                const float* row = KK_ROW_PTR(r);
                float Jr[16], Wr[16], jv;
                KK_ROW_LOAD4(Jr, row, KK_ROW_J)
                KK_ROW_LOAD4(Wr, row, KK_ROW_W)
                KK_ROW_DOT(Jr, jv)
                const float s = fminf(fmaxf(fmaf(Jr[KK_ROW_TGT] - jv, Jr[KK_ROW_INVD], c_lam[r]), lo), hi);
                const float d = s - c_lam[r];
                if (d == 0.f) continue;       // inactive (separating) contact: nothing to apply
                c_lam[r] = s;
#pragma unroll
                for (int j = 0; j < KK_NB + 1; ++j) v[j] = fmaf(Wr[j], d, v[j]);
                if (TWOB) v[ND - 1] = fmaf(Wr[KK_NB + 1], d, v[ND - 1]);
            }
        }
    }
#undef KK_MOTOR_ROWS
#undef KK_MOTOR_ROWS_WATCH
#undef KK_ROW_PTR
#undef KK_ROW_LOAD4
#undef KK_ROW_DOT
    // back to velocities
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) v[i] = fmaf(v[i], P.sat_isig[i], tgt[i]);
    // ---- semi-implicit Euler ----
#pragma unroll
    for (int i = 0; i < KK_NB; ++i) { e.qd[i] = v[i]; e.q[i] = fmaf(P.dt, v[i], e.q[i]); }
    e.qdb = v[KK_NB]; e.qb = fmaf(P.dt, v[KK_NB], e.qb);
    if (TWOB) { e.qdb2 = v[ND - 1]; e.qb2 = fmaf(P.dt, v[ND - 1], e.qb2); }
}
