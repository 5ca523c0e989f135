// On-device trot gait generator (wbc_gait_init, wbc_gait_step): per robot, turns a velocity command, the robot's state and the
// contact plant's flags into the contact mode and the six desired-trajectory arrays of wbc_inputs, so that
// gait_step -> wbc_cycle -> contact plant is a chain of device launches.  The law is DESIGN.md 4.8; in short, per step:
//   1. touchdown: in a swing phase past s = (tick+1)/Nw > 0.5, both swing feet in contact (previous plant step) -> landed = 1;
//   2. lift-off (tick 0 of a swing phase): p0 = the swing feet now, p1 = their touchdown targets (gait_target);
//   3. the reference velocity v_ref = (vx, vy heading frame, omega) ramps toward the command, |dv_xy| <= acc_lin dt, |dw| <= acc_yaw dt;
//   4. yaw_ref += omega dt, xy_ref += R_z(yaw_ref) v dt, clamped to a disc of radius leash around the measured CoM; z_ref is the
//      captured clearance above the ground at xy_ref;
//   5. emit mode, com_des_* and the swing curve p0 + (p1 - p0) sigma(s) + z h sin^2(pi s) with its exact time derivatives;
//   6. advance tick / phase (0 stance, 1 swing{BR,FL}, 2 stance, 3 swing{BL,FR}).
// Positions only: the kinematics helper below is the position part of front_dynamics, not a call to it.
#pragma once
#include <math.h>

#include "wbc_front.cuh"

namespace wbc {

struct GaitParams {        // wbc_gait_params
    int ns, nw;            // stance and swing phase lengths (control cycles)
    double step_height, k_v, max_step, acc_lin, acc_yaw, leash;
};

struct GaitIO {
    const double *base_pos, *base_rot, *base_rpy, *base_vel, *q;   // plant state, SoA [k][ld]
    const double* cmd;         // [3][ld] (vx, vy heading frame, omega) or nullptr (0)
    const int* contact;        // [4][ld] or nullptr (no touchdown)
    const double *terrain, *plane_d;   // [40][ld] or nullptr (flat ground z = 0); [4][ld] or nullptr (0)
    const int* k0;             // gait_init: [ld] start offsets or nullptr (0)
    int *phase, *tick, *landed;          // gait state [ld]
    double *com_ref, *v_ref, *liftoff, *target, *offset;   // gait state [4], [3], [6], [6], [8] x [ld]
    int* mode;                 // [ld]
    double* des[6];            // com_des_pos, com_des_vel, com_des_acc, sw_des_pos, sw_des_vel, sw_des_acc, [6][out_ld]
    long out_ld;
    int* status;               // [ld] or nullptr
    long ld;
};

constexpr double GAIT_TOUCHDOWN_S = 0.5;     // a swing can end by touchdown only past this fraction of its phase
constexpr int GAIT_ST_BAD_MODE = -20;        // WBC_ST_BAD_MODE: phase outside 0..3 or tick outside the phase
constexpr int GAIT_ST_NONFINITE = -21;       // WBC_ST_NONFINITE
constexpr int GAIT_ST_BAD_TERRAIN = -24;     // WBC_ST_BAD_TERRAIN

struct GaitKin {
    V3 com;          // whole-body CoM
    V3 hip[4];       // hip (roll-joint) points, stacked foot order BR, BL, FL, FR
    V3 foot[4];      // foot points, stacked order
};

// Positions of front_dynamics' kinematic chain: base at p with rotation R, joint angles q (canonical DoF order).
WBC_DEVFN inline void gait_kinematics(const V3& p, const M3& R, const double* q, GaitKin& K)
{
    using namespace dogbot;
    V3 mr = v3(0, 0, 0);
    for (int leg = 0; leg < 4; leg++) {
        M3 Rp = R;
        V3 pp = v3(0, 0, 0);
        for (int k = 0; k < 3; k++) {
            const V3 org = v3(kJointOrigin[leg][k][0], kJointOrigin[leg][k][1], kJointOrigin[leg][k][2]);
            const V3 ax = v3(kJointAxis[leg][k][0], kJointAxis[leg][k][1], kJointAxis[leg][k][2]);
            const V3 pj = pp + mul(Rp, org);
            const M3 Rk = mul(Rp, axis_rotation(ax, q[dof_index(leg, k)]));
            mr = mr + kLinkMass[leg][k] * (pj + mul(Rk, v3(kLinkCom[leg][k][0], kLinkCom[leg][k][1], kLinkCom[leg][k][2])));
            Rp = Rk; pp = pj;
        }
        int sf = 0;
        while (kFootLeg[sf] != leg) sf++;
        K.hip[sf] = p + mul(R, v3(kJointOrigin[leg][0][0], kJointOrigin[leg][0][1], kJointOrigin[leg][0][2]));
        K.foot[sf] = p + pp + mul(Rp, v3(kFootOffset[leg][0], kFootOffset[leg][1], kFootOffset[leg][2]));
    }
    K.com = p + (1.0 / kTotalMass) * mr;
}

// Everything a gait call reads of one robot, validated.
struct GaitIn {
    V3 p, vmeas;
    M3 R;
    double yaw, q[12];
    double fr[4][4];      // per stacked foot: n_x, n_y, n_z, d (terrain form)
    bool terrain;
    int status;
};

WBC_HD bool gait_finite(double x) { return x - x == 0.0; }

WBC_DEVFN inline void gait_read(const GaitIO& io, long i, GaitIn& g)
{
    const long ld = io.ld;
    bool finite = true;
    double b[3];
    for (int k = 0; k < 3; k++) { b[k] = io.base_pos[k * ld + i]; finite = finite && gait_finite(b[k]); }
    g.p = v3(b[0], b[1], b[2]);
    for (int k = 0; k < 3; k++) { b[k] = io.base_vel[k * ld + i]; finite = finite && gait_finite(b[k]); }
    g.vmeas = v3(b[0], b[1], b[2]);
    for (int k = 0; k < 9; k++) { g.R.m[k] = io.base_rot[k * ld + i]; finite = finite && gait_finite(g.R.m[k]); }
    g.yaw = io.base_rpy[2 * ld + i];
    finite = finite && gait_finite(g.yaw);
    for (int k = 0; k < 12; k++) { g.q[k] = io.q[k * ld + i]; finite = finite && gait_finite(g.q[k]); }
    g.terrain = io.terrain != nullptr;
    bool frames_ok = true;
    for (int sf = 0; sf < 4; sf++) {
        g.fr[sf][0] = g.fr[sf][1] = 0.0; g.fr[sf][2] = 1.0; g.fr[sf][3] = 0.0;
        if (!g.terrain) continue;
        double fr[9];
        for (int k = 0; k < 9; k++) { fr[k] = io.terrain[(10 * sf + k) * ld + i]; finite = finite && gait_finite(fr[k]); }
        for (int a = 0; a < 3; a++)
            for (int c = a; c < 3; c++) {
                const double e = fr[3 * a] * fr[3 * c] + fr[3 * a + 1] * fr[3 * c + 1] + fr[3 * a + 2] * fr[3 * c + 2];
                frames_ok = frames_ok && fabs(e - (a == c ? 1.0 : 0.0)) <= 1e-9;
            }
        frames_ok = frames_ok && fr[2] >= 0.5;
        for (int k = 0; k < 3; k++) g.fr[sf][k] = fr[k];
        if (io.plane_d) { g.fr[sf][3] = io.plane_d[sf * ld + i]; finite = finite && gait_finite(g.fr[sf][3]); }
    }
    g.status = !finite ? GAIT_ST_NONFINITE : (!frames_ok ? GAIT_ST_BAD_TERRAIN : 0);
}

// Height of stacked foot sf's plane n . p = d above (x, y); 0 on flat ground.
WBC_HD double gait_plane_z(const GaitIn& g, int sf, double x, double y)
{
    return g.terrain ? (g.fr[sf][3] - g.fr[sf][0] * x - g.fr[sf][1] * y) / g.fr[sf][2] : 0.0;
}

// Ground height under (x, y): the mean of the four feet's plane heights.
WBC_HD double gait_ground_z(const GaitIn& g, double x, double y)
{
    if (!g.terrain) return 0.0;
    return 0.25 * (gait_plane_z(g, 0, x, y) + gait_plane_z(g, 1, x, y) + gait_plane_z(g, 2, x, y) + gait_plane_z(g, 3, x, y));
}

// The two stacked feet of the swing pair of `phase` (phases 0, 1: BR, FL; 2, 3: BL, FR), in Jsw row order.
WBC_HD void gait_pair(int phase, int& f0, int& f1) { f0 = phase < 2 ? 0 : 1; f1 = phase < 2 ? 2 : 3; }

// Touchdown target of stacked swing foot sf lifting off now from p0 (DESIGN.md 4.8): a Raibert-style point ahead of the hip by the
// reference velocity over tau = the rest of the swing plus half the coming ground period, plus the captured foot offset, corrected by
// k_v (v_meas - v_ref) and kept within max_step of that neutral point.  cref: com_ref (x, y, clearance, yaw), vref: v_ref.
WBC_HD V3 gait_target(const GaitParams& G, double dt, const GaitIn& g, const GaitKin& K, int sf, const V3& p0, const double* cref,
                      const double* vref, const double* off)
{
    const double tau = G.nw * dt + (2 * G.ns + G.nw) * dt / 2.0;
    const double cy = cos(cref[3]), sy = sin(cref[3]);
    const double vwx = cy * vref[0] - sy * vref[1], vwy = sy * vref[0] + cy * vref[1];
    const double rx = K.hip[sf].x - cref[0], ry = K.hip[sf].y - cref[1];
    const double nx = K.hip[sf].x + tau * (vwx - vref[2] * ry) + (cy * off[0] - sy * off[1]);
    const double ny = K.hip[sf].y + tau * (vwy + vref[2] * rx) + (sy * off[0] + cy * off[1]);
    double dx = G.k_v * (g.vmeas.x - vwx), dy = G.k_v * (g.vmeas.y - vwy);
    const double d = sqrt(dx * dx + dy * dy);
    if (d > G.max_step) { dx *= G.max_step / d; dy *= G.max_step / d; }
    const double x = nx + dx, y = ny + dy;
    return v3(x, y, g.terrain ? gait_plane_z(g, sf, x, y) : p0.z);
}

// Map a start offset k0 (taken modulo the gait period) to (phase, tick).
WBC_HD void gait_phase_of(const GaitParams& G, int k0, int& phase, int& tick)
{
    const int period = 2 * (G.ns + G.nw);
    int k = k0 % period;
    if (k < 0) k += period;
    phase = 0;
    for (;;) {
        const int len = (phase & 1) ? G.nw : G.ns;
        if (k < len) break;
        k -= len;
        phase++;
    }
    tick = k;
}

WBC_DEVFN inline void gait_init_instance(const GaitParams& G, double dt, const GaitIO& io, long i)
{
    const long ld = io.ld;
    GaitIn g;
    gait_read(io, i, g);
    if (io.status) io.status[i] = g.status;
    if (g.status != 0) return;
    GaitKin K;
    gait_kinematics(g.p, g.R, g.q, K);
    const double cref[4] = {K.com.x, K.com.y, K.com.z - gait_ground_z(g, K.com.x, K.com.y), g.yaw};
    const double vref[3] = {0.0, 0.0, 0.0};
    const double cy = cos(g.yaw), sy = sin(g.yaw);
    double off[8];
    for (int sf = 0; sf < 4; sf++) {
        const double dx = K.foot[sf].x - K.hip[sf].x, dy = K.foot[sf].y - K.hip[sf].y;
        off[2 * sf] = cy * dx + sy * dy;
        off[2 * sf + 1] = -sy * dx + cy * dy;
    }
    int phase, tick;
    gait_phase_of(G, io.k0 ? io.k0[i] : 0, phase, tick);
    int f[2];
    gait_pair(phase, f[0], f[1]);
    for (int j = 0; j < 2; j++) {
        const V3 p0 = K.foot[f[j]];
        const V3 p1 = (phase & 1) ? gait_target(G, dt, g, K, f[j], p0, cref, vref, off + 2 * f[j]) : p0;
        for (int a = 0; a < 3; a++) {
            io.liftoff[(3 * j + a) * ld + i] = comp(p0, a);
            io.target[(3 * j + a) * ld + i] = comp(p1, a);
        }
    }
    io.phase[i] = phase; io.tick[i] = tick; io.landed[i] = 0;
    for (int k = 0; k < 4; k++) io.com_ref[k * ld + i] = cref[k];
    for (int k = 0; k < 3; k++) io.v_ref[k * ld + i] = vref[k];
    for (int k = 0; k < 8; k++) io.offset[k * ld + i] = off[k];
}

WBC_DEVFN inline void gait_step_instance(const GaitParams& G, double dt, const GaitIO& io, long i)
{
    const long ld = io.ld, old = io.out_ld;
    GaitIn g;
    gait_read(io, i, g);
    int phase = io.phase[i], tick = io.tick[i], landed = io.landed[i];
    double cref[4], vref[3], p0[6], p1[6], off[8], cmd[3] = {0.0, 0.0, 0.0};
    bool finite = true;
    for (int k = 0; k < 4; k++) { cref[k] = io.com_ref[k * ld + i]; finite = finite && gait_finite(cref[k]); }
    for (int k = 0; k < 3; k++) { vref[k] = io.v_ref[k * ld + i]; finite = finite && gait_finite(vref[k]); }
    for (int k = 0; k < 6; k++) { p0[k] = io.liftoff[k * ld + i]; p1[k] = io.target[k * ld + i]; finite = finite && gait_finite(p0[k]) && gait_finite(p1[k]); }
    for (int k = 0; k < 8; k++) { off[k] = io.offset[k * ld + i]; finite = finite && gait_finite(off[k]); }
    if (io.cmd)
        for (int k = 0; k < 3; k++) { cmd[k] = io.cmd[k * ld + i]; finite = finite && gait_finite(cmd[k]); }
    int status = g.status;
    if (status == 0 && !finite) status = GAIT_ST_NONFINITE;
    const bool swing = (phase & 1) != 0;
    const int len = swing ? G.nw : G.ns;
    if (status == 0 && (phase < 0 || phase > 3 || tick < 0 || tick >= len)) status = GAIT_ST_BAD_MODE;
    if (io.status) io.status[i] = status;
    if (status != 0) return;
    int f[2];
    gait_pair(phase, f[0], f[1]);

    // 1. touchdown
    if (swing && !landed && (double)(tick + 1) / G.nw > GAIT_TOUCHDOWN_S && io.contact && io.contact[f[0] * ld + i] != 0 &&
        io.contact[f[1] * ld + i] != 0)
        landed = 1;
    GaitKin K;
    gait_kinematics(g.p, g.R, g.q, K);
    // 2. lift-off
    if (swing && tick == 0)
        for (int j = 0; j < 2; j++) {
            const V3 a = K.foot[f[j]];
            const V3 b = gait_target(G, dt, g, K, f[j], a, cref, vref, off + 2 * f[j]);
            for (int c = 0; c < 3; c++) { p0[3 * j + c] = comp(a, c); p1[3 * j + c] = comp(b, c); }
        }
    // 3. command ramp
    double dvx = cmd[0] - vref[0], dvy = cmd[1] - vref[1], dw = cmd[2] - vref[2];
    const double lim = G.acc_lin * dt, dn = sqrt(dvx * dvx + dvy * dvy);
    if (dn > lim) {
        dvx *= lim / dn; dvy *= lim / dn;
        vref[0] += dvx; vref[1] += dvy;
    } else {
        vref[0] = cmd[0]; vref[1] = cmd[1];
    }
    const double wlim = G.acc_yaw * dt;
    if (dw > wlim) { dw = wlim; vref[2] += dw; }
    else if (dw < -wlim) { dw = -wlim; vref[2] += dw; }
    else vref[2] = cmd[2];
    // 4. CoM reference
    const double w = vref[2];
    cref[3] += w * dt;
    const double cy = cos(cref[3]), sy = sin(cref[3]);
    const double vwx = cy * vref[0] - sy * vref[1], vwy = sy * vref[0] + cy * vref[1];
    cref[0] += vwx * dt;
    cref[1] += vwy * dt;
    {
        const double ex = cref[0] - K.com.x, ey = cref[1] - K.com.y, e = sqrt(ex * ex + ey * ey);
        if (e > G.leash) { cref[0] = K.com.x + ex * (G.leash / e); cref[1] = K.com.y + ey * (G.leash / e); }
    }
    const double zref = cref[2] + gait_ground_z(g, cref[0], cref[1]);
    // 5. emit
    const int mode = landed ? MODE_STANCE : (phase == 1 ? MODE_SWING_BR_FL : (phase == 3 ? MODE_SWING_BL_FR : MODE_STANCE));
    const double pi = 3.14159265358979323846;
    double dyaw = cref[3] - g.yaw;
    dyaw -= 2.0 * pi * floor((dyaw + pi) / (2.0 * pi));
    const double ax = dvx / dt, ay = dvy / dt;
    const double cp[6] = {cref[0], cref[1], zref, 0.0, 0.0, g.yaw + dyaw};
    const double cv[6] = {vwx, vwy, 0.0, 0.0, 0.0, w};
    const double ca[6] = {cy * ax - sy * ay - w * vwy, sy * ax + cy * ay + w * vwx, 0.0, 0.0, 0.0, dw / dt};
    double sp[6], sv[6], sa[6];
    if (swing) {
        const double s = (double)(tick + 1) / G.nw, r = 1.0 / (G.nw * dt);
        const double s2 = s * s, s3 = s2 * s;
        const double sig = s3 * (10.0 - 15.0 * s + 6.0 * s2);
        const double dsig = 30.0 * s2 * (1.0 - 2.0 * s + s2) * r;
        const double ddsig = 60.0 * s * (1.0 - 3.0 * s + 2.0 * s2) * r * r;
        const double sn = sin(pi * s), s2p = sin(2.0 * pi * s), c2p = cos(2.0 * pi * s);
        for (int a = 0; a < 6; a++) {
            const double d = p1[a] - p0[a], up = (a % 3 == 2) ? G.step_height : 0.0;
            sp[a] = p0[a] + d * sig + up * sn * sn;
            sv[a] = d * dsig + up * pi * s2p * r;
            sa[a] = d * ddsig + up * 2.0 * pi * pi * c2p * r * r;
        }
    } else {
        for (int j = 0; j < 2; j++)
            for (int c = 0; c < 3; c++) { sp[3 * j + c] = comp(K.foot[f[j]], c); sv[3 * j + c] = 0.0; sa[3 * j + c] = 0.0; }
    }
    io.mode[i] = mode;
    for (int k = 0; k < 6; k++) {
        io.des[0][k * old + i] = cp[k]; io.des[1][k * old + i] = cv[k]; io.des[2][k * old + i] = ca[k];
        io.des[3][k * old + i] = sp[k]; io.des[4][k * old + i] = sv[k]; io.des[5][k * old + i] = sa[k];
    }
    // 6. advance
    if (++tick >= len) { phase = (phase + 1) & 3; tick = 0; landed = 0; }
    io.phase[i] = phase; io.tick[i] = tick; io.landed[i] = landed;
    for (int k = 0; k < 4; k++) io.com_ref[k * ld + i] = cref[k];
    for (int k = 0; k < 3; k++) io.v_ref[k * ld + i] = vref[k];
    for (int k = 0; k < 6; k++) { io.liftoff[k * ld + i] = p0[k]; io.target[k * ld + i] = p1[k]; }
}

}  // namespace wbc
