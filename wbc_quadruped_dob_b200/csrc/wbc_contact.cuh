// Contact plant: forward dynamics with unilateral, frictional point contacts at the feet (wbc_plant_contact_step).
//
// One control period (params.obs_dt) of one instance in `substeps` steps of dt.  Per step:
//   1. front_dynamics at the current state (M, h, foot Jacobians J; the same dynamics as fdyn_step_instance);
//   2. free velocity  nu_free = nu + dt M^-1 (S'tau + push_gen - h);
//   3. candidate feet by geometry alone: gap phi_k = p_k,z - ground_z[k] <= margin (the contact mode is not read);
//   4. impulses lambda (3 per candidate foot, world axes): the unique minimiser of the strictly convex QP
//          min 1/2 lambda'(G + eps D) lambda + lambda'(J nu_free - b),   G = J M^-1 J', D = diag(G),
//      over the friction pyramid of every candidate foot (lambda_z >= 0, |lambda_x| <= mu lambda_z, |lambda_y| <= mu lambda_z;
//      the controller's own cfr rows, 5 per foot); b = 0 tangentially and -phi/dt (phi >= 0: speculative, the gap may close but
//      the foot may not cross the plane) or -beta phi/dt (phi < 0: Baumgarte push-out) along the normal.  This is the convex
//      (Anitescu-type) relaxation of Coulomb contact: a sticking foot is exact, a sliding foot is pushed off the plane at a normal
//      velocity of at most mu times its slip speed;
//   5. nu+ = nu_free + M^-1 J' lambda, then semi-implicit Euler and the exponential map of the base rotation, as fdyn_step_instance.
// The QP is solved to its KKT optimum by a thread-level Goldfarb-Idnani dual active-set method on the Cholesky factor of
// G + eps D (contact_qp below), warm-started from the previous step's active rows.
//
// The M^-1 block elimination is a copy of fdyn_step_instance's rather than a function shared with it, so that the bilateral
// plant's code (and its results) stay exactly as they are.
//
// Terrain form (TERRAIN = true, wbc_plant_contact_step_terrain): foot k has the plane {p : n_k . p = d_k} and its own frame
// F_k = [t1 t2 n] and mu_k, in the controller's terrain layout [40][ld] (rows 10k..10k+2 n, +3..+5 t1, +6..+8 t2, +9 mu); d_k is
// read where the flat form reads ground_z.  The gap is measured along n_k, each candidate foot's three Jacobian rows are rotated
// into its frame (J_local = F_k' J_world), so lambda = (lambda_t1, lambda_t2, lambda_n) and the same pyramid rows describe the
// controller's cone rows; the forces leave as R_foot' F_k lambda / dt.  With F_k = I the arithmetic is the flat form's.
#pragma once
#include <math.h>

#include "wbc_front.cuh"

namespace wbc {

struct ContactParams {     // wbc_contact_params
    double beta, eps, margin;
    int max_iter;
};

struct ContactIO {
    double *base_pos, *base_rot, *base_rpy, *base_vel, *q, *dq, *foot_force;   // state, SoA [k][ld], advanced in place on success
    const double *tau, *push;        // [12][ld], [6][ld]
    const double *ground_z, *mu;     // [4][ld] or nullptr (0), [ld] or nullptr (Params::mu); terrain form: plane offsets d, mu unused
    int* contact;                    // [4][ld] or nullptr: 0 no contact force, 1 sticking, 2 sliding (last step)
    double* diag;                    // [4][ld] or nullptr: max penetration, min normal force, max KKT residual, active-set iterations
    int* status;                     // [ld] or nullptr
    long ld;
};

constexpr int CONTACT_ST_NONFINITE = -21;   // WBC_ST_NONFINITE
constexpr int CONTACT_ST_BAD_TERRAIN = -24; // WBC_ST_BAD_TERRAIN
constexpr int CONTACT_ST_MAX_ITER = -100;

// Row t of a foot's friction pyramid in "n . lambda_foot >= 0" form, unit length: 0 normal, 1/2 -+x, 3/4 -+y.
WBC_HD void pyramid_row(int t, double mu, double* n)
{
    const double s = 1.0 / sqrt(1.0 + mu * mu);
    n[0] = n[1] = 0.0; n[2] = 1.0;
    if (t == 0) return;
    n[2] = mu * s;
    n[(t - 1) >> 1] = ((t & 1) ? -1.0 : 1.0) * s;
}

struct ContactQpResult {
    int status;         // 0, or CONTACT_ST_MAX_ITER
    int iters;          // dual steps taken
    double kkt;         // scaled KKT residual of the result
};

// Goldfarb-Idnani dual active-set solve of  min 1/2 x'Hx + g'x  s.t.  n_r . x_foot(r) >= 0  for the 5 pyramid rows of each of the
// nf feet (variables 3f..3f+2 of foot f, row id 5 f + t).  H (nv x nv, stride 12, nv = 3 nf) is overwritten with its Cholesky
// factor.  `warm` (bit r: row r) lists rows to start from; it returns the final active rows.  J = L^-T Q and the upper-triangular R
// of the active rows are updated by Givens rotations (quadprog's formulation); the result is x, and u holds the multipliers of
// the rows in act[0..q).  Rows of a warm set that depend on the rows already added are skipped; after the warm rows, the point
// and multipliers are those of the equality problem on them, and negative multipliers are dropped before the dual loop.
WBC_HD ContactQpResult contact_qp(double* H, const double* g, int nf, const double* mu, unsigned& warm, int max_iter, double* x)
{
    const int nv = 3 * nf, nr = 5 * nf;
    double J[144], R[144], u[12], d[12], z[12], r[12], xs = 0.0;
    int act[12], q = 0;
    ContactQpResult res; res.status = 0; res.iters = 0; res.kkt = 0.0;
    double Hs[144];
    for (int k = 0; k < nv * 12; k++) Hs[k] = H[k];
    // H = L L' in place (lower), J = L^-T (upper triangular)
    for (int j = 0; j < nv; j++) {
        double dd = H[j * 12 + j];
        for (int k = 0; k < j; k++) dd -= H[j * 12 + k] * H[j * 12 + k];
        dd = sqrt(dd);
        H[j * 12 + j] = dd;
        for (int i = j + 1; i < nv; i++) {
            double sacc = H[i * 12 + j];
            for (int k = 0; k < j; k++) sacc -= H[i * 12 + k] * H[j * 12 + k];
            H[i * 12 + j] = sacc / dd;
        }
    }
    for (int c = 0; c < nv; c++)                     // column c of L^-T: solve L' y = e_c
        for (int i = nv - 1; i >= 0; i--) {
            double sacc = (i == c) ? 1.0 : 0.0;
            for (int k = i + 1; k < nv; k++) sacc -= H[k * 12 + i] * J[k * 12 + c];
            J[i * 12 + c] = sacc / H[i * 12 + i];
        }
    auto row_n = [&](int p, double* n) { pyramid_row(p % 5, mu[p / 5], n); };
    auto n_dot = [&](int p, const double* v) {
        double n[3]; row_n(p, n);
        const int b = 3 * (p / 5);
        return n[0] * v[b] + n[1] * v[b + 1] + n[2] * v[b + 2];
    };
    // d = J' n_p; returns |d[q..nv)|^2 and |d|^2
    auto jt_n = [&](int p, double& all) {
        double n[3]; row_n(p, n);
        const int b = 3 * (p / 5);
        double tail = 0.0; all = 0.0;
        for (int j = 0; j < nv; j++) {
            d[j] = J[b * 12 + j] * n[0] + J[(b + 1) * 12 + j] * n[1] + J[(b + 2) * 12 + j] * n[2];
            all += d[j] * d[j];
            if (j >= q) tail += d[j] * d[j];
        }
        return tail;
    };
    // append row p (d = J' n_p already computed): rotate d[q+1..nv) into d[q], then R[:, q] = d[0..q]
    auto add_row = [&](int p) {
        for (int j = nv - 1; j > q; j--) {
            const double a = d[j - 1], b = d[j];
            if (b == 0.0) continue;
            const double h = sqrt(a * a + b * b), c = a / h, s = b / h;
            d[j - 1] = h; d[j] = 0.0;
            for (int i = 0; i < nv; i++) {
                const double ja = J[i * 12 + j - 1], jb = J[i * 12 + j];
                J[i * 12 + j - 1] = c * ja + s * jb;
                J[i * 12 + j] = s * ja - c * jb;
            }
        }
        for (int i = 0; i <= q; i++) R[i * 12 + q] = d[i];
        act[q] = p;
        q++;
    };
    // remove active entry l: shift R's columns, act and u left, restore the triangle with Givens rotations (applied to J as well)
    auto drop = [&](int l) {
        for (int c = l; c < q - 1; c++) {
            for (int i = 0; i <= c + 1; i++) R[i * 12 + c] = R[i * 12 + c + 1];
            act[c] = act[c + 1]; u[c] = u[c + 1];
        }
        q--;
        for (int j = l; j < q; j++) {
            const double a = R[j * 12 + j], b = R[(j + 1) * 12 + j];
            if (b == 0.0) continue;
            const double h = sqrt(a * a + b * b), c = a / h, s = b / h;
            for (int k = j; k < q; k++) {
                const double ra = R[j * 12 + k], rb = R[(j + 1) * 12 + k];
                R[j * 12 + k] = c * ra + s * rb;
                R[(j + 1) * 12 + k] = s * ra - c * rb;
            }
            R[(j + 1) * 12 + j] = 0.0;
            for (int i = 0; i < nv; i++) {
                const double ja = J[i * 12 + j], jb = J[i * 12 + j + 1];
                J[i * 12 + j] = c * ja + s * jb;
                J[i * 12 + j + 1] = s * ja - c * jb;
            }
        }
    };
    // the equality problem on the active rows: x = -J2 J2' g, u = R^-1 J1' g
    auto solve_active = [&]() {
        double jg[12];
        for (int j = 0; j < nv; j++) {
            double sacc = 0.0;
            for (int i = 0; i < nv; i++) sacc += J[i * 12 + j] * g[i];
            jg[j] = sacc;
        }
        for (int i = 0; i < nv; i++) {
            double sacc = 0.0;
            for (int j = q; j < nv; j++) sacc += J[i * 12 + j] * jg[j];
            x[i] = -sacc;
        }
        for (int i = q - 1; i >= 0; i--) {
            double sacc = jg[i];
            for (int k = i + 1; k < q; k++) sacc -= R[i * 12 + k] * u[k];
            u[i] = sacc / R[i * 12 + i];
        }
    };
    // ---- warm start: add the warm rows (ascending), then drop negative multipliers one at a time
    for (int p = 0; p < nr; p++) {
        if (!((warm >> p) & 1u) || q == nv) continue;
        double all;
        const double tail = jt_n(p, all);
        if (tail > 1e-24 * all) add_row(p);
    }
    solve_active();
    for (;;) {
        int l = -1; double umin = 0.0;
        for (int j = 0; j < q; j++) if (u[j] < umin) { umin = u[j]; l = j; }
        if (l < 0) break;
        drop(l);
        solve_active();
    }
    for (int i = 0; i < nv; i++) xs = fmax(xs, fabs(x[i]));
    {   // scale of the solution: |x*|_H <= 2 |x_unconstrained|_H, x_unconstrained = -J J' g
        double jg[12];
        for (int j = 0; j < nv; j++) { double sacc = 0.0; for (int i = 0; i < nv; i++) sacc += J[i * 12 + j] * g[i]; jg[j] = sacc; }
        for (int i = 0; i < nv; i++) { double sacc = 0.0; for (int j = 0; j < nv; j++) sacc += J[i * 12 + j] * jg[j]; xs = fmax(xs, fabs(sacc)); }
    }
    const double tol = 1e-13 * xs;
    // ---- dual loop
    for (;;) {
        int p = -1; double smin = -tol;
        for (int rr = 0; rr < nr; rr++) {
            bool in = false;
            for (int j = 0; j < q; j++) in = in || act[j] == rr;
            if (in) continue;
            const double sv = n_dot(rr, x);
            if (sv < smin) { smin = sv; p = rr; }
        }
        if (p < 0) break;
        double up = 0.0;
        for (;;) {
            if (res.iters >= max_iter) { res.status = CONTACT_ST_MAX_ITER; warm = 0u; return res; }
            res.iters++;
            double all;
            const double tail = jt_n(p, all);
            for (int i = 0; i < nv; i++) {
                double sacc = 0.0;
                for (int j = q; j < nv; j++) sacc += J[i * 12 + j] * d[j];
                z[i] = sacc;
            }
            for (int i = q - 1; i >= 0; i--) {
                double sacc = d[i];
                for (int k = i + 1; k < q; k++) sacc -= R[i * 12 + k] * r[k];
                r[i] = sacc / R[i * 12 + i];
            }
            int l = -1; double t1 = 1e300;
            for (int j = 0; j < q; j++)
                if (r[j] > 0.0 && u[j] / r[j] < t1) { t1 = u[j] / r[j]; l = j; }
            const bool full = tail > 1e-24 * all;           // z . n_p = |d[q..nv)|^2: 0 when n_p depends on the active rows
            const double t2 = full ? -n_dot(p, x) / tail : 1e300;
            if (!full && l < 0) { res.status = CONTACT_ST_MAX_ITER; warm = 0u; return res; }   // infeasible: cannot happen (0 is feasible)
            if (full && t2 <= t1) {
                for (int i = 0; i < nv; i++) x[i] += t2 * z[i];
                for (int j = 0; j < q; j++) u[j] -= t2 * r[j];
                up += t2;
                add_row(p);
                u[q - 1] = up;
                break;
            }
            if (full) for (int i = 0; i < nv; i++) x[i] += t1 * z[i];
            for (int j = 0; j < q; j++) u[j] -= t1 * r[j];
            up += t1;
            drop(l);
        }
    }
    // ---- KKT residual, scaled: stationarity |Hx + g - N'u| / max(|g|, |Hx|), primal and dual feasibility, complementarity; the
    // scale of x is xs (the solution's and the unconstrained minimiser's), which stays meaningful when every foot carries nothing
    {
        double gs = 1e-300, st = 0.0, pv = 0.0, dv = 0.0, cp = 0.0, xm = fmax(xs, 1e-300);
        double grad[12];
        for (int i = 0; i < nv; i++) {
            double sacc = 0.0;
            for (int k = 0; k < nv; k++) sacc += Hs[i * 12 + k] * x[k];
            gs = fmax(gs, fmax(fabs(sacc), fabs(g[i])));
            grad[i] = sacc + g[i];
        }
        for (int j = 0; j < q; j++) {
            double n[3]; row_n(act[j], n);
            const int b = 3 * (act[j] / 5);
            for (int a = 0; a < 3; a++) grad[b + a] -= u[j] * n[a];
            dv = fmax(dv, -u[j]);
            cp = fmax(cp, fabs(u[j] * n_dot(act[j], x)));
        }
        for (int i = 0; i < nv; i++) st = fmax(st, fabs(grad[i]));
        for (int rr = 0; rr < nr; rr++) pv = fmax(pv, -n_dot(rr, x));
        res.kkt = fmax(fmax(st / gs, pv / xm), fmax(dv / gs, cp / (gs * xm)));
    }
    warm = 0u;
    for (int j = 0; j < q; j++) warm |= 1u << act[j];
    return res;
}

// TERRAIN: the terrain form (see the top of this file); `terrain` [40][ld] is then required and io.ground_z holds the plane offsets.
template <bool TERRAIN = false>
WBC_DEVFN inline void contact_step_instance(const Params& P, const ContactParams& cp, const ContactIO& io, long i, int nsub,
                                            const double* terrain = nullptr)
{
    using namespace dogbot;
    const long ld = io.ld;
    // the state is advanced in a local copy, written back only when every step succeeded
    double s[45];   // base_pos 3 | base_rot 9 | base_rpy 3 | base_vel 6 | q 12 | dq 12
    double* const sp[6] = {io.base_pos, io.base_rot, io.base_rpy, io.base_vel, io.q, io.dq};
    const int so[7] = {0, 3, 12, 15, 21, 33, 45};
    double tau[12], push[6], gz[4], mu = io.mu ? io.mu[i] : P.mu;
    bool finite = (mu - mu == 0.0);
    for (int f = 0; f < 6; f++)
        for (int k = so[f]; k < so[f + 1]; k++) { s[k] = sp[f][(long)(k - so[f]) * ld + i]; finite = finite && (s[k] - s[k] == 0.0); }
    for (int k = 0; k < 12; k++) { tau[k] = io.tau[(long)k * ld + i]; finite = finite && (tau[k] - tau[k] == 0.0); }
    for (int k = 0; k < 6; k++) { push[k] = io.push[(long)k * ld + i]; finite = finite && (push[k] - push[k] == 0.0); }
    for (int k = 0; k < 4; k++) { gz[k] = io.ground_z ? io.ground_z[(long)k * ld + i] : 0.0; finite = finite && (gz[k] - gz[k] == 0.0); }
    bool frames_ok = true;            // terrain form: every foot's frame orthonormal to 1e-9 and mu >= 0
    if (TERRAIN)
        for (int sf = 0; sf < 4; sf++) {
            double fr[10];
            for (int k = 0; k < 10; k++) { fr[k] = terrain[(long)(10 * sf + k) * ld + i]; finite = finite && (fr[k] - fr[k] == 0.0); }
            for (int a = 0; a < 3; a++)
                for (int c = a; c < 3; c++) {
                    const double e = fr[3 * a] * fr[3 * c] + fr[3 * a + 1] * fr[3 * c + 1] + fr[3 * a + 2] * fr[3 * c + 2];
                    frames_ok = frames_ok && fabs(e - (a == c ? 1.0 : 0.0)) <= 1e-9;
                }
            frames_ok = frames_ok && fr[9] >= 0.0;
        }
    DevInputs in;
    in.base_pos = s; in.base_rot = s + 3; in.base_rpy = s + 12; in.base_vel = s + 15; in.q = s + 21; in.dq = s + 33;
    in.com_des_pos = in.com_des_vel = in.com_des_acc = in.sw_des_pos = in.sw_des_vel = in.sw_des_acc = nullptr;
    in.foot_force = nullptr; in.terrain = nullptr; in.mode = nullptr; in.obs_gain = nullptr; in.ld = 1;
    const double dt = P.obs_dt / (double)nsub;
    double pen = 0.0, fzmin = 1.0e300, kkt = 0.0, iters = 0.0;
    double fs_out[12];
    int flag_out[4] = {0, 0, 0, 0};
    int status = finite ? 0 : CONTACT_ST_NONFINITE;
    if (TERRAIN && status == 0 && !frames_ok) status = CONTACT_ST_BAD_TERRAIN;
    unsigned warm = 0u;               // active rows of the previous step, row id 5 * stacked foot + pyramid row
    for (int k = 0; k < 12; k++) fs_out[k] = 0.0;
    for (int it = 0; it < nsub && status == 0; it++) {
        FrontDyn D;
        front_dynamics(P, in, 0, D);
        // M^-1 by block elimination (as in fdyn_step_instance): four 3 x 3 leg factors, Z_l = Mjj_l^-1 Mbj_l', Schur complement Sb
        double Lj[4][6], Z[4][18];
        double Sb[36];
        for (int k = 0; k < 36; k++) Sb[k] = D.Mb[k];
        for (int leg = 0; leg < 4; leg++) {
            const int i0 = dof_index(leg, 0), i1 = dof_index(leg, 1), i2 = i1 + 1;
            double* l = Lj[leg];
            const double m00 = D.Mjj[i0 * 12 + i0], m10 = D.Mjj[i1 * 12 + i0], m11 = D.Mjj[i1 * 12 + i1];
            const double m20 = D.Mjj[i2 * 12 + i0], m21 = D.Mjj[i2 * 12 + i1], m22 = D.Mjj[i2 * 12 + i2];
            const double d0 = sqrt(m00);
            l[0] = 1.0 / d0; l[1] = m10 * l[0]; l[3] = m20 * l[0];
            const double d1 = sqrt(m11 - l[1] * l[1]);
            l[2] = 1.0 / d1; l[4] = (m21 - l[3] * l[1]) * l[2];
            const double d2 = sqrt(m22 - l[3] * l[3] - l[4] * l[4]);
            l[5] = 1.0 / d2;
            for (int k = 0; k < 6; k++) {
                double y0 = D.Mbj[k * 12 + i0] * l[0];
                double y1 = (D.Mbj[k * 12 + i1] - l[1] * y0) * l[2];
                double y2 = (D.Mbj[k * 12 + i2] - l[3] * y0 - l[4] * y1) * l[5];
                y2 = y2 * l[5]; y1 = (y1 - l[4] * y2) * l[2]; y0 = (y0 - l[1] * y1 - l[3] * y2) * l[0];
                Z[leg][0 * 6 + k] = y0; Z[leg][1 * 6 + k] = y1; Z[leg][2 * 6 + k] = y2;
            }
            for (int r = 0; r < 6; r++)
                for (int c2 = 0; c2 < 6; c2++)
                    Sb[r * 6 + c2] -= D.Mbj[r * 12 + i0] * Z[leg][0 * 6 + c2] + D.Mbj[r * 12 + i1] * Z[leg][1 * 6 + c2] + D.Mbj[r * 12 + i2] * Z[leg][2 * 6 + c2];
        }
        chol6(Sb);
        auto solveM = [&](const double* rb, const double* rj, unsigned legs, double* xb, double* xj) {
            double t[6], y[12];
            for (int k = 0; k < 6; k++) t[k] = rb[k];
            for (int leg = 0; leg < 4; leg++) {
                const int i0 = dof_index(leg, 0), i1 = dof_index(leg, 1), i2 = i1 + 1;
                if (!(legs & (1u << leg))) { y[i0] = y[i1] = y[i2] = 0.0; continue; }
                const double* l = Lj[leg];
                double y0 = rj[i0] * l[0];
                double y1 = (rj[i1] - l[1] * y0) * l[2];
                double y2 = (rj[i2] - l[3] * y0 - l[4] * y1) * l[5];
                y2 = y2 * l[5]; y1 = (y1 - l[4] * y2) * l[2]; y0 = (y0 - l[1] * y1 - l[3] * y2) * l[0];
                y[i0] = y0; y[i1] = y1; y[i2] = y2;
                for (int r = 0; r < 6; r++) t[r] -= D.Mbj[r * 12 + i0] * y0 + D.Mbj[r * 12 + i1] * y1 + D.Mbj[r * 12 + i2] * y2;
            }
            chol6_solve(Sb, t);
            for (int k = 0; k < 6; k++) xb[k] = t[k];
            for (int leg = 0; leg < 4; leg++) {
                const int i0 = dof_index(leg, 0), i1 = dof_index(leg, 1), i2 = i1 + 1;
                const int id[3] = {i0, i1, i2};
                for (int a = 0; a < 3; a++) {
                    double sacc = y[id[a]];
                    for (int k = 0; k < 6; k++) sacc -= Z[leg][a * 6 + k] * t[k];
                    xj[id[a]] = sacc;
                }
            }
        };
        // nu_free = nu + dt M^-1 (S'tau - h + push_gen)
        double nu[18], b[18], a0[18];
        for (int k = 0; k < 6; k++) nu[k] = s[15 + k];
        for (int k = 0; k < 12; k++) nu[6 + k] = s[33 + k];
        const V3 xbc = (1.0 / kTotalMass) * D.mr;
        const V3 tq = cross(xbc, v3(push[0], push[1], push[2]));
        for (int k = 0; k < 6; k++) b[k] = -D.hb[k] + push[k];
        b[3] += tq.x; b[4] += tq.y; b[5] += tq.z;
        for (int k = 0; k < 12; k++) b[6 + k] = -D.hj[k] + tau[k];
        solveM(b, b + 6, 0xfu, a0, a0 + 6);
        for (int a = 0; a < 18; a++) nu[a] += dt * a0[a];
        // candidate feet (geometry only) and their Jacobian rows
        double Jb[12 * 6], Jl[12 * 3], phi[4], g[12];
        int rleg[12], cand[4], nf = 0;
        double mu_f[4];
        unsigned wsub = 0u;           // the previous step's active rows, renumbered to this step's candidate feet
        for (int sf = 0; sf < 4; sf++) {
            const int leg = kFootLeg[sf];
            const V3 rf = D.footp[leg];
            double fr[10];            // terrain form: this foot's n, t1, t2, mu
            if (TERRAIN) {
                for (int k = 0; k < 10; k++) fr[k] = terrain[(long)(10 * sf + k) * ld + i];
                phi[sf] = fr[0] * (s[0] + rf.x) + fr[1] * (s[1] + rf.y) + fr[2] * (s[2] + rf.z) - gz[sf];
            } else {
                phi[sf] = s[2] + rf.z - gz[sf];
            }
            pen = fmax(pen, -phi[sf]);
            if (phi[sf] > cp.margin) continue;
            const double nSf[9] = {0, rf.z, -rf.y, -rf.z, 0, rf.x, rf.y, -rf.x, 0};
            if (TERRAIN) {
                // the world rows x, y, z, then local row c = (t1, t2, n)[c]' J_world
                double wb[18], wl[9];
                for (int a = 0; a < 3; a++)
                    for (int k = 0; k < 3; k++) { wb[a * 6 + k] = (k == a) ? 1.0 : 0.0; wb[a * 6 + 3 + k] = nSf[a * 3 + k]; wl[a * 3 + k] = D.Jleg[leg][a * 3 + k]; }
                for (int c = 0; c < 3; c++) {
                    const double* e = fr + (c == 2 ? 0 : 3 + 3 * c);
                    const int r = 3 * nf + c;
                    rleg[r] = leg;
                    for (int k = 0; k < 6; k++) Jb[r * 6 + k] = e[0] * wb[k] + e[1] * wb[6 + k] + e[2] * wb[12 + k];
                    for (int k = 0; k < 3; k++) Jl[r * 3 + k] = e[0] * wl[k] + e[1] * wl[3 + k] + e[2] * wl[6 + k];
                    double jn = 0.0;
                    for (int k = 0; k < 6; k++) jn += Jb[r * 6 + k] * nu[k];
                    for (int k = 0; k < 3; k++) jn += Jl[r * 3 + k] * nu[6 + dof_index(leg, k)];
                    g[r] = jn;
                }
            } else {
                for (int a = 0; a < 3; a++) {
                    const int r = 3 * nf + a;
                    rleg[r] = leg;
                    for (int k = 0; k < 3; k++) { Jb[r * 6 + k] = (k == a) ? 1.0 : 0.0; Jb[r * 6 + 3 + k] = nSf[a * 3 + k]; Jl[r * 3 + k] = D.Jleg[leg][a * 3 + k]; }
                    double jn = 0.0;
                    for (int k = 0; k < 6; k++) jn += Jb[r * 6 + k] * nu[k];
                    for (int k = 0; k < 3; k++) jn += Jl[r * 3 + k] * nu[6 + dof_index(leg, k)];
                    g[r] = jn;
                }
            }
            g[3 * nf + 2] += (phi[sf] >= 0.0 ? 1.0 : cp.beta) * phi[sf] / dt;
            wsub |= ((warm >> (5 * sf)) & 31u) << (5 * nf);
            mu_f[nf] = TERRAIN ? fr[9] : mu;
            cand[nf++] = sf;
        }
        const int nc = 3 * nf;
        // X = M^-1 J' (column r: Xb[r], Xj[r]), G = J X
        double Xb[12 * 6], Xj[12 * 12], H[144], lam[12];
        for (int rr = 0; rr < nc; rr++) {
            double rj[12];
            for (int k = 0; k < 12; k++) rj[k] = 0.0;
            for (int k = 0; k < 3; k++) rj[dof_index(rleg[rr], k)] = Jl[rr * 3 + k];
            solveM(Jb + rr * 6, rj, 1u << rleg[rr], Xb + rr * 6, Xj + rr * 12);
        }
        for (int p_ = 0; p_ < nc; p_++) {
            const int lp = rleg[p_];
            for (int q_ = 0; q_ <= p_; q_++) {
                double sacc = 0.0;
                for (int k = 0; k < 6; k++) sacc += Jb[p_ * 6 + k] * Xb[q_ * 6 + k];
                for (int k = 0; k < 3; k++) sacc += Jl[p_ * 3 + k] * Xj[q_ * 12 + dof_index(lp, k)];
                H[p_ * 12 + q_] = sacc; H[q_ * 12 + p_] = sacc;
            }
        }
        for (int p_ = 0; p_ < nc; p_++) H[p_ * 12 + p_] *= 1.0 + cp.eps;
        warm = 0u;
        for (int k = 0; k < 12; k++) fs_out[k] = 0.0;
        for (int k = 0; k < 4; k++) flag_out[k] = 0;
        if (nf > 0) {
            const ContactQpResult qr = contact_qp(H, g, nf, mu_f, wsub, cp.max_iter, lam);
            iters += qr.iters;
            kkt = fmax(kkt, qr.kkt);
            if (qr.status != 0) { status = qr.status; break; }
            for (int f = 0; f < nf; f++) {
                const int sf = cand[f];
                const unsigned rows = (wsub >> (5 * f)) & 31u;
                warm |= rows << (5 * sf);
                // an active normal row, or an active pair of opposite friction rows (mu > 0), means lambda_z = 0 and with it the
                // whole pyramid: the foot carries exactly nothing (rather than a rounding residue)
                const bool zero = (rows & 1u) || ((TERRAIN ? mu_f[f] : mu) > 0.0 && ((rows & 6u) == 6u || (rows & 24u) == 24u)) || lam[3 * f + 2] <= 0.0;
                if (zero) { lam[3 * f] = lam[3 * f + 1] = lam[3 * f + 2] = 0.0; }
                flag_out[sf] = lam[3 * f + 2] > 0.0 ? ((rows & 30u) ? 2 : 1) : 0;
                fzmin = fmin(fzmin, lam[3 * f + 2] / dt);
                const M3& Rf = D.footR[kFootLeg[sf]];
                if (TERRAIN) {
                    double lw[3];             // world impulse F lambda = t1 lambda_t1 + t2 lambda_t2 + n lambda_n
                    for (int a = 0; a < 3; a++)
                        lw[a] = terrain[(long)(10 * sf + 3 + a) * ld + i] * lam[3 * f] + terrain[(long)(10 * sf + 6 + a) * ld + i] * lam[3 * f + 1] +
                                terrain[(long)(10 * sf + a) * ld + i] * lam[3 * f + 2];
                    for (int k = 0; k < 3; k++) fs_out[3 * sf + k] = (Rf.m[k] * lw[0] + Rf.m[3 + k] * lw[1] + Rf.m[6 + k] * lw[2]) / dt;
                } else {
                    for (int k = 0; k < 3; k++)
                        fs_out[3 * sf + k] = (Rf.m[k] * lam[3 * f] + Rf.m[3 + k] * lam[3 * f + 1] + Rf.m[6 + k] * lam[3 * f + 2]) / dt;
                }
            }
            // nu+ = nu_free + X lambda
            for (int rr = 0; rr < nc; rr++) {
                for (int k = 0; k < 6; k++) nu[k] += Xb[rr * 6 + k] * lam[rr];
                for (int k = 0; k < 12; k++) nu[6 + k] += Xj[rr * 12 + k] * lam[rr];
            }
        }
        // semi-implicit Euler with the new velocities, exponential map of the base rotation
        for (int k = 0; k < 6; k++) s[15 + k] = nu[k];
        for (int k = 0; k < 12; k++) { s[33 + k] = nu[6 + k]; s[21 + k] += dt * nu[6 + k]; }
        for (int k = 0; k < 3; k++) s[k] += dt * nu[k];
        M3 Rn = D.R0;
        const double wn = sqrt(nu[3] * nu[3] + nu[4] * nu[4] + nu[5] * nu[5]);
        if (wn > 0.0) Rn = mul(axis_rotation(v3(nu[3] / wn, nu[4] / wn, nu[5] / wn), wn * dt), D.R0);
        for (int k = 0; k < 9; k++) s[3 + k] = Rn.m[k];
        s[12] = atan2(Rn.m[7], Rn.m[8]);
        s[13] = atan2(-Rn.m[6], sqrt(Rn.m[7] * Rn.m[7] + Rn.m[8] * Rn.m[8]));
        s[14] = atan2(Rn.m[3], Rn.m[0]);
    }
    if (status == 0) {
        bool ok = true;
        for (int k = 0; k < 45; k++) ok = ok && (s[k] - s[k] == 0.0);
        for (int k = 0; k < 12; k++) ok = ok && (fs_out[k] - fs_out[k] == 0.0);
        if (!ok) status = CONTACT_ST_NONFINITE;
    }
    if (status == 0) {
        for (int f = 0; f < 6; f++)
            for (int k = so[f]; k < so[f + 1]; k++) sp[f][(long)(k - so[f]) * ld + i] = s[k];
        for (int k = 0; k < 12; k++) io.foot_force[(long)k * ld + i] = fs_out[k];
    } else {
        for (int k = 0; k < 4; k++) flag_out[k] = 0;
    }
    if (io.contact)
        for (int k = 0; k < 4; k++) io.contact[(long)k * ld + i] = flag_out[k];
    if (io.diag) {
        io.diag[0 * ld + i] = pen;
        io.diag[1 * ld + i] = fzmin < 1.0e300 ? fzmin : 0.0;
        io.diag[2 * ld + i] = kkt;
        io.diag[3 * ld + i] = iters;
    }
    if (io.status) io.status[i] = status;
}

}  // namespace wbc
