// Exact QP mode: a Goldfarb-Idnani dual active-set solver (Goldfarb & Idnani, Math. Programming 27, 1983; the update
// formulas of quadprog / eiquadprog) for the OPT operator's QP
//     minimise 0.5 x'Hx + c'x   subject to   a_i.x = b_i (i < neq),   a_i.x <= b_i (neq <= i < nrows),
// H the lower triangle of Q mirrored (the rule of the DENSE-AUL path).  Unlike DENSE-AUL at the reference's settings, it
// stops at the optimum: every inactive row feasible on its row-scaled residual, every active inequality multiplier >= 0.
//
// Execution model: one warp per QP, like qp_warp.cuh and written against the same executors (WarpEx on the device, HostEx for
// the g++ build of tests/host_emu).  Lane i owns row i of the factor J = L^-T Q (G = L L', 30 registers); the upper
// triangular R (J' N = [R; 0] for the active normals N), the vectors and the active-row list live in shared memory (dual::
// layout below); the constraint matrix [nrows][31] stays in the warp's global scratch where the assembly or the dense
// path put it, and is scaled in place.
//
// A row joins the active set through one Householder reflection of J's null-space columns, and leaves it through Givens
// rotations of R and J (eiquadprog uses rotations for both).
//
// Numerics:
//   * scaled variables y = x / s, s_i = 1/sqrt(H_ii) (the swing slack weight is 1e8), every constraint row normalised in
//     the scaled variables; x = s y is returned;
//   * equalities first; an equality that depends on those already active (|d2| <= TOL_DEP |d|) is skipped when its
//     residual is within the feasibility tolerance and reports WBC_ST_INFEASIBLE otherwise;
//   * a violated row whose normal depends on the active set (a degenerate vertex: e.g. the 5 friction rows of an unloaded foot
//     through one point of its 3 force components) is never added: the method takes dual steps, dropping active rows,
//     until it is independent -- or reports WBC_ST_INFEASIBLE when no row can be dropped.  Before any such step, a dependent
//     row that the active rows imply is met (n = sum r_k n_k and b - sum r_k b_k within the feasibility tolerance), and that
//     is violated only by rounding (TOL_HOLD), is held out of the search until the next drop: with mu = 0 each tangential
//     friction row comes with its negation, and the second of a pair must not end the solve;
//   * iterations (one per d = J'n evaluation) are capped at 2 nrows + 30; an overrun returns -100.
// A failed solve returns x = 0.
#pragma once
#include "qp_warp.cuh"

namespace wbcdual {

using wbcqp::HostEx;
constexpr int N = 30;
constexpr int LD = 31;
constexpr int MAXROWS = 88;
constexpr double TOL_DEP = 1.0e-10;     // |d2| <= TOL_DEP |d|: the row is a combination of the active rows
constexpr double TOL_FEAS = 1.0e-12;    // row-scaled residual counted as feasible (relative to max(1, |b|, sum |a_j y_j|))
constexpr double TOL_PIV = 1.0e-14;     // Cholesky pivot of the unit-diagonal scaled H below which H is not positive definite
constexpr double TOL_HOLD = 1.0e-9;     // row-scaled violation up to which a dependent, consistent row counts as rounding

// status (include/wbc_b200.h)
constexpr int ST_OK = 0;
constexpr int ST_INFEASIBLE = -22;
constexpr int ST_NOT_PD = -23;
constexpr int ST_ITERATIONS = -100;
// flags (qp_info[5])
constexpr int FL_EXACT = 256;           // set on every exact-mode result (no DENSE-AUL path uses this bit)
constexpr int FL_DEP_EQ = 512;          // a dependent, consistent equality row was skipped
constexpr int FL_DUAL_STEP = 1024;      // a violated row depended on the active set: pure dual steps were taken
constexpr int FL_DEP_HELD = 4096;       // a violated, dependent, consistent inequality row was held out (rounding)

// shared-memory layout of one warp (doubles)
namespace ds {
constexpr int OFF_R = 0;                 // [30][31] R (column k: active row k); the QP record is staged here around a solve
constexpr int OFF_H = OFF_R + N * LD;    // [30][31] H, then its Cholesky factor; afterwards the products J' v
constexpr int OFF_Y = OFF_H + N * LD;    // [32] the point (scaled), at the end x
constexpr int OFF_CV = OFF_Y + 32;       // [32] linear term c
constexpr int OFF_SC = OFF_CV + 32;      // [32] variable scales s_i; 1 / L_ii during the factorisation
constexpr int OFF_D = OFF_SC + 32;       // [32] d = J' n
constexpr int OFF_NP = OFF_D + 32;       // [32] n = -a of the row being added
constexpr int OFF_U = OFF_NP + 32;       // [32] multipliers of the active rows, then of the row being added
constexpr int OFF_RV = OFF_U + 32;       // [32] r = R^-1 d1
constexpr int OFF_RDI = OFF_RV + 32;     // [32] 1 / R_kk
constexpr int OFF_CS = OFF_RDI + 32;     // [32] Givens cosines of a drop
constexpr int OFF_SN = OFF_CS + 32;      // [32] ... and sines
constexpr int OFF_A = OFF_SN + 32;       // ints [32]: the active rows, in R's column order
constexpr int TOTAL = OFF_A + 16;
constexpr int BYTES = TOTAL * 8;
static_assert(OFF_Y % 2 == 0, "alignment");
}  // namespace ds
// global scratch of one warp: the constraint matrix
constexpr int SCRATCH_DOUBLES = MAXROWS * LD + 8;   // 2736

struct DualStats {
    int status;      // ST_*
    int nfact;       // factorisations (1, or 0 when H has a non-positive diagonal)
    int adds;        // rows added to the active set (equalities included)
    int drops;       // rows dropped
    int nact_ineq;   // active inequality rows at the end
    int nact;        // active-set size at the end
    int flags;       // FL_*
    double flops;    // instrumented algorithmic flop count
};
// What a caller that keeps active sets needs besides DualStats (solve_dual's `ws`, may be NULL)
struct WarmStats {
    int adds;        // warm start (WARM = true): rows of the warm set added before the GI loop ...
    int drops;       // ... and dropped again for a negative multiplier before it
    unsigned act[3]; // active inequality rows at the end (bit r: row r); 0 on failure
};

// Per-phase cycle counters of a solve (the kernel's profiled instantiation, PROF = true; see solve_dual).  Slots 0 and 8 are the
// kernel's (record staging, validation and assembly; torque map and outputs).
enum { PH_ASSEMBLE = 0, PH_SETUP, PH_SWEEP, PH_D, PH_ZR, PH_STEP, PH_ADD, PH_DROP, PH_OUTPUT, NPH };
WBC_HD long long dual_clock()
{
#if defined(__CUDA_ARCH__)
    return clock64();
#else
    return 0;
#endif
}

// index of the lowest set bit (b != 0)
WBC_HD int low_bit(unsigned b)
{
#if defined(__CUDA_ARCH__)
    return __ffs((int)b) - 1;
#else
    return __builtin_ctz(b);
#endif
}

template <class Ex>
struct Rows { static constexpr int RPL = (N + Ex::NL - 1) / Ex::NL; };   // rows of J per lane

// v_out[j] = sum_i J[i][j] v[i]  (J' v): each lane writes its rows' products, then sums columns.  P: [30][31] scratch.
template <class Ex>
WBC_HD void jt_times(const Ex& ex, const double (&J)[Rows<Ex>::RPL][N], const double* v, double* P, double* out)
{
    constexpr int RPL = Rows<Ex>::RPL;
#pragma unroll
    for (int q = 0; q < RPL; q++) {
        const int i = ex.lane() + q * Ex::NL;
        if (i < N) {
            const double vi = v[i];
#pragma unroll
            for (int j = 0; j < N; j++) P[i * LD + j] = J[q][j] * vi;
        }
    }
    ex.sync();
    for (int j = ex.lane(); j < N; j += Ex::NL) {
        double s = 0.0;
#pragma unroll 10
        for (int i = 0; i < N; i++) s += P[i * LD + j];
        out[j] = s;
    }
    ex.sync();
}

// the most violated inequality row not in the active set: (violation / tolerance-normalised value, row), or (0, -1)
template <class Ex>
WBC_HD int most_violated(const Ex& ex, const double* C, const double* y, int nrows, int neq, const unsigned (&act)[3])
{
    double best = 0.0;
    int bi = -1;
    for (int r = neq + ex.lane(); r < nrows; r += Ex::NL) {
        if ((act[r >> 5] >> (r & 31)) & 1u) continue;
        const double* a = C + r * LD;
        double s = 0.0, m = 0.0;
#pragma unroll 10
        for (int j = 0; j < N; j++) { const double t = a[j] * y[j]; s += t; m += fabs(t); }
        const double b = a[N];
        const double v = s - b;                                   // > 0: violated
        const double tol = TOL_FEAS * fmax(1.0, fmax(fabs(b), m));
        if (v > tol) {
            const double sv = v / fmax(1.0, fabs(b));             // the row-scaled residual picks the row
            if (sv > best) { best = sv; bi = r; }
        }
    }
    const double vmax = wbcqp::red_max1(ex, best);
    if (!(vmax > 0.0)) return -1;
    const double cand = (best == vmax && bi >= 0) ? -(double)bi : -1.0e9;
    return (int)(-wbcqp::red_max1(ex, cand));                    // lowest row index among the ties
}

// n . y + b for the row in NP (n = -a): the constraint value, >= 0 when feasible, and its tolerance
template <class Ex>
WBC_HD double row_value(const Ex& ex, const double* np, const double* y, double b, double* tol)
{
    double p[2] = {0.0, 0.0};
    for (int k = ex.lane(); k < N; k += Ex::NL) { const double t = np[k] * y[k]; p[0] += t; p[1] += fabs(t); }
    wbcqp::red_sum<2>(ex, p);
    *tol = TOL_FEAS * fmax(1.0, fmax(fabs(b), p[1]));
    return p[0] + b;
}

// Solve.  On entry: sm + OFF_H holds Q (lower triangle read, ld 31), sm + OFF_CV holds c, C holds [nrows][31] = [a | b].
// On exit: sm + OFF_Y holds x (0 on failure); C and the rest of the shared block are overwritten.
// PROF = true adds the SM cycles spent in each phase to pc[PH_*] (measurement only; the shipped path is PROF = false).
//
// ws (may be NULL) receives the final active inequality rows, and the warm phase's counters.
// WARM = true: warm start from the inequality rows of `wset` (bit r: row r; a guess -- bits at equality rows, at rows >= nrows and
// at rows that depend on those already active are skipped).  After the equalities, the rows of wset are added in ascending order
// without steps (d = J'n, the dependence test, add_row); then the point and the multipliers of that active set are recomputed from
// the factorisation, and the most negative inequality multiplier is dropped until none is negative.  That leaves the GI loop a
// valid start: linearly independent active rows, y optimal with them held as equalities, every inequality multiplier >= 0.
// The warm phase is bounded by the size of wset and does not count against the iteration cap; its time goes to PH_D, PH_ADD,
// PH_ZR (the recomputation) and PH_DROP.  WARM = false compiles to the cold solver.
//
// The factorisation is not qp_warp.cuh's chol_cols / tri_solve: those work on DENSE-AUL's packed, transposed factor (with its
// column-dependency and ambiguity tests for rank-deficient working sets), whereas here H is positive definite or the solve stops,
// and the factor is only read once more -- row by row, with ld 31, by every lane forming its own row of J = L^-T in registers.
template <class Ex, bool PROF = false, bool WARM = false>
WBC_HDN void solve_dual(const Ex& ex, double* sm, double* C, int nrows, int neq, DualStats& st, unsigned long long* pc = nullptr,
                        const unsigned* wset = nullptr, WarmStats* ws = nullptr)
{
    long long tmark = PROF ? dual_clock() : 0;
    auto mark = [&](int k) {
        if constexpr (PROF) {
            const long long t = dual_clock();
            pc[k] += (unsigned long long)(t - tmark);
            tmark = t;
        }
    };
    constexpr int RPL = Rows<Ex>::RPL;
    const int lane = ex.lane();
    double* R = sm + ds::OFF_R;
    double* H = sm + ds::OFF_H;
    double* Y = sm + ds::OFF_Y;
    double* CV = sm + ds::OFF_CV;
    double* SC = sm + ds::OFF_SC;
    double* D = sm + ds::OFF_D;
    double* NP = sm + ds::OFF_NP;
    double* U = sm + ds::OFF_U;
    double* RV = sm + ds::OFF_RV;
    double* RDI = sm + ds::OFF_RDI;
    double* CS = sm + ds::OFF_CS;
    double* SN = sm + ds::OFF_SN;
    int* A = reinterpret_cast<int*>(sm + ds::OFF_A);
    st.status = ST_OK; st.nfact = 0; st.adds = 0; st.drops = 0; st.nact_ineq = 0; st.nact = 0; st.flags = FL_EXACT; st.flops = 0.0;
    if (ws) { ws->adds = 0; ws->drops = 0; ws->act[0] = 0u; ws->act[1] = 0u; ws->act[2] = 0u; }
    double flops = 0.0;

    // ---- scaling: s_i = 1 / sqrt(H_ii); H <- S H S, c <- S c, rows a <- a S / |a S|, b <- b / |a S|
    double bad = 0.0;
    for (int i = lane; i < N; i += Ex::NL) {
        const double h = H[i * LD + i];
        SC[i] = h > 0.0 ? 1.0 / sqrt(h) : 0.0;
        if (!(h > 0.0)) bad = 1.0;
    }
    bad = wbcqp::red_max1(ex, bad);
    ex.sync();
    if (bad > 0.0) {
        for (int k = lane; k < N; k += Ex::NL) Y[k] = 0.0;
        ex.sync();
        st.status = ST_NOT_PD;
        return;
    }
    for (int i = lane; i < N; i += Ex::NL) {
        for (int j = 0; j <= i; j++) H[i * LD + j] *= SC[i] * SC[j];
        CV[i] *= SC[i];
    }
    for (int r = lane; r < nrows; r += Ex::NL) {
        double* a = C + r * LD;
        double s = 0.0;
        for (int j = 0; j < N; j++) { const double v = a[j] * SC[j]; a[j] = v; s += v * v; }
        if (s > 0.0) {
            const double inv = 1.0 / sqrt(s);
            for (int j = 0; j <= N; j++) a[j] *= inv;
        }
    }
    ex.sync();
    flops += 2.0 * 465 + 30 + 3.0 * 31 * nrows;

    // ---- Cholesky H = L L' in place (lower triangle; lane i computes row i), 1 / L_jj in RDI until J is formed
    st.nfact = 1;
    for (int j = 0; j < N; j++) {
        double dj = H[j * LD + j];
        for (int k = 0; k < j; k++) dj -= H[j * LD + k] * H[j * LD + k];
        if (!(dj > TOL_PIV)) { bad = 1.0; break; }
        const double rinv = 1.0 / sqrt(dj);
        for (int i = lane; i < N; i += Ex::NL)
            if (i > j) {
                double v = H[i * LD + j];
                for (int k = 0; k < j; k++) v -= H[i * LD + k] * H[j * LD + k];
                H[i * LD + j] = v * rinv;
            }
        if (lane == 0) RDI[j] = rinv;
        ex.sync();
    }
    flops += 9455.0;        // sum over j of 2j + (29 - j)(2j + 2): the n^3/3 of a 30 x 30 factorisation
    if (bad > 0.0) {
        for (int k = lane; k < N; k += Ex::NL) Y[k] = 0.0;
        ex.sync();
        st.status = ST_NOT_PD;
        st.flops = flops;
        return;
    }
    // ---- J = L^-T: row i of J solves L v = e_i (zero before i)
    double J[RPL][N];
#pragma unroll
    for (int q = 0; q < RPL; q++) {
        const int i = lane + q * Ex::NL;
#pragma unroll
        for (int j = 0; j < N; j++) {
            double s = (j == i) ? 1.0 : 0.0;
#pragma unroll
            for (int k = 0; k < j; k++) s -= H[j * LD + k] * J[q][k];
            J[q][j] = s * RDI[j];
        }
    }
    ex.sync();
    flops += 8990.0;
    // ---- unconstrained minimiser y = -J J' c
    jt_times(ex, J, CV, H, D);
#pragma unroll
    for (int q = 0; q < RPL; q++) {
        const int i = lane + q * Ex::NL;
        if (i < N) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < N; j++) s += J[q][j] * D[j];
            Y[i] = -s;
        }
    }
    for (int k = lane; k < 32; k += Ex::NL) { U[k] = 0.0; RV[k] = 0.0; A[k] = -1; }
    for (int k = lane; k < N * LD; k += Ex::NL) R[k] = 0.0;
    ex.sync();
    flops += 3600.0;
    mark(PH_SETUP);

    int iq = 0;                        // active rows
    int peq = 0;                       // of which equalities (positions [0, peq))
    unsigned act[3] = {0u, 0u, 0u};    // active inequality rows (bit mask, uniform)
    unsigned held[3] = {0u, 0u, 0u};   // dependent, consistent rows held out of the search until the next drop (uniform)
    double z[RPL];
    int warm_adds = 0, warm_drops = 0;

    // d = J' n, |d2|^2 = sum_{j >= iq} d_j^2 and |d|^2 (uniform)
    auto compute_d = [&](double& nd2, double& nd) {
        jt_times(ex, J, NP, H, D);
        nd2 = 0.0; nd = 0.0;
        for (int j = 0; j < N; j++) { const double v = D[j] * D[j]; nd += v; if (j >= iq) nd2 += v; }
        flops += 1800.0 + 60.0;
    };
    // z = J2 d2 (this lane's rows)
    auto compute_z = [&]() {
#pragma unroll
        for (int q = 0; q < RPL; q++) {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < N; j++) s += (j >= iq) ? J[q][j] * D[j] : 0.0;
            z[q] = s;
        }
        flops += 2.0 * N * (N - iq);
    };
    // r = R^-1 d1 by columns (RV[k] keeps the partial right-hand side until the final scaling)
    auto compute_r = [&]() {
        for (int k = lane; k < iq; k += Ex::NL) RV[k] = D[k];
        ex.sync();
        for (int k = iq - 1; k > 0; k--) {
            const double rk = RV[k] * RDI[k];
            ex.sync();
            for (int i = lane; i < k; i += Ex::NL) RV[i] -= R[i * LD + k] * rk;
            ex.sync();
        }
        for (int k = lane; k < iq; k += Ex::NL) RV[k] *= RDI[k];
        ex.sync();
        flops += (double)iq * iq;
    };
    // y += t z
    auto step_y = [&](double t) {
#pragma unroll
        for (int q = 0; q < RPL; q++) {
            const int i = lane + q * Ex::NL;
            if (i < N) Y[i] += t * z[q];
        }
        ex.sync();
        flops += 2.0 * N;
    };
    // u_k -= t r_k (k < iq), u_iq += t
    auto step_u = [&](double t) {
        for (int k = lane; k <= iq; k += Ex::NL) U[k] = (k < iq) ? U[k] - t * RV[k] : U[k] + t;
        ex.sync();
        flops += 2.0 * iq;
    };
    // append the row in D's direction: rotate d[iq..29] onto d[iq] (J columns alike), R column iq = d[0..iq]
    // append the row in D's direction: one Householder reflection P = I - beta v v' on columns iq..29 folds d2 = d[iq..29] onto
    // d[iq] = alpha = -sign(d_iq) |d2| (J2 <- J2 P, so that J'n stays d with d2 folded); R column iq = (d[0..iq-1], alpha).
    // nd2 = |d2|^2 from compute_d.  (A chain of Givens rotations does the same with up to 29 dependent rotations, each with FP64
    // divisions and a square root: measured 64 % of the solve at trot_65536, DESIGN.md 4.7.)  Each lane updates its own rows.
    auto add_row = [&](int row, double nd2) {
        const double dq = D[iq];
        const double nrm = sqrt(nd2);
        const double alpha = dq >= 0.0 ? -nrm : nrm;
        const double viq = dq - alpha;                       // v = d2 - alpha e_iq, v'v = 2 |d2| (|d2| + |d_iq|)
        const double beta = 1.0 / (nrm * (nrm + fabs(dq)));   // 2 / v'v
#pragma unroll
        for (int q = 0; q < RPL; q++) {
            double w = 0.0;
#pragma unroll
            for (int j = 0; j < N; j++)
                if (j >= iq) w += J[q][j] * (j == iq ? viq : D[j]);
            w *= beta;
#pragma unroll
            for (int j = 0; j < N; j++)
                if (j >= iq) J[q][j] -= w * (j == iq ? viq : D[j]);
        }
        for (int k = lane; k <= iq; k += Ex::NL) R[k * LD + iq] = (k < iq) ? D[k] : alpha;
        ex.sync();
        if (lane == 0) { RDI[iq] = 1.0 / alpha; A[iq] = row; }
        if (row >= neq) act[row >> 5] |= 1u << (row & 31);
        iq++;
        st.adds++;
        ex.sync();
        flops += 4.0 * N * (N - (iq - 1)) + 10.0;
    };
    // drop the active row at position kp (>= peq); the multiplier of the row being added (position iq) moves down with it
    auto drop_at = [&](int kp) {
        const int row = A[kp];
        ex.sync();
        for (int i = lane; i < N; i += Ex::NL) {
            for (int k = kp; k < iq - 1; k++) R[i * LD + k] = R[i * LD + k + 1];
            R[i * LD + iq - 1] = 0.0;
        }
        if (lane == 0) {
            for (int k = kp; k < iq; k++) { A[k] = A[k + 1]; U[k] = U[k + 1]; }
            A[iq] = -1; U[iq] = 0.0;
        }
        act[row >> 5] &= ~(1u << (row & 31));
        held[0] = 0u; held[1] = 0u; held[2] = 0u;
        iq--;
        st.drops++;
        ex.sync();
        // R is upper Hessenberg from column kp on: rotate rows j, j+1 to zero R[j+1][j]
        for (int j = kp; j < iq; j++) {
            const double f = R[j * LD + j], g = R[(j + 1) * LD + j];
            double cs, sn, rr;
            wbcqp::generaterotation(f, g, cs, sn, rr);
            ex.sync();
            for (int k = j + 1 + lane; k < iq; k += Ex::NL) {
                const double t1 = R[j * LD + k], t2 = R[(j + 1) * LD + k];
                R[j * LD + k] = cs * t1 + sn * t2;
                R[(j + 1) * LD + k] = cs * t2 - sn * t1;
            }
            if (lane == 0) {
                R[j * LD + j] = rr; R[(j + 1) * LD + j] = 0.0;
                RDI[j] = 1.0 / rr;
                CS[j] = cs; SN[j] = sn;
            }
            ex.sync();
            flops += 6.0 * (iq - j) + 6.0 * N;
        }
        if (kp < iq) {
#pragma unroll
            for (int j = 0; j < N - 1; j++) {
                if (j >= kp && j < iq) {
                    const double cs = CS[j], sn = SN[j];
#pragma unroll
                    for (int q = 0; q < RPL; q++) {
                        const double t1 = J[q][j], t2 = J[q][j + 1];
                        J[q][j] = cs * t1 + sn * t2;
                        J[q][j + 1] = cs * t2 - sn * t1;
                    }
                }
            }
        }
    };
    auto load_row = [&](int row) {      // NP = -a of the row, and its b
        for (int k = lane; k < N; k += Ex::NL) NP[k] = -C[row * LD + k];
        ex.sync();
        return C[row * LD + N];
    };

    const int maxit = 2 * nrows + 30;
    int iters = 0;
    // ---- equalities
    for (int e = 0; e < neq && st.status == ST_OK; e++) {
        const double b = load_row(e);
        double tol;
        const double s = row_value(ex, NP, Y, b, &tol);
        double nd2, nd;
        compute_d(nd2, nd);
        mark(PH_D);
        if (nd2 <= TOL_DEP * TOL_DEP * nd) {
            if (fabs(s) <= tol) { st.flags |= FL_DEP_EQ; continue; }
            st.status = ST_INFEASIBLE;
            break;
        }
        compute_z();
        compute_r();
        mark(PH_ZR);
        const double t = -s / nd2;
        step_y(t);
        for (int k = lane; k <= iq; k += Ex::NL) U[k] = (k < iq) ? U[k] - t * RV[k] : t;
        ex.sync();
        mark(PH_STEP);
        add_row(e, nd2);
        mark(PH_ADD);
        peq = iq;
    }
    if constexpr (WARM) {
        // ---- warm start: force the rows of wset into the active set (no steps), then recompute y and u for that set.  With
        // b'_k = -b of active row k (N'y = b' on the active rows), J = [J1 J2], J1'N = R and J2'N = 0:
        //     y = J1 R^-T b' - J2 J2' c,      u = R^-1 (R^-T b' + J1' c).
        // NP holds b', then w = R^-T b'; D holds J' c, then w + J1' c.
        auto fwd = [&]() {                               // NP <- R^-T NP, forward by columns of R
            for (int k = 0; k < iq; k++) {
                const double wk = NP[k] * RDI[k];
                ex.sync();
                for (int i = k + 1 + lane; i < iq; i += Ex::NL) NP[i] -= R[k * LD + i] * wk;
                if (lane == 0) NP[k] = wk;
                ex.sync();
            }
        };
        auto recompute = [&]() {
            for (int k = lane; k < iq; k += Ex::NL) NP[k] = -C[A[k] * LD + N];
            ex.sync();
            fwd();
            jt_times(ex, J, CV, H, D);
#pragma unroll
            for (int q = 0; q < RPL; q++) {
                const int i = lane + q * Ex::NL;
                if (i < N) {
                    double s = 0.0;
#pragma unroll
                    for (int j = 0; j < N; j++) s += (j < iq) ? J[q][j] * NP[j] : -(J[q][j] * D[j]);
                    Y[i] = s;
                }
            }
            for (int k = lane; k < iq; k += Ex::NL) D[k] += NP[k];
            ex.sync();
            // one refinement of y on the active rows' residuals b' - N'y = a.y - b (y += J1 R^-T r): the forced rows meet at
            // degenerate vertices, where a residual left by the cancellation in J1 w - J2 J2' c would show a row through the
            // vertex as violated and cost the GI loop a dual step
            for (int k = lane; k < iq; k += Ex::NL) {
                const double* a = C + A[k] * LD;
                double s = -a[N];
                for (int j = 0; j < N; j++) s += a[j] * Y[j];
                NP[k] = s;
            }
            ex.sync();
            fwd();
#pragma unroll
            for (int q = 0; q < RPL; q++) {
                const int i = lane + q * Ex::NL;
                if (i < N) {
                    double s = 0.0;
#pragma unroll
                    for (int j = 0; j < N; j++) s += (j < iq) ? J[q][j] * NP[j] : 0.0;
                    Y[i] += s;
                }
            }
            ex.sync();
            compute_r();
            for (int k = lane; k < 32; k += Ex::NL) U[k] = (k < iq) ? RV[k] : 0.0;
            ex.sync();
            flops += 3.0 * iq * iq + 1800.0 + 2.0 * N * N + 4.0 * N * iq;
        };
        if (st.status == ST_OK && wset) {
#pragma unroll 1
            for (int w = 0; w < 3; w++) {
                unsigned bits = wset[w];
                while (bits) {
                    const int row = 32 * w + low_bit(bits);
                    bits &= bits - 1u;
                    if (row < neq || row >= nrows) continue;
                    load_row(row);
                    double nd2, nd;
                    compute_d(nd2, nd);
                    mark(PH_D);
                    if (nd2 <= TOL_DEP * TOL_DEP * nd) continue;     // depends on the active rows (or 30 are active)
                    add_row(row, nd2);
                    mark(PH_ADD);
                    warm_adds++;
                }
            }
            while (warm_adds > 0) {
                recompute();
                mark(PH_ZR);
                double umin = 0.0;
                int kp = -1;
                for (int k = peq; k < iq; k++)
                    if (U[k] < umin) { umin = U[k]; kp = k; }
                if (kp < 0) break;
                drop_at(kp);
                warm_drops++;
                mark(PH_DROP);
            }
        }
    }
    // ---- inequalities
    while (st.status == ST_OK) {
        const unsigned skip[3] = {act[0] | held[0], act[1] | held[1], act[2] | held[2]};
        const int ip = most_violated(ex, C, Y, nrows, neq, skip);
        flops += 2.0 * N * (nrows - neq);
        mark(PH_SWEEP);
        if (ip < 0) break;                                   // every row feasible: optimal
        const double b = load_row(ip);
        double tol;
        double s = row_value(ex, NP, Y, b, &tol);
        if (lane == 0) U[iq] = 0.0;
        ex.sync();
        mark(PH_D);
        for (bool first = true;; first = false) {
            if (++iters > maxit) { st.status = ST_ITERATIONS; break; }
            double nd2, nd;
            compute_d(nd2, nd);
            mark(PH_D);
            const bool dep = nd2 <= TOL_DEP * TOL_DEP * nd;
            if (!dep) compute_z();
            compute_r();
            mark(PH_ZR);
            if (dep && first) {
                // where the active rows hold (n_k.y = -b_k), n.y + b = b - sum r_k b_k: the row is implied, not violated
                double p[2] = {0.0, 0.0};
                for (int k = lane; k < iq; k += Ex::NL) { const double t = RV[k] * C[A[k] * LD + N]; p[0] += t; p[1] += fabs(t); }
                wbcqp::red_sum<2>(ex, p);
                if (b - p[0] >= -TOL_FEAS * fmax(1.0, fabs(b) + p[1]) && s >= -(TOL_HOLD / TOL_FEAS) * tol) {
                    held[ip >> 5] |= 1u << (ip & 31);
                    st.flags |= FL_DEP_HELD;
                    break;
                }
            }
            // dual step length t1: the first active inequality multiplier to reach zero
            double t1 = 1.0e300;
            int kp = -1;
            for (int k = peq; k < iq; k++)
                if (RV[k] > 0.0 && U[k] / RV[k] < t1) { t1 = U[k] / RV[k]; kp = k; }
            // primal step length t2: onto the row
            const double t2 = dep ? 1.0e300 : -s / nd2;
            if (kp < 0 && dep) { st.status = ST_INFEASIBLE; break; }
            if (dep) {
                st.flags |= FL_DUAL_STEP;
                step_u(t1);
                mark(PH_STEP);
                drop_at(kp);
                mark(PH_DROP);
                continue;
            }
            const double t = t2 <= t1 ? t2 : t1;
            step_y(t);
            step_u(t);
            mark(PH_STEP);
            if (t2 <= t1) {
                add_row(ip, nd2);
                mark(PH_ADD);
                break;
            }
            drop_at(kp);
            mark(PH_DROP);
            s = row_value(ex, NP, Y, b, &tol);
            mark(PH_D);
        }
    }
    // ---- result: x = S y
    for (int i = lane; i < N; i += Ex::NL) Y[i] = (st.status == ST_OK) ? Y[i] * SC[i] : 0.0;
    ex.sync();
    st.nact = iq;
    st.nact_ineq = iq - peq;
    st.flops = flops;
    if (ws) {
        ws->adds = warm_adds; ws->drops = warm_drops;
        for (int w = 0; w < 3; w++) ws->act[w] = (st.status == ST_OK) ? act[w] : 0u;
    }
    mark(PH_STEP);
}

}  // namespace wbcdual
