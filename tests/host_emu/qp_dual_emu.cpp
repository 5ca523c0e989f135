// TEST-ONLY host emulation of the exact-mode QP solver: compiles the product header
// wbc_quadruped_dob_b200/csrc/qp_dual.cuh with g++ and the single-lane `HostEx` executor, so that its
// decisions (additions, drops, dependence and feasibility tests) can be unit-tested without a GPU.  It is NOT
// linked into libwbc_b200.so; GPU tests call the CUDA kernels through the C ABI instead.
#include <cstring>
#include <vector>

#include "../../wbc_quadruped_dob_b200/csrc/qp_dual.cuh"

using namespace wbcdual;

// Q [30*30] row-major (lower triangle read), c [30], L [nrows*31]; x [30]; info [8] as qp_info in exact mode; flops [1].
// Returns the status word.
extern "C" int emu_qp_dual_solve(const double* Q, const double* c, const double* L, int nrows, int neq, double* x, int* info,
                                 double* flops)
{
    static thread_local std::vector<double> sm(ds::TOTAL, 0.0), C(SCRATCH_DOUBLES, 0.0);
    double* H = sm.data() + ds::OFF_H;
    for (int i = 0; i < 30; i++)
        for (int j = 0; j < 30; j++) H[i * LD + j] = Q[i * 30 + j];
    memcpy(sm.data() + ds::OFF_CV, c, 30 * sizeof(double));
    memcpy(C.data(), L, (size_t)nrows * 31 * sizeof(double));
    DualStats st;
    HostEx ex;
    solve_dual(ex, sm.data(), C.data(), nrows, neq, st);
    memcpy(x, sm.data() + ds::OFF_Y, 30 * sizeof(double));
    if (info) {
        info[0] = st.nfact; info[1] = st.adds; info[2] = st.drops; info[3] = st.nact_ineq; info[4] = st.nact; info[5] = st.flags;
        info[6] = 0; info[7] = 0;
    }
    if (flops) flops[0] = st.flops;
    return st.status;
}

// The exact solver as the live oracle's QP callback (wbc_qp_fn, oracle/wbc_oracle.h).
extern "C" int emu_qp_dual_oracle(const double* Q, const double* c, const double* L, int nrows, int neq, double* x, int* ncholesky,
                                  int* termtype)
{
    int info[8];
    const int rc = emu_qp_dual_solve(Q, c, L, nrows, neq, x, info, nullptr);
    if (ncholesky) *ncholesky = info[0];
    if (termtype) *termtype = rc == 0 ? 2 : rc;
    return rc == 0 ? 0 : -1;
}
