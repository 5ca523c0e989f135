// TEST-ONLY host emulation of the device QP solver: compiles the product header
// wbc_quadruped_dob_b200/csrc/qp_warp.cuh with g++ and the single-lane `HostEx` executor so the
// solver's host-visible logic (working-set decisions, phase switching, multiplier update) can be
// unit-tested without a GPU.  It is NOT linked into libwbc_b200.so and is never used by bench.py
// or by the product path; GPU parity tests call the CUDA kernels through the C-ABI instead.
#include "emu_work.h"

#include <cstdlib>
#include <cstring>

using namespace wbcqp;

extern "C" int emu_qp_solve(const double* Q, const double* c, const double* L, int nrows, int neq,
                            double epsx, double rho, int outerits, int kkt_mode, double* x, int* istats,
                            double* dstats)
{
    static thread_local EmuWork ew;
    const Work& w = ew.w;
    for (int i = 0; i < 30; i++)
        for (int j = 0; j < 30; j++) W_H(w)[i * LDH + j] = Q[i * 30 + j];
    memcpy(W_EXB(w), c, 30 * sizeof(double));
    memcpy(W_C(w), L, (size_t)nrows * 31 * sizeof(double));
    Settings cfg;
    cfg.epsx = epsx; cfg.rho = rho; cfg.outerits = outerits; cfg.kkt_mode = kkt_mode;
    Stats st;
    HostEx ex;
    solve_denseaul(ex, w, cfg, nrows, neq, st);
    if (st.termination == 2) memcpy(x, W_XS(w), 30 * sizeof(double));
    if (istats) {
        istats[0] = st.termination; istats[1] = st.ncholesky; istats[2] = st.outer_its; istats[3] = st.qqp_calls;
        istats[4] = st.nicwork; istats[5] = st.kkt_dim_max; istats[6] = st.flags;
    }
    if (dstats) dstats[0] = st.flops;
    return st.termination == 2 ? 0 : -1;
}

// The CPU oracle's QP callback (wbc_qp_fn, oracle/wbc_oracle.h): the reference settings (1e-2, 1e4, 5; lopt.cpp:101, 138) and
// the literal multiplier update (kkt_mode 0), not the reduced form the device code runs by default.  Lets the oracle's control
// cycle run where the reference ALGLIB is not built; this restatement's parity with it is pinned by tests/golden/qp_*.npz.
extern "C" int emu_qp_solve_oracle(const double* Q, const double* c, const double* L, int nrows, int neq,
                                   double* x, int* ncholesky, int* termtype)
{
    int ist[8] = {0};
    int rc = emu_qp_solve(Q, c, L, nrows, neq, 1.0e-2, 1.0e+4, 5, 0, x, ist, nullptr);
    if (ncholesky) *ncholesky = ist[1];
    if (termtype) *termtype = ist[0];
    return rc;
}
