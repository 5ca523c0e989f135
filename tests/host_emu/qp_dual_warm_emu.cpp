// TEST-ONLY host emulation of the exact-mode QP solver's warm start: compiles the product header
// wbc_quadruped_dob_b200/csrc/qp_dual.cuh (solve_dual with WARM = true) with g++ and the single-lane `HostEx` executor, so that
// the warm phase (forced additions, the recomputation of y and u, the drops of negative multipliers) can be unit-tested without a
// GPU.  It is NOT linked into libwbc_b200.so; GPU tests call the CUDA kernels through the C ABI instead.
#include <cstring>
#include <vector>

#include "../../wbc_quadruped_dob_b200/csrc/qp_dual.cuh"

using namespace wbcdual;

// Q [30*30] row-major (lower triangle read), c [30], L [nrows*31]; x [30]; info [8] as qp_info in warm exact mode; flops [1].
// active [3] is read as the warm set (bit r of word r / 32: row r; all zero = a cold start) and overwritten with the final active
// inequality rows (0 on failure); info[6], info[7] are the warm rows added and dropped before the GI loop.  Returns the status word.
extern "C" int emu_qp_dual_solve_warm(const double* Q, const double* c, const double* L, int nrows, int neq, double* x, int* info,
                                      double* flops, unsigned* active)
{
    static thread_local std::vector<double> sm(ds::TOTAL, 0.0), C(SCRATCH_DOUBLES, 0.0);
    double* H = sm.data() + ds::OFF_H;
    for (int i = 0; i < 30; i++)
        for (int j = 0; j < 30; j++) H[i * LD + j] = Q[i * 30 + j];
    memcpy(sm.data() + ds::OFF_CV, c, 30 * sizeof(double));
    memcpy(C.data(), L, (size_t)nrows * 31 * sizeof(double));
    DualStats st;
    HostEx ex;
    const unsigned wset[3] = {active[0], active[1], active[2]};
    WarmStats ws;
    solve_dual<HostEx, false, true>(ex, sm.data(), C.data(), nrows, neq, st, nullptr, wset, &ws);
    memcpy(x, sm.data() + ds::OFF_Y, 30 * sizeof(double));
    if (info) {
        info[0] = st.nfact; info[1] = st.adds; info[2] = st.drops; info[3] = st.nact_ineq; info[4] = st.nact; info[5] = st.flags;
        info[6] = ws.adds; info[7] = ws.drops;
    }
    if (flops) flops[0] = st.flops;
    for (int w = 0; w < 3; w++) active[w] = ws.act[w];
    return st.status;
}
