// libwbc_b200.so -- sm_100a kernels and the C ABI (include/wbc_b200.h) of the batched WBC control cycle.
//
// Two kernels per cycle, no intermediate dense QP ever reaches HBM:
//   wbc_front_kernel   thread-per-instance: update() + Fgrf + estimate() + Wcom_des -> 4.2 KB QP record
//   wbc_solve_kernel   warp-per-instance, one warp per CTA, 12 resident CTAs per SM (18.3 KB of shared memory and 168
//                      registers each), persistent warps pulling instances from an atomic queue (iteration counts vary
//                      4..50 Cholesky per solve): assemble (Q,c,L) from the record, DENSE-AUL/QQP solve with the
//                      hot state in shared memory (qp_warp.cuh), torque map.
//   wbc_solve_exact_kernel  (WBC_QP_EXACT) in place of wbc_solve_kernel: the same warp-per-instance persistent shape around the
//                      Goldfarb-Idnani dual active-set solver of qp_dual.cuh (the exact optimum of each QP); its WARM
//                      instantiation (WBC_QP_WARM) starts each instance from the active set of its previous exact-mode cycle.
// There is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <stddef.h>
#include <stdlib.h>

#include <new>

#include "../../include/wbc_b200.h"
#include "qp_warp.cuh"
#include "qp_dual.cuh"
#include "wbc_assemble.cuh"
#include "wbc_contact.cuh"
#include "wbc_front.cuh"
#include "wbc_front_leg.cuh"
#include "wbc_gait.cuh"
#include "wbc_traj.cuh"
#include "wbc_types.h"

using namespace wbc;
using namespace wbcqp;

static_assert(sizeof(wbc_params) == sizeof(wbc::Params), "wbc_params and wbc::Params must have identical layout");

constexpr int SOLVE_T = 32;                   // one warp per instance, one warp per CTA
// resident solver CTAs per SM that the shared-memory request allows (228 KB per SM, 1 KB reserved per CTA); the launch
// shape takes the occupancy calculator's answer, which also accounts for registers
constexpr int SOLVE_CTAS_PER_SM = (228 * 1024) / (sl::BYTES + 1024);

// ------------------------------------------------------------------------------------------------
// kernels
// ---- longest-first dispatch of the solver's work queue.
// A solve takes 4..50 Cholesky factorisations, i.e. its duration varies ~10x between instances, and a batch of a few
// thousand instances is only a few waves of the resident warps: with first-come dispatch the step ends when the
// longest solve that happened to start late finishes (measured: 4096 instances take 1.5x their share of the
// steady-state rate).  Consecutive control cycles of one robot are 2.5 ms apart and hit nearly the same active set,
// so the duration of an instance's previous solve predicts this one: the solve kernel records each instance's cycle
// count and a histogram of it, and the NEXT cycle's front kernel turns them into a dispatch order, longest first
// (a counting sort: bucket bases from the histogram, one atomic per instance).  Results do not depend on the order.
constexpr int ORD_NB = 256;                   // cost buckets of 65536 cycles (cost unit = 1024 cycles)
struct DispatchOrder {
    const unsigned* cost;     // [n] duration of the previous solve of instance i, 1024-cycle units (NULL: keep ticket order)
    const int* hist;          // [ORD_NB] histogram of bucket(cost) over the n instances
    int* cursor;              // [ORD_NB] zeroed
    int* order;               // [n] out: instance index per ticket
    int* lanes;               // express-lane block of the solve launch that follows (ExpressLanes below), zeroed here; may be NULL
};
constexpr int LANES_INTS = 2 + 256;           // head ticket counter, tail ticket counter, arrivals per SM
__device__ __forceinline__ int cost_bucket(unsigned cost) { const unsigned b = cost >> 6; return b < ORD_NB ? (int)b : ORD_NB - 1; }

// (stage_reset: the staged solver's queue block and rings, reset here for the solve launch that follows; see StageCtl below)
struct StageReset { int* ctl; int nctl; int free_tail_index; int free_avail_index; int* ring; int rsize; int nslots; };

__global__ void __launch_bounds__(64) wbc_front_kernel(Params P, DevInputs in, FrontState st, int n, double* __restrict__ recs,
                                                       double* __restrict__ w_out, long w_ld, DevDebug dbg, int has_dbg, DispatchOrder ord,
                                                       StageReset sr)
{
    __shared__ int base[ORD_NB];
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (sr.ctl) {
        const long nth = (long)gridDim.x * blockDim.x;
        for (long k = i; k < sr.nctl; k += nth) sr.ctl[k] = (k == sr.free_tail_index || k == sr.free_avail_index) ? sr.nslots : 0;
        for (long k = i; k < 3L * sr.rsize; k += nth) sr.ring[k] = (k >= 2L * sr.rsize && k - 2L * sr.rsize < sr.nslots) ? (int)(k - 2L * sr.rsize) : -1;
    }
    if (ord.lanes) {
        const long nth = (long)gridDim.x * blockDim.x;
        for (long k = i; k < LANES_INTS; k += nth) ord.lanes[k] = 0;
    }
    if (ord.cost) {
        // base[b] = number of instances in costlier buckets: lane l scans buckets 255-8l .. 248-8l
        if (threadIdx.x < 32) {
            const int l = threadIdx.x;
            int h[8], sum = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) { h[k] = ord.hist[ORD_NB - 1 - (8 * l + k)]; sum += h[k]; }
            int incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (l >= o) incl += t; }
            int run = incl - sum;
#pragma unroll
            for (int k = 0; k < 8; k++) { base[ORD_NB - 1 - (8 * l + k)] = run; run += h[k]; }
        }
        __syncthreads();
        if (i < n) {
            const int b = cost_bucket(ord.cost[i]);
            ord.order[base[b] + atomicAdd(ord.cursor + b, 1)] = (int)i;
        }
    }
    if (i >= n) return;
    front_cycle(P, in, st, i, recs + i * QPREC_DOUBLES, w_out, w_ld, has_dbg ? &dbg : nullptr);
}

// Four lanes per instance (wbc_front_leg.cuh): the control cycle's front kernel.  Same prelude as wbc_front_kernel (the dispatch
// order of the solve launch that follows and the staged solver's queue reset ride along, indexed by thread).
__global__ void __launch_bounds__(128) wbc_front_leg_kernel(Params P, DevInputs in, FrontState st, int n, double* __restrict__ recs,
                                                            double* __restrict__ w_out, long w_ld, DispatchOrder ord, StageReset sr)
{
    __shared__ int base[ORD_NB];
    const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (sr.ctl) {
        const long nth = (long)gridDim.x * blockDim.x;
        for (long k = t; k < sr.nctl; k += nth) sr.ctl[k] = (k == sr.free_tail_index || k == sr.free_avail_index) ? sr.nslots : 0;
        for (long k = t; k < 3L * sr.rsize; k += nth) sr.ring[k] = (k >= 2L * sr.rsize && k - 2L * sr.rsize < sr.nslots) ? (int)(k - 2L * sr.rsize) : -1;
    }
    if (ord.lanes) {
        const long nth = (long)gridDim.x * blockDim.x;
        for (long k = t; k < LANES_INTS; k += nth) ord.lanes[k] = 0;
    }
    if (ord.cost) {
        if (threadIdx.x < 32) {
            const int l = threadIdx.x;
            int h[8], sum = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) { h[k] = ord.hist[ORD_NB - 1 - (8 * l + k)]; sum += h[k]; }
            int incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, incl, o); if (l >= o) incl += u; }
            int run = incl - sum;
#pragma unroll
            for (int k = 0; k < 8; k++) { base[ORD_NB - 1 - (8 * l + k)] = run; run += h[k]; }
        }
        __syncthreads();
        if (t < n) {
            const int b = cost_bucket(ord.cost[t]);
            ord.order[base[b] + atomicAdd(ord.cursor + b, 1)] = (int)t;
        }
    }
    const long first = (t & ~31L) >> 2;              // first instance of this warp
    if (first >= n) return;
    long i = t >> 2;
    const bool valid = i < n;
    if (!valid) i = n - 1;                            // lanes past the batch compute along (the shuffles need them) and store nothing
    wbc::front_cycle_leg(P, in, st, i, valid, (int)(t & 3), recs + i * QPREC_DOUBLES, w_out, w_ld);
}

struct SolveOut {
    double* tau; double* x; double* qp_obj; int* status; int* qp_info; double* qp_flops; long ld;
    double* tau_prev; long ld_prev;      // [12][max_batch] last good torque of every instance index (main.cpp:242), owned by the ctx
};

__device__ __forceinline__ void write_info(const Stats& st, long i, long ld, int* status, int* info, double* flops)
{
    if (status) status[i] = (st.termination == 2) ? 0 : (st.termination < 0 ? st.termination : -100);
    if (info) {
        info[0 * ld + i] = st.ncholesky; info[1 * ld + i] = st.outer_its; info[2 * ld + i] = st.qqp_calls;
        info[3 * ld + i] = st.nicwork; info[4 * ld + i] = st.kkt_dim_max; info[5 * ld + i] = st.flags;
        info[6 * ld + i] = st.chol_reused; info[7 * ld + i] = 0;
    }
    if (flops) flops[i] = st.flops;
}

__device__ __forceinline__ int next_instance(int* queue)
{
    int i = 0;
    if ((threadIdx.x & 31) == 0) i = atomicAdd(queue, 1);
    return __shfl_sync(0xffffffffu, i, 0);
}

// Express lanes.  A batch of a few thousand instances is two or three solves per resident warp, and its step ends with its LONGEST
// solve: measured at 4 096 standing instances with twelve warps per SM, the sum of all solve latencies is 2.62 ms per warp but the
// longest solve alone takes 3.28 ms (with eight warps per SM: 2.88 and 2.45 -- which is why eight used to win).  A solve runs
// almost twice as fast on an SM it shares with three warps instead of eleven.  So a few SM pairs keep only `keep` of their warps
// (the others leave at once), and those express warps serve the `head` longest solves of the dispatch order, which everybody else
// skips; either side continues in the other's range when its own is used up, so no ticket is left behind.
struct ExpressLanes {
    int* lanes;        // [0] head tickets drawn, [1] tail tickets drawn, [2 + smid] arrivals on SM smid
    int head;          // tickets [0, head) are the express range
    int period, keep;  // every period-th SM pair is express and keeps `keep` warps per SM; period 0: off
    unsigned* cycles;  // [n] the solve's duration (2^10 cycles) when the dispatch cost is not the duration (express lanes on)
    unsigned long long* prof;   // [grid][12] per-warp timeline (WBC_STAGE_PROF=1), else NULL
    float time_scale;  // 0: rank by flop count; > 0: rank by duration, an express warp's multiplied by this
};
__device__ __forceinline__ int next_instance_lanes(const ExpressLanes& xl, bool express, int n)
{
    int t = 0;
    if ((threadIdx.x & 31) == 0) {
        if (express) {
            t = atomicAdd(xl.lanes, 1);
            if (t >= xl.head) t = xl.head + atomicAdd(xl.lanes + 1, 1);
        } else {
            t = xl.head + atomicAdd(xl.lanes + 1, 1);
            if (t >= n) { t = atomicAdd(xl.lanes, 1); if (t >= xl.head) t = n; }
        }
    }
    return __shfl_sync(0xffffffffu, t, 0);
}

__global__ void __launch_bounds__(SOLVE_T) wbc_solve_kernel(Params P, int n, const double* __restrict__ recs, SolveOut out,
                                                            double* __restrict__ scratch_base, double* __restrict__ kkt_base, int* __restrict__ queue,
                                                            const int* __restrict__ order, unsigned* __restrict__ cost,
                                                            int* __restrict__ hist_next, ExpressLanes xl)
{
    Work w;
    w.g = scratch_base + (long)blockIdx.x * gl::TOTAL;
    w.kkt = kkt_base + (long)blockIdx.x * gl::KKT_DOUBLES;
    w.sm = nullptr;
    const WarpEx ex;
    // Express lanes (small batches): on every `period`-th SM pair only the first `keep` warps to arrive stay, and they serve the
    // head of the longest-first order; everybody else starts behind the head.  See ExpressLanes.
    bool express = false;
    if (xl.period > 0) {
        int verdict = 0;                                  // 0 regular, 1 express, 2 leave
        if (ex.lane() == 0) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            if (((smid >> 1) % (unsigned)xl.period) == (unsigned)(xl.period >> 1) && smid < 256u)
                verdict = atomicAdd(xl.lanes + 2 + smid, 1) < xl.keep ? 1 : 2;
        }
        verdict = __shfl_sync(0xffffffffu, verdict, 0);
        if (verdict == 2) {
            if (xl.prof && ex.lane() < 12) xl.prof[(long)blockIdx.x * 12 + ex.lane()] = 0ull;      // no stale row from an earlier launch
            return;
        }
        express = verdict == 1;
    }
    Settings cfg;
    cfg.epsx = P.qp_epsx; cfg.rho = P.qp_rho; cfg.outerits = P.qp_outerits; cfg.kkt_mode = P.qp_literal_kkt ? 0 : 1;
    // every value later read from shared memory is finite (out-of-range lanes read neighbours and drop the result)
    for (int k = ex.lane(); k < sl::TOTAL; k += SOLVE_T) WBC_SM(w)[k] = 0.0;
    ex.sync();
    unsigned long long pr_busy = 0, pr_jobs = 0, pr_first = 0, pr_last = 0, pr_t0 = 0, pr_longest = 0;
    if (xl.prof) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(pr_t0));
    for (;;) {
        const int ticket = xl.period > 0 ? next_instance_lanes(xl, express, n) : next_instance(queue);
        if (ticket >= n) break;
        const int i = order ? order[ticket] : ticket;
        const long long t0 = clock64();
        // the record is staged in the (still idle) CI | EXXC arrays: one cp.async round trip instead of scattered global reads
        double* rec = SM_(w, sl::OFF_CI);
        static_assert(QR_MODE + 1 <= NICCAP * LDH + 104, "QP record fits the staging area");
        ex.copy_in(rec, recs + (long)i * QPREC_DOUBLES, QR_MODE + 1);
        {
            // Inputs the cycle refuses to process: a contact mode outside {0, 1, 2}, or anything non-finite in the record
            // (x * 0 is NaN exactly for NaN and the infinities).  The reference would spin or publish garbage
            // (main.cpp:584-588, lopt.cpp:114-116); here the instance gets a status word and a defined torque.
            double chk = 0.0;
#pragma unroll 1
            for (int k = ex.lane(); k <= QR_MODE; k += SOLVE_T) chk += rec[k] * 0.0;
            const bool nonfinite = __any_sync(0xffffffffu, chk != 0.0);
            const double md = rec[QR_MODE];
            if (nonfinite || !(md == 0.0 || md == 1.0 || md == 2.0)) {
                for (int k = ex.lane(); k < 12; k += SOLVE_T)
                    out.tau[(long)k * out.ld + i] = P.hold_tau_on_failure ? out.tau_prev[(long)k * out.ld_prev + i] : 0.0;
                if (out.x)
                    for (int k = ex.lane(); k < 30; k += SOLVE_T) out.x[(long)k * out.ld + i] = 0.0;
                if (ex.lane() == 0) {
                    Stats st;
                    st.termination = nonfinite ? WBC_ST_NONFINITE : WBC_ST_BAD_MODE;
                    st.ncholesky = 0; st.outer_its = 0; st.qqp_calls = 0; st.nicwork = 0; st.kkt_dim_max = 0; st.chol_reused = 0; st.flags = 0; st.flops = 0.0;
                    write_info(st, i, out.ld, out.status, out.qp_info, out.qp_flops);
                    if (out.qp_obj) out.qp_obj[i] = 0.0;
                    cost[i] = 0u;
                    atomicAdd(hist_next, 1);
                }
                ex.sync();
                continue;
            }
        }
        const QpShape sh = qp_shape((int)rec[QR_MODE]);
        // Q -> H array (ld 31), c -> exb, L -> the warp's global C array (scaled in place by the solver)
        assemble_qp<LDH>(ex, P, rec, sh, W_H(w), W_EXB(w), W_C(w));
        // the lower torque limits and the lower joint-acceleration limits are the negated upper ones (wbc_assemble.cuh)
        {
            const int rt = sh.neq + 5 * sh.nst, rq = rt + 24 + (sh.nst == 2 ? 12 : 0);
            cfg.dup_start[0] = rt + 12; cfg.dup_count[0] = 12;
            cfg.dup_start[1] = rq + 12; cfg.dup_count[1] = 12;
        }
        Stats st;
        solve_denseaul(ex, w, cfg, sh.nrows, sh.neq, st);
        double* xs = W_XS(w);
        if (st.termination != 2) {
            for (int k = ex.lane(); k < 30; k += SOLVE_T) xs[k] = 0.0;
            ex.sync();
        }
        ex.copy_in(rec, recs + (long)i * QPREC_DOUBLES, QR_MODE + 1);     // the solver used the arrays; stage again
        torque_and_objective(ex, P, rec, sh, xs, out.tau + i, out.ld, out.qp_obj ? out.qp_obj + i : nullptr);
        // last good torque of this instance index (main.cpp:242): refreshed on success, handed out instead of the x = 0 torque
        // on failure when the caller asked for it
        if (st.termination == 2) {
            for (int k = ex.lane(); k < 12; k += SOLVE_T) out.tau_prev[(long)k * out.ld_prev + i] = out.tau[(long)k * out.ld + i];
        } else if (P.hold_tau_on_failure) {
            for (int k = ex.lane(); k < 12; k += SOLVE_T) out.tau[(long)k * out.ld + i] = out.tau_prev[(long)k * out.ld_prev + i];
        }
        if (out.x)
            for (int k = ex.lane(); k < 30; k += SOLVE_T) out.x[(long)k * out.ld + i] = xs[k];
        if (ex.lane() == 0) {
            write_info(st, i, out.ld, out.status, out.qp_info, out.qp_flops);
            const unsigned long long dt = (unsigned long long)(clock64() - t0) >> 10;
            unsigned cu = dt > 0xffffffffull ? 0xffffffffu : (unsigned)dt;
            // With express lanes a solve's duration depends on where it ran (an express warp is almost twice as fast), and a cost
            // that does would make the order oscillate: rank by the solve's instrumented flop count instead (correlation with the
            // duration 0.97; the literal multiplier update, which the count does not see, is a flat surcharge).  Same unit: 2^10 cycles.
            if (xl.prof) {
                const unsigned long long d = (unsigned long long)(clock64() - t0);
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                pr_busy += d; pr_jobs++; pr_last = now; if (d > pr_longest) pr_longest = d;
                if (pr_jobs == 1) pr_first = now - (unsigned long long)((double)d / 1.965);      // start of the first solve, ns
            }
            if (xl.period > 0) {
                xl.cycles[i] = cu;
                if (xl.time_scale > 0.0f) cu = express ? (unsigned)((float)cu * xl.time_scale) : cu;
                else cu = (unsigned)(st.flops * (1.0 / 512.0)) + ((st.flags & 8) ? 2000u : 0u);
            }
            cost[i] = cu;
            atomicAdd(hist_next + cost_bucket(cu), 1);
        }
        ex.sync();
    }
    if (xl.prof && ex.lane() == 0) {
        // per-warp timeline: busy cycles, solves, [kernel entry, first solve start, last solve end, exit] (globaltimer, ns), longest solve, express flag, SM
        unsigned long long now; unsigned smid;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        unsigned long long* p = xl.prof + (long)blockIdx.x * 12;
        p[0] = pr_busy; p[1] = pr_jobs; p[2] = pr_t0; p[3] = pr_first; p[4] = pr_last; p[5] = now; p[6] = pr_longest; p[7] = express ? 1 : 0; p[8] = smid;
        p[9] = 0; p[10] = 0; p[11] = 0;
    }
}

// ---- exact QP mode (WBC_QP_EXACT): the Goldfarb-Idnani dual active-set solver of qp_dual.cuh, one warp per solve.
// Its shared block is 17.2 KB (R, the factor / product scratch and a few vectors) and J lives in registers; the constraint matrix
// stays in the warp's global scratch.  Residency: with the 1 KB the SM reserves per CTA, shared memory admits 12 CTAs per SM
// (13 x 18.6 KB > 228 KB), and __launch_bounds__(32, 12) lets the compiler use all 168 registers that 12 CTAs leave per thread
// (ptxas: 165, no spills).  Fewer warps with more registers lost: -DWBC_EXACT_MIN_CTAS=8 (no spills then either) measured 0.93x at
// 65 536 and 0.73x at 4 096 instances (profiles/r03_exact_ctas_ab.txt).
constexpr int EXACT_T = 32;
#ifndef WBC_EXACT_MIN_CTAS
#define WBC_EXACT_MIN_CTAS 12
#endif
constexpr int EXACT_MIN_CTAS = WBC_EXACT_MIN_CTAS;
static_assert(wbc::QR_MODE + 1 <= wbcdual::N * wbcdual::LD, "the QP record is staged in R's place");

// ws (warm mode): [6], [7] are the warm rows added and dropped before the GI loop (0 in cold exact mode)
__device__ __forceinline__ void write_info_exact(const wbcdual::DualStats& st, long i, long ld, int* status, int* info, double* flops,
                                                 const wbcdual::WarmStats* ws = nullptr)
{
    if (status) status[i] = st.status;
    if (info) {
        info[0 * ld + i] = st.nfact; info[1 * ld + i] = st.adds; info[2 * ld + i] = st.drops; info[3 * ld + i] = st.nact_ineq;
        info[4 * ld + i] = st.nact; info[5 * ld + i] = st.flags; info[6 * ld + i] = ws ? ws->adds : 0; info[7 * ld + i] = ws ? ws->drops : 0;
    }
    if (flops) flops[i] = st.flops;
}

// qp_info[5] flag of an instance that wbc_cycle with WBC_QP_WARM started from its stored active set
constexpr int FL_WARM_STARTED = 2048;

// PROF = true (a ctx created with WBC_STAGE_PROF=1): per-warp cycle counters by phase, rows of 12 in `prof` (wbc_stage_profile):
// [0..8] the wbcdual::PH_* phases summed over the warp's solves, [9] solves, [10] rows added + dropped, [11] cycles in the kernel.
// aset [4][aset_ld]: the ctx's stored active set per instance index -- words 0..2 the active inequality rows, word 3 the contact
// mode they were solved in + 1 (0: none).  Every instance writes its own (its final set, or none when it failed or was refused);
// WARM = true (WBC_QP_WARM) first reads it and starts from it when the stored mode is the instance's mode.
template <bool PROF, bool WARM = false>
__global__ void __launch_bounds__(EXACT_T, EXACT_MIN_CTAS) wbc_solve_exact_kernel(Params P, int n, const double* __restrict__ recs, SolveOut out,
                                                                                 double* __restrict__ scratch_base, int* __restrict__ queue,
                                                                                 const int* __restrict__ order, unsigned* __restrict__ cost,
                                                                                 int* __restrict__ hist_next, unsigned long long* __restrict__ prof,
                                                                                 int prof_rows, unsigned* __restrict__ aset, long aset_ld)
{
    const WarpEx ex;
    unsigned long long pc[12];
#pragma unroll
    for (int k = 0; k < 12; k++) pc[k] = 0ull;
    const long long k0 = PROF ? clock64() : 0;
    double* sm = wbc_smem;
    double* C = scratch_base + (long)blockIdx.x * wbcdual::SCRATCH_DOUBLES;
    for (int k = ex.lane(); k < wbcdual::ds::TOTAL; k += EXACT_T) sm[k] = 0.0;
    ex.sync();
    for (;;) {
        const int ticket = next_instance(queue);
        if (ticket >= n) break;
        const int i = order ? order[ticket] : ticket;
        const long long t0 = clock64();
        double* rec = sm + wbcdual::ds::OFF_R;
        ex.copy_in(rec, recs + (long)i * QPREC_DOUBLES, QR_MODE + 1);
        wbcdual::DualStats st;
        {
            // the record validation of wbc_solve_kernel
            double chk = 0.0;
#pragma unroll 1
            for (int k = ex.lane(); k <= QR_MODE; k += EXACT_T) chk += rec[k] * 0.0;
            const bool nonfinite = __any_sync(0xffffffffu, chk != 0.0);
            const double md = rec[QR_MODE];
            if (nonfinite || !(md == 0.0 || md == 1.0 || md == 2.0)) {
                for (int k = ex.lane(); k < 12; k += EXACT_T)
                    out.tau[(long)k * out.ld + i] = P.hold_tau_on_failure ? out.tau_prev[(long)k * out.ld_prev + i] : 0.0;
                if (out.x)
                    for (int k = ex.lane(); k < 30; k += EXACT_T) out.x[(long)k * out.ld + i] = 0.0;
                if (ex.lane() == 0) {
                    st.status = nonfinite ? WBC_ST_NONFINITE : WBC_ST_BAD_MODE;
                    st.nfact = 0; st.adds = 0; st.drops = 0; st.nact_ineq = 0; st.nact = 0; st.flags = wbcdual::FL_EXACT; st.flops = 0.0;
                    write_info_exact(st, i, out.ld, out.status, out.qp_info, out.qp_flops);
                    if (out.qp_obj) out.qp_obj[i] = 0.0;
                    cost[i] = 0u;
                    atomicAdd(hist_next, 1);
                    for (int k = 0; k < 4; k++) aset[k * aset_ld + i] = 0u;
                }
                ex.sync();
                continue;
            }
        }
        const QpShape sh = qp_shape((int)rec[QR_MODE]);
        assemble_qp<wbcdual::LD>(ex, P, rec, sh, sm + wbcdual::ds::OFF_H, sm + wbcdual::ds::OFF_CV, C);
        if (PROF) pc[wbcdual::PH_ASSEMBLE] += (unsigned long long)(clock64() - t0);
        unsigned wset[3] = {0u, 0u, 0u};
        if constexpr (WARM) {
            if (aset[3 * aset_ld + i] == (unsigned)rec[QR_MODE] + 1u)
                for (int k = 0; k < 3; k++) wset[k] = aset[k * aset_ld + i];
        }
        wbcdual::WarmStats ws;
        wbcdual::solve_dual<WarpEx, PROF, WARM>(ex, sm, C, sh.nrows, sh.neq, st, pc, wset, &ws);
        const long long t1 = PROF ? clock64() : 0;
        const double* xs = sm + wbcdual::ds::OFF_Y;          // x, or 0 when the solve failed
        ex.copy_in(rec, recs + (long)i * QPREC_DOUBLES, QR_MODE + 1);     // R's place was the solver's; stage again
        torque_and_objective(ex, P, rec, sh, xs, out.tau + i, out.ld, out.qp_obj ? out.qp_obj + i : nullptr);
        if (st.status == 0) {
            for (int k = ex.lane(); k < 12; k += EXACT_T) out.tau_prev[(long)k * out.ld_prev + i] = out.tau[(long)k * out.ld + i];
        } else if (P.hold_tau_on_failure) {
            for (int k = ex.lane(); k < 12; k += EXACT_T) out.tau[(long)k * out.ld + i] = out.tau_prev[(long)k * out.ld_prev + i];
        }
        if (out.x)
            for (int k = ex.lane(); k < 30; k += EXACT_T) out.x[(long)k * out.ld + i] = xs[k];
        if (ex.lane() == 0) {
            const unsigned mode1 = (unsigned)rec[QR_MODE] + 1u;      // rec is staged again: the mode is read after the solve
            if (WARM && aset[3 * aset_ld + i] == mode1) st.flags |= FL_WARM_STARTED;
            write_info_exact(st, i, out.ld, out.status, out.qp_info, out.qp_flops, WARM ? &ws : nullptr);
            for (int k = 0; k < 3; k++) aset[k * aset_ld + i] = ws.act[k];
            aset[3 * aset_ld + i] = st.status == 0 ? mode1 : 0u;
            // the duration orders the next cycle's dispatch (longest first), as in wbc_solve_kernel: one bucket entry per instance
            const unsigned long long dt = (unsigned long long)(clock64() - t0) >> 10;
            const unsigned cu = dt > 0xffffffffull ? 0xffffffffu : (unsigned)dt;
            cost[i] = cu;
            atomicAdd(hist_next + cost_bucket(cu), 1);
        }
        ex.sync();
        if (PROF) {
            pc[wbcdual::PH_OUTPUT] += (unsigned long long)(clock64() - t1);
            pc[9]++;
            pc[10] += (unsigned long long)(st.adds + st.drops);
        }
    }
    if (PROF && ex.lane() == 0 && (int)blockIdx.x < prof_rows) {
        pc[11] = (unsigned long long)(clock64() - k0);
        for (int k = 0; k < 12; k++) prof[(long)blockIdx.x * 12 + k] = pc[k];
    }
}

// Dense-input form of the exact solver (wbc_qp_solve with WBC_QP_EXACT): Q [n][900], c [n][30], L [n][nrows*31], x [n][30].
// WARM = true (wbc_qp_solve_warm): active [n][3] is read as each instance's warm set and overwritten with its final active
// inequality rows (0 on failure).
template <bool WARM = false>
__global__ void __launch_bounds__(EXACT_T, EXACT_MIN_CTAS) wbc_dense_qp_exact_kernel(int n, const double* __restrict__ Q, const double* __restrict__ c,
                                                                                    const double* __restrict__ L, int nrows, int neq, double* __restrict__ x,
                                                                                    int* status, int* info, double* flops, double* __restrict__ scratch_base,
                                                                                    int* __restrict__ queue, unsigned* __restrict__ active = nullptr)
{
    const WarpEx ex;
    double* sm = wbc_smem;
    double* C = scratch_base + (long)blockIdx.x * wbcdual::SCRATCH_DOUBLES;
    for (int k = ex.lane(); k < wbcdual::ds::TOTAL; k += EXACT_T) sm[k] = 0.0;
    ex.sync();
    for (;;) {
        const int i = next_instance(queue);
        if (i >= n) break;
        double* H = sm + wbcdual::ds::OFF_H;
        double chk = 0.0;                      // x * 0 is NaN exactly for NaN and the infinities
        for (int k = ex.lane(); k < 900; k += EXACT_T) { const double v = Q[(long)i * 900 + k]; H[(k / 30) * wbcdual::LD + (k % 30)] = v; chk += v * 0.0; }
        for (int k = ex.lane(); k < 30; k += EXACT_T) { const double v = c[(long)i * 30 + k]; sm[wbcdual::ds::OFF_CV + k] = v; chk += v * 0.0; }
        for (int k = ex.lane(); k < nrows * 31; k += EXACT_T) { const double v = L[(long)i * nrows * 31 + k]; C[k] = v; chk += v * 0.0; }
        ex.sync();
        wbcdual::DualStats st;
        wbcdual::WarmStats ws;
        if (__any_sync(0xffffffffu, chk != 0.0)) {
            st.status = WBC_ST_NONFINITE; st.nfact = 0; st.adds = 0; st.drops = 0; st.nact_ineq = 0; st.nact = 0; st.flags = wbcdual::FL_EXACT; st.flops = 0.0;
            if constexpr (WARM) { ws.adds = 0; ws.drops = 0; ws.act[0] = 0u; ws.act[1] = 0u; ws.act[2] = 0u; }
            for (int k = ex.lane(); k < 30; k += EXACT_T) sm[wbcdual::ds::OFF_Y + k] = 0.0;
            ex.sync();
        } else if constexpr (WARM) {
            wbcdual::solve_dual<WarpEx, false, true>(ex, sm, C, nrows, neq, st, nullptr, active + (long)i * 3, &ws);
        } else
            wbcdual::solve_dual(ex, sm, C, nrows, neq, st);
        for (int k = ex.lane(); k < 30; k += EXACT_T) x[(long)i * 30 + k] = sm[wbcdual::ds::OFF_Y + k];
        if (ex.lane() == 0) {   // instance-major info [n][8] on this path
            if (status) status[i] = st.status;
            if (flops) flops[i] = st.flops;
            if (info) {
                int* q = info + (long)i * 8;
                q[0] = st.nfact; q[1] = st.adds; q[2] = st.drops; q[3] = st.nact_ineq; q[4] = st.nact; q[5] = st.flags;
                q[6] = WARM ? ws.adds : 0; q[7] = WARM ? ws.drops : 0;
            }
            if constexpr (WARM)
                for (int k = 0; k < 3; k++) active[(long)i * 3 + k] = ws.act[k];
        }
        ex.sync();
    }
}

// ------------------------------------------------------------------------------------------------
// The solver as a persistent kernel of STAGE TASKS (qp_warp.cuh, solve_stage_*).
//
// What bounds wbc_solve_kernel above is instruction supply: its hot code is ~140 KB, an SM's instruction cache holds ~32 KB
// (tools/ubench/icache.cu), the twelve warps of an SM are in twelve different places of it, and every miss is served by the
// GPC-level cache at ~4 bytes per cycle and SM -- ncu shows that cache at 80-90 % of its peak request rate and more resident
// warps buy nothing (profiles/README.md).  Here a solve is not bound to a warp.  It lives in a slot of global memory (the
// scratch block it always had, plus a 1 KB header) and moves through three kinds of task,
//     SETUP  (assemble + set-up)      ->   QLOOP (model, QQP, working set)   <->   UPDATE (multipliers, feasibility)   -> torque map
// each executed by whichever warp pops it.  Warps prefer the task kind of their SM's ROLE (QLOOP on two thirds of the SMs,
// SETUP/UPDATE on the rest) and take the other kind only when theirs has run dry, so an SM's warps run one third of the code
// most of the time and the GPC caches serve far fewer misses.  Hand-over = three lock-free rings of slot indices in global
// memory (QLOOP tasks, UPDATE tasks, free slots); a push is preceded and a pop followed by __threadfence(), which on sm_100
// is MEMBAR.SC.GPU + CCTL.IVALL, i.e. also drops the popping SM's stale L1 lines of the slot.  Same arithmetic as the
// monolithic kernel: results are bit-identical (tools/gpu_dump.py).
struct StageCtl {
    int ticket; int pad0[31];          // next new solve (dispatch ticket)
    int done; int pad1[31];            // finished solves
    int head[3][32];                   // [q][0] is the counter; one 128-byte line each
    int tail[3][32];
    int avail[3][32];                  // published entries not yet claimed by a pop
};
constexpr int SQ_QLOOP = 0, SQ_UPDATE = 1, SQ_FREE = 2;
constexpr int HDR_INST = gl::HDR_DOUBLES - 1, HDR_CYCLES = gl::HDR_DOUBLES - 2;      // header tail: instance index, cycles so far
static_assert(sizeof(SolveState) <= (gl::HDR_DOUBLES - 2) * sizeof(double), "header tail is free");

struct StageQueues {
    StageCtl* ctl;
    int* ring;          // [3][rmask + 1], -1 = empty
    int rmask;
    int nslots;
};

// Fetch-add rings: no compare-and-swap loop anywhere (a CAS loop on one counter serialises at one success per L2 round trip once
// a few hundred warps contend, ~1 M pops/s against the 4 M/s this kernel needs -- measured: warps spent a third of their cycles
// in pop).  `avail` counts published entries minus pops in progress; a pop that takes it from > 0 owns the next head position.
__device__ __forceinline__ void sq_push(const StageQueues& q, int which, int slot)
{
    // caller: every lane has fenced its writes to the slot and the warp has synchronised; lane 0 only
    const int pos = atomicAdd(&q.ctl->tail[which][0], 1);
    atomicExch(q.ring + which * (q.rmask + 1) + (pos & q.rmask), slot);
    atomicAdd(&q.ctl->avail[which][0], 1);      // (a pop that sees the count before the entry spins on the entry)
}
__device__ __forceinline__ int sq_pop(const StageQueues& q, int which)
{
    // lane 0 only; -1 when the ring is empty
    if (*(volatile int*)&q.ctl->avail[which][0] <= 0) return -1;
    if (atomicSub(&q.ctl->avail[which][0], 1) <= 0) { atomicAdd(&q.ctl->avail[which][0], 1); return -1; }
    const int h = atomicAdd(&q.ctl->head[which][0], 1);
    int* e = q.ring + which * (q.rmask + 1) + (h & q.rmask);
    int sIdx;
    while ((sIdx = atomicExch(e, -1)) < 0) __nanosleep(20);      // an earlier position's push is still in flight
    return sIdx;
}

__global__ void __launch_bounds__(SOLVE_T) wbc_solve_staged_kernel(Params P, int n, const double* __restrict__ recs, SolveOut out,
                                                                   double* __restrict__ slot_base, double* __restrict__ kkt_base, StageQueues sq,
                                                                   const int* __restrict__ order, unsigned* __restrict__ cost,
                                                                   int* __restrict__ hist_next, int m_period, int m_group, unsigned long long* __restrict__ prof)
{
    Work w;
    w.g = nullptr;
    w.kkt = kkt_base + (long)blockIdx.x * gl::KKT_DOUBLES;
    w.sm = nullptr;
    const WarpExS ex;                                              // bulk copies through the shared routine (qp_warp.cuh)
    Settings cfg;
    cfg.epsx = P.qp_epsx; cfg.rho = P.qp_rho; cfg.outerits = P.qp_outerits; cfg.kkt_mode = P.qp_literal_kkt ? 0 : 1;
    for (int k = ex.lane(); k < sl::TOTAL; k += SOLVE_T) WBC_SM(w)[k] = 0.0;
    ex.sync();
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    // Role of this SM.  m_period packs (nS << 16 | nP << 8 | den): of every `den` groups of m_group SMs (an SM pair = a TPC shares
    // its instruction supply, so roles go by pairs), nS start new solves first (SETUP tasks: assemble + set-up), nP take POST tasks
    // first (violations, working set, multiplier update, next model), the others QQP tasks.  Group indices are spread with a
    // stride so that the roles interleave across the chip.
    const unsigned r_ns = ((unsigned)m_period >> 16) & 255u, r_np = ((unsigned)m_period >> 8) & 255u, r_den = (unsigned)m_period & 255u;
    int role = 0;                                                    // 0: QQP, 1: POST, 2: SETUP
    if (r_den > 0) {
        const unsigned gi = ((smid / (unsigned)m_group) * 7u) % r_den;
        role = gi < r_ns ? 2 : (gi < r_ns + r_np ? 1 : 0);
    }
    const bool role_m = role != 0;
    volatile int* donep = &sq.ctl->done;
    volatile int* ticketp = &sq.ctl->ticket;
    int idle = 0;
    // profile (optional): cycles and counts per task kind, cycles spent looking for a task, cycles in the two fences
    unsigned long long pr_cyc[3] = {0, 0, 0}, pr_cnt[3] = {0, 0, 0}, pr_wait = 0, pr_fence = 0, pr_steal = 0;
    const long long k0 = clock64();
    long long tq = k0;
    for (;;) {
        // ---- take a task: (kind, slot); kind 0 = QLOOP, 1 = UPDATE, 2 = SETUP (slot fresh, ticket drawn)
        int kind = -1, slot = -1, ticket = -1;
        if (ex.lane() == 0) {
            // preference order of the three sources of work by role; a source that has run dry is skipped
            //   QQP SMs:   QQP ring, POST ring, new solve        POST SMs:  POST ring, new solve, QQP ring
            //   SETUP SMs: new solve, POST ring, QQP ring
            const int order3[3][3] = {{SQ_QLOOP, SQ_UPDATE, 2}, {SQ_UPDATE, 2, SQ_QLOOP}, {2, SQ_UPDATE, SQ_QLOOP}};
#pragma unroll 1
            for (int t = 0; t < 3 && kind < 0; t++) {
                const int src = order3[role][t];
                if (src == 2) {
                    if (*ticketp < n) {                              // start a new solve: a free slot and a dispatch ticket
                        slot = sq_pop(sq, SQ_FREE);
                        if (slot >= 0) {
                            ticket = atomicAdd(&sq.ctl->ticket, 1);
                            if (ticket < n) kind = 2;
                            else { sq_push(sq, SQ_FREE, slot); slot = -1; }
                        }
                    }
                } else {
                    slot = sq_pop(sq, src);
                    if (slot >= 0) kind = src;
                }
            }
            if (kind < 0 && *donep >= n) kind = -2;
        }
        kind = __shfl_sync(0xffffffffu, kind, 0);
        if (kind == -2) break;
        if (kind < 0) {
            idle = idle < 8 ? idle + 1 : 8;
            __nanosleep(64u << idle);
            continue;
        }
        idle = 0;
        slot = __shfl_sync(0xffffffffu, slot, 0);
        ticket = __shfl_sync(0xffffffffu, ticket, 0);
        const long long tf0 = clock64();
        pr_wait += (unsigned long long)(tf0 - tq);
        __threadfence();                                             // acquire: the slot as its last stage left it (also drops stale L1 lines)
        const long long t0 = clock64();
        pr_fence += (unsigned long long)(t0 - tf0);
        if (kind != role) pr_steal++;
        w.g = slot_base + (long)slot * gl::TOTAL;
        double* hdr = w.g + gl::OFF_HDR;
        double* rec = SM_(w, sl::OFF_CI);
        SolveState st;
        int i;
        long long cyc0 = 0;
        int next = -1;                                               // ring the slot goes to afterwards (-1: the solve is finished)
        bool finished = false;
        if (kind == 2) {
            i = order ? order[ticket] : ticket;
            ex.copy_in(rec, recs + (long)i * QPREC_DOUBLES, QR_MODE + 1);
            double chk = 0.0;
#pragma unroll 1
            for (int k = ex.lane(); k <= QR_MODE; k += SOLVE_T) chk += rec[k] * 0.0;
            const bool nonfinite = __any_sync(0xffffffffu, chk != 0.0);
            const double md = rec[QR_MODE];
            if (nonfinite || !(md == 0.0 || md == 1.0 || md == 2.0)) {
                for (int k = ex.lane(); k < 12; k += SOLVE_T)
                    out.tau[(long)k * out.ld + i] = P.hold_tau_on_failure ? out.tau_prev[(long)k * out.ld_prev + i] : 0.0;
                if (out.x)
                    for (int k = ex.lane(); k < 30; k += SOLVE_T) out.x[(long)k * out.ld + i] = 0.0;
                if (ex.lane() == 0) {
                    Stats z;
                    z.termination = nonfinite ? WBC_ST_NONFINITE : WBC_ST_BAD_MODE;
                    z.ncholesky = 0; z.outer_its = 0; z.qqp_calls = 0; z.nicwork = 0; z.kkt_dim_max = 0; z.chol_reused = 0; z.flags = 0; z.flops = 0.0;
                    write_info(z, i, out.ld, out.status, out.qp_info, out.qp_flops);
                    if (out.qp_obj) out.qp_obj[i] = 0.0;
                    cost[i] = 0u;
                    atomicAdd(hist_next, 1);
                }
                finished = true;
            } else {
                const QpShape sh = qp_shape((int)md);
                assemble_qp<LDH>(ex, P, rec, sh, W_H(w), W_EXB(w), W_C(w));
                const int rt = sh.neq + 5 * sh.nst, rq = rt + 24 + (sh.nst == 2 ? 12 : 0);
                cfg.dup_start[0] = rt + 12; cfg.dup_count[0] = 12;
                cfg.dup_start[1] = rq + 12; cfg.dup_count[1] = 12;
                solve_stage_setup(ex, w, cfg, sh.nrows, sh.neq, st);
                if (!st.done) {
                    st.outer_its++;
                    if (stage_post_and_model(ex, w, cfg, st, false)) next = SQ_QLOOP;
                }
            }
        } else {
            i = (int)hdr[HDR_INST];
            cyc0 = (long long)hdr[HDR_CYCLES];
            stage_load(ex, w, st);
            if (kind == SQ_QLOOP) { stage_qqp(ex, w, st); next = SQ_UPDATE; }
            else if (stage_post_and_model(ex, w, cfg, st, true)) next = SQ_QLOOP;
        }
        if (!finished && st.done) {
            // ---- the solve is complete: torque map and outputs (as in wbc_solve_kernel)
            double* xs = W_XS(w);
            if (st.termination != 2) {
                for (int k = ex.lane(); k < 30; k += SOLVE_T) xs[k] = 0.0;
                ex.sync();
            }
            ex.copy_in(rec, recs + (long)i * QPREC_DOUBLES, QR_MODE + 1);
            const QpShape sh = qp_shape((int)rec[QR_MODE]);
            torque_and_objective(ex, P, rec, sh, xs, out.tau + i, out.ld, out.qp_obj ? out.qp_obj + i : nullptr);
            if (st.termination == 2) {
                for (int k = ex.lane(); k < 12; k += SOLVE_T) out.tau_prev[(long)k * out.ld_prev + i] = out.tau[(long)k * out.ld + i];
            } else if (P.hold_tau_on_failure) {
                for (int k = ex.lane(); k < 12; k += SOLVE_T) out.tau[(long)k * out.ld + i] = out.tau_prev[(long)k * out.ld_prev + i];
            }
            if (out.x)
                for (int k = ex.lane(); k < 30; k += SOLVE_T) out.x[(long)k * out.ld + i] = xs[k];
            if (ex.lane() == 0) {
                Stats z;
                stage_stats(st, z);
                write_info(z, i, out.ld, out.status, out.qp_info, out.qp_flops);
                const unsigned long long dt = (unsigned long long)(cyc0 + (clock64() - t0)) >> 10;
                const unsigned cu = dt > 0xffffffffull ? 0xffffffffu : (unsigned)dt;
                cost[i] = cu;
                atomicAdd(hist_next + cost_bucket(cu), 1);
            }
            finished = true;
        }
        if (!finished) {
            stage_store(ex, w, st);
            if (ex.lane() == 0) {
                hdr[HDR_INST] = (double)i;
                hdr[HDR_CYCLES] = (double)(cyc0 + (clock64() - t0));
            }
        }
        const long long t1 = clock64();
        pr_cyc[kind] += (unsigned long long)(t1 - t0); pr_cnt[kind]++;
        __threadfence();                                             // release: the slot (or the outputs) before the hand-over
        ex.sync();
        if (ex.lane() == 0) {
            if (finished) { sq_push(sq, SQ_FREE, slot); atomicAdd(&sq.ctl->done, 1); }
            else sq_push(sq, next, slot);
        }
        tq = clock64();
        pr_fence += (unsigned long long)(tq - t1);
    }
    if (prof && ex.lane() == 0) {
        unsigned long long* p = prof + (long)blockIdx.x * 12;
        p[0] = pr_cyc[0]; p[1] = pr_cyc[1]; p[2] = pr_cyc[2]; p[3] = pr_cnt[0]; p[4] = pr_cnt[1]; p[5] = pr_cnt[2];
        p[6] = pr_wait; p[7] = pr_fence; p[8] = pr_steal; p[9] = (unsigned long long)(clock64() - k0); p[10] = (unsigned long long)role; p[11] = smid;
    }
}

// Thread per instance: evaluate the plan's four splines at the instance's time (wbc_traj.cuh).
__global__ void __launch_bounds__(128) wbc_traj_kernel(int n, int nseg, const double* __restrict__ dur, const double* __restrict__ nodes, long ld,
                                                       const double* __restrict__ t, double t_all, wbc::TrajOut out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    wbc::TrajOut o;
#pragma unroll
    for (int b = 0; b < 6; b++) o.p[b] = out.p[b] + i;
    o.ld = out.ld;
    wbc::sample_trajectory_instance(nseg, dur + i, nodes + i, ld, t ? t[i] : t_all, o);
}

// OPT-operator path: dense, instance-major (Q [n][900], c [n][30], L [n][nrows*31], x [n][30]).
__global__ void __launch_bounds__(SOLVE_T) wbc_dense_qp_kernel(Params P, int n, const double* __restrict__ Q, const double* __restrict__ c,
                                                               const double* __restrict__ L, int nrows, int neq, double* __restrict__ x,
                                                               int* status, int* info, double* flops, double* __restrict__ scratch_base,
                                                               double* __restrict__ kkt_base, int* __restrict__ queue)
{
    Work w;
    w.g = scratch_base + (long)blockIdx.x * gl::TOTAL;
    w.kkt = kkt_base + (long)blockIdx.x * gl::KKT_DOUBLES;
    w.sm = nullptr;
    const WarpEx ex;
    Settings cfg;
    cfg.epsx = P.qp_epsx; cfg.rho = P.qp_rho; cfg.outerits = P.qp_outerits; cfg.kkt_mode = P.qp_literal_kkt ? 0 : 1;
    // every value later read from shared memory is finite (out-of-range lanes read neighbours and drop the result)
    for (int k = ex.lane(); k < sl::TOTAL; k += SOLVE_T) WBC_SM(w)[k] = 0.0;
    ex.sync();
    for (;;) {
        const int i = next_instance(queue);
        if (i >= n) break;
        double* H = W_H(w);
        double chk = 0.0;                      // x * 0 is NaN exactly for NaN and the infinities
        for (int k = ex.lane(); k < 900; k += SOLVE_T) { const double v = Q[(long)i * 900 + k]; H[(k / 30) * LDH + (k % 30)] = v; chk += v * 0.0; }
        for (int k = ex.lane(); k < 30; k += SOLVE_T) { const double v = c[(long)i * 30 + k]; W_EXB(w)[k] = v; chk += v * 0.0; }
        for (int k = ex.lane(); k < nrows * 31; k += SOLVE_T) { const double v = L[(long)i * nrows * 31 + k]; W_C(w)[k] = v; chk += v * 0.0; }
        ex.sync();
        Stats st;
        if (__any_sync(0xffffffffu, chk != 0.0)) {
            // a non-finite coefficient: nothing is solved (ALGLIB would throw or return garbage; the reference swallows both, lopt.cpp:114-116)
            st.termination = WBC_ST_NONFINITE; st.ncholesky = 0; st.outer_its = 0; st.qqp_calls = 0; st.nicwork = 0; st.kkt_dim_max = 0;
            st.chol_reused = 0; st.flags = 0; st.flops = 0.0;
        } else
            solve_denseaul(ex, w, cfg, nrows, neq, st);
        // a failed instance returns x = 0, like wbc_cycle (never a previous call's solution left in the staging block)
        for (int k = ex.lane(); k < 30; k += SOLVE_T) x[(long)i * 30 + k] = (st.termination == 2) ? W_XS(w)[k] : 0.0;
        if (ex.lane() == 0) {   // instance-major info [n][8] on this path
            write_info(st, i, n, status, nullptr, flops);
            if (info) {
                int* q = info + (long)i * 8;
                q[0] = st.ncholesky; q[1] = st.outer_its; q[2] = st.qqp_calls; q[3] = st.nicwork; q[4] = st.kkt_dim_max;
                q[5] = st.flags; q[6] = st.chol_reused; q[7] = 0;
            }
        }
        ex.sync();
    }
}

// Synthetic plant of BASELINE config 5 (see wbc_plant_step in wbc_b200.h): thread per instance, reads the momentum
// balance the front kernel left in the QP record.
__global__ void __launch_bounds__(128) wbc_plant_kernel(Params P, int n, const double* __restrict__ recs, double* base_pos, double* base_vel,
                                                        double* foot_force, const double* __restrict__ x, const double* __restrict__ push, long ld)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* rec = recs + i * QPREC_DOUBLES;
    double L[36], y[6];
    for (int k = 0; k < 36; k++) L[k] = rec[QR_MC + k];
    if (foot_force) {
        // closed loop: the ground reacts with the commanded forces f* = x[18:30] (stance layout, main.cpp:1126); they
        // are what the contact sensors report next cycle, in the foot frames (Fgrf = R_foot f, main.cpp:1022-1026)
        double f[12];
        for (int r = 0; r < 12; r++) f[r] = x[(long)(18 + r) * ld + i];
        for (int a = 0; a < 6; a++) {
            double fc = 0.0;
            for (int r = 0; r < 12; r++) fc += rec[QR_JC + r * 6 + a] * f[r];
            y[a] = rec[QR_RHO + a] + P.obs_dt * (-dogbot::kTotalMass * (a == 2 ? P.g_acc : 0.0) + fc + push[(long)a * ld + i]);
        }
        for (int sf = 0; sf < 4; sf++) {
            const double* R = rec + QR_FOOTR + 9 * sf;
            for (int k = 0; k < 3; k++)
                foot_force[(long)(3 * sf + k) * ld + i] = R[k] * f[3 * sf] + R[3 + k] * f[3 * sf + 1] + R[6 + k] * f[3 * sf + 2];
        }
    } else {
        for (int a = 0; a < 6; a++) y[a] = rec[QR_RHO + a] + P.obs_dt * (rec[QR_DD + a] + push[(long)a * ld + i]);
    }
    // Mc is symmetric positive definite: Cholesky, two triangular solves
    for (int c = 0; c < 6; c++) {
        double d = L[c * 6 + c];
        for (int k = 0; k < c; k++) d -= L[c * 6 + k] * L[c * 6 + k];
        d = sqrt(d);
        L[c * 6 + c] = d;
        for (int r = c + 1; r < 6; r++) {
            double v = L[r * 6 + c];
            for (int k = 0; k < c; k++) v -= L[r * 6 + k] * L[c * 6 + k];
            L[r * 6 + c] = v / d;
        }
    }
    for (int r = 0; r < 6; r++) {
        double v = y[r];
        for (int k = 0; k < r; k++) v -= L[r * 6 + k] * y[k];
        y[r] = v / L[r * 6 + r];
    }
    for (int r = 5; r >= 0; r--) {
        double v = y[r];
        for (int k = r + 1; k < 6; k++) v -= L[k * 6 + r] * y[k];
        y[r] = v / L[r * 6 + r];
    }
    const double bx = rec[QR_XBC], by = rec[QR_XBC + 1], bz = rec[QR_XBC + 2];
    const double vx = y[0] - (y[4] * bz - y[5] * by), vy = y[1] - (y[5] * bx - y[3] * bz), vz = y[2] - (y[3] * by - y[4] * bx);
    base_vel[0 * ld + i] = vx; base_vel[1 * ld + i] = vy; base_vel[2 * ld + i] = vz;
    base_vel[3 * ld + i] = y[3]; base_vel[4 * ld + i] = y[4]; base_vel[5 * ld + i] = y[5];
    if (base_pos) {
        base_pos[0 * ld + i] += P.obs_dt * vx; base_pos[1 * ld + i] += P.obs_dt * vy; base_pos[2 * ld + i] += P.obs_dt * vz;
    }
}

// Forward-dynamics plant (SURVEY.md 8f-2), thread per instance (wbc_front.cuh, fdyn_step_instance).
__global__ void __launch_bounds__(64) wbc_fdyn_kernel(Params P, wbc::FdynIO io, int n, int nsub, double gamma)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    wbc::fdyn_step_instance(P, io, i, nsub, gamma);
}

// Contact plant (unilateral, frictional foot contacts), thread per instance (wbc_contact.cuh, contact_step_instance).
__global__ void __launch_bounds__(64) wbc_contact_kernel(Params P, wbc::ContactParams cp, wbc::ContactIO io, int n, int nsub)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    wbc::contact_step_instance(P, cp, io, i, nsub);
}

// Contact plant on per-foot planes and contact frames (the terrain form of contact_step_instance); io.ground_z holds the plane offsets.
__global__ void __launch_bounds__(64) wbc_contact_terrain_kernel(Params P, wbc::ContactParams cp, wbc::ContactIO io, int n, int nsub,
                                                                 const double* terrain)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    wbc::contact_step_instance<true>(P, cp, io, i, nsub, terrain);
}

// Trot gait generator, thread per robot (wbc_gait.cuh): capture the gait state, and one gait step.
__global__ void __launch_bounds__(128) wbc_gait_init_kernel(wbc::GaitParams G, double dt, wbc::GaitIO io, int n)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    wbc::gait_init_instance(G, dt, io, i);
}

__global__ void __launch_bounds__(128) wbc_gait_kernel(wbc::GaitParams G, double dt, wbc::GaitIO io, int n)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    wbc::gait_step_instance(G, dt, io, i);
}

// FP64 DFMA peak: 8 independent chains per thread, fully unrolled.
__global__ void __launch_bounds__(256) wbc_dfma_peak_kernel(double* out, int iters)
{
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, b = 1e-7;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
            a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
            a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
        }
    }
    out[(long)blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ------------------------------------------------------------------------------------------------
// host side
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, const char* a = "", const char* b = "")
{
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return code;
}
#define CU(call)                                                                         \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) return fail(WBC_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

// field table of wbc_inputs for staging host buffers
struct FieldDesc { int k; };
static const int kInFieldK[15] = {3, 9, 3, 6, 12, 12, 6, 6, 6, 6, 6, 6, 12, 40, 1};
static const int kInDoublesNoTerrain = 3 + 9 + 3 + 6 + 12 + 12 + 6 + 6 + 6 + 6 + 6 + 6 + 12;   // 93
static const int kOutDoubles = 12 + 6 + 30 + 1 + 1 + 12;   // tau, w, x, obj, flops, w3
static const int kOutInts = 1 + 8;

struct wbc_ctx {
    int device;
    int max_batch;
    int sm_count;
    Params params;
    cudaStream_t stream;
    cudaEvent_t ev0, ev1, ev2;
    double* recs;        // [max_batch][QPREC_DOUBLES]
    double* yd;          // [6][max_batch]
    double* yw;
    double* yg;          // [6][max_batch] ygamma of the second-order observer
    double* w_dev;       // [6][max_batch] (when the caller passes no w)
    double* tau_prev;    // [12][max_batch] last good torque per instance index (hold_tau_on_failure)
    double* scratch;     // [nslots][gl::TOTAL] one block per solve in flight (the monolithic kernels use the first nblocks)
    double* kkt;         // [nblocks][gl::KKT_DOUBLES] literal multiplier update's matrix, one per resident warp
    int nslots;          // solves in flight in the staged solver (2 per resident warp)
    StageCtl* sq_ctl;    // staged solver: counters
    int* sq_ring;        // staged solver: rings [3][sq_rsize]
    int sq_rsize;
    int staged;          // 0: wbc_solve_kernel, 1: wbc_solve_staged_kernel, 2 (default): by batch size (staged from staged_min_n instances)
    int staged_min_n;
    unsigned* cycles;    // [max_batch] solve durations of the last cycle when express lanes were on (the cost array then ranks by flop count)
    int cycles_valid;
    int* lanes;          // [LANES_INTS] express-lane counters of the solve launch (zeroed by the front kernel)
    int xl_period, xl_keep, xl_min_n, xl_warps;
    float xl_time_scale;    // express lanes: every xl_period-th SM pair keeps xl_keep warps per SM; batches from xl_min_n instances
    double xl_head_mult; // express range of the dispatch order = xl_head_mult x the number of express warps
    int front_leg;       // 1 (default): wbc_front_leg_kernel, four lanes per instance; 0: wbc_front_kernel, a thread per instance (WBC_FRONT=thread)
    int last_staged;     // which kernel the last wbc_cycle launched
    int m_period, m_group;   // SM roles of the staged solver
    unsigned long long* prof;   // [prof_rows][12] per-warp profile of the last staged or exact-mode launch (WBC_STAGE_PROF=1)
    int prof_rows;
    int* queue;          // [cost histogram A | work-queue counter | dispatch cursors | cost histogram B]: counter and cursors sit between
                         // the two histograms so that "counter + cursors + the histogram being filled" is one contiguous memset either way
    unsigned* cost;      // [max_batch] duration of each instance's last solve (1024-cycle units)
    int* order;          // [max_batch] dispatch order built by the front kernel
    int order_n;         // batch size `cost` and the current histogram describe (0 = none)
    int hist_sel;        // which histogram the last solve filled
    int nblocks, threads;   // solver launch shape
    int occ_per_sm;         // resident solver CTAs per SM (occupancy calculator)
    int occ_forced;         // WBC_SOLVE_CTAS_PER_SM was given: no per-launch adaptation
    int last_grid;          // solver grid of the last wbc_cycle
    int solve_smem;         // dynamic shared memory per solver CTA (sl::BYTES, or padded by WBC_SOLVE_CTAS_PER_SM)
    int exact_per_sm;       // exact-mode kernel (WBC_QP_EXACT): resident CTAs per SM (occupancy calculator) ...
    int exact_blocks;       // ... its persistent grid: every resident CTA that has a scratch block (wbcdual::SCRATCH_DOUBLES each)
    unsigned* aset;         // [4][max_batch] exact mode: each instance's active inequality rows (words 0..2) and contact mode + 1 (word 3,
                            // 0 = none) of its last exact-mode solve; the warm set of WBC_QP_WARM
    // staging for WBC_HOST_PTRS
    double* d_in;        // [93+40][max_batch]
    double* d_out;       // [62][max_batch]
    int* d_mode;         // [max_batch]
    int* d_iout;         // [9][max_batch]
    double* h_pin;       // pinned bounce buffer, max(in,out) doubles
    int* h_pin_i;
    size_t dense_cap;    // bytes of dense staging
    double* d_dense;     // dense QP staging (Q, c, L, x)
    // on-device trajectory sampling (wbc_traj.cuh): plan tables and the last samples, ld = max_batch
    int traj_nseg, traj_n;        // segments per spline of the uploaded plan (0 = none), instances it covers
    double* traj_dur;             // [4 * TRAJ_MAX_SEG][max_batch]
    double* traj_nodes;           // [4 * (TRAJ_MAX_SEG + 1) * 6][max_batch]
    double* traj_s;               // [36][max_batch] samples of the last wbc_sample_trajectory(out = NULL)
    double* traj_t;               // [max_batch] staging of per-instance times
    int traj_sampled_n;           // instances the samples cover (0 = none)
    float front_ms, solve_ms;
    int launches;
    int last_n;          // instances of the last wbc_cycle (wbc_plant_step reads their records)
};

extern "C" {

void wbc_default_params(wbc_params* p)
{
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->kcom = 2500.0; p->dcom = 50.0; p->q1_weight = 50.0; p->slack_weight = 1.0e8; p->mu = 0.6; p->tau_max = 60.0;
    p->joint_dt = 0.025; p->kp_sw = 300.0; p->kd_sw = 20.0; p->g_acc = 9.81; p->obs_gain = 10.0; p->obs_dt = 0.0025;
    p->gravity[0] = 0.0; p->gravity[1] = 0.0; p->gravity[2] = -9.8;
    p->qp_epsx = 1.0e-2; p->qp_rho = 1.0e4; p->qp_outerits = 5;
    p->observer_enabled = 1; p->fix_swing_rhs = 0; p->qp_literal_kkt = 0; p->hold_tau_on_failure = 0;
    p->obs_gain2 = 1.0; p->obs_order = 1; p->obs_form = 0;
}

void wbc_default_contact_params(wbc_contact_params* cp)
{
    if (!cp) return;
    memset(cp, 0, sizeof(*cp));
    cp->beta = 0.2; cp->eps = 1.0e-8; cp->margin = 2.0e-3; cp->max_iter = 64;
}

void wbc_default_gait_params(wbc_gait_params* gp)
{
    if (!gp) return;
    memset(gp, 0, sizeof(*gp));
    gp->stance_cycles = 46; gp->swing_cycles = 46; gp->step_height = 0.03;
    gp->k_v = 0.1; gp->max_step = 0.1; gp->acc_lin = 1.0; gp->acc_yaw = 2.0; gp->leash = 0.05;
}

const char* wbc_last_error(void) { return g_err; }
const char* wbc_version(void) { return "wbc_b200 0.1 (sm_100a)"; }

int wbc_destroy(wbc_ctx* c)
{
    if (!c) return WBC_OK;
    cudaSetDevice(c->device);
    cudaFree(c->recs); cudaFree(c->yd); cudaFree(c->yw); cudaFree(c->yg); cudaFree(c->w_dev); cudaFree(c->tau_prev); cudaFree(c->scratch); cudaFree(c->kkt); cudaFree(c->sq_ctl); cudaFree(c->sq_ring); cudaFree(c->prof); cudaFree(c->queue); cudaFree(c->lanes); cudaFree(c->cost); cudaFree(c->cycles); cudaFree(c->order); cudaFree(c->aset);
    cudaFree(c->traj_dur); cudaFree(c->traj_nodes); cudaFree(c->traj_s); cudaFree(c->traj_t);
    cudaFree(c->d_in); cudaFree(c->d_out); cudaFree(c->d_mode); cudaFree(c->d_iout); cudaFree(c->d_dense);
    if (c->h_pin) cudaFreeHost(c->h_pin);
    if (c->h_pin_i) cudaFreeHost(c->h_pin_i);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->ev2) cudaEventDestroy(c->ev2);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return WBC_OK;
}

int wbc_create(wbc_ctx** out, int device, int max_batch, const wbc_params* params)
{
    if (!out || max_batch <= 0) return fail(WBC_EINVAL, "wbc_create: bad arguments");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return fail(WBC_ENODEV, "no CUDA device (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(WBC_EINVAL, "wbc_create: device ordinal out of range");
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(WBC_ENODEV, "device is not sm_100 class; this library ships sm_100a code only");
    CU(cudaSetDevice(device));
    wbc_ctx* c = new (std::nothrow) wbc_ctx();
    if (!c) return fail(WBC_ENOMEM, "out of host memory");
    memset(c, 0, sizeof(*c));
    c->device = device; c->max_batch = max_batch; c->sm_count = prop.multiProcessorCount;
    wbc_params def;
    wbc_default_params(&def);
    memcpy(&c->params, params ? params : &def, sizeof(Params));
    const size_t nb = (size_t)max_batch;
    c->threads = SOLVE_T;
    c->solve_smem = sl::BYTES;
    int per_sm = SOLVE_CTAS_PER_SM;
    // occupancy experiment knob: fewer resident solver warps per SM (the shared-memory request is padded so that
    // exactly that many CTAs fit); used by tools/ to measure how throughput scales with resident warps
    if (const char* ev = getenv("WBC_SOLVE_CTAS_PER_SM")) {
        const int k = atoi(ev);
        c->occ_forced = 1;
        if (k >= 1 && k < SOLVE_CTAS_PER_SM) {
            per_sm = k;
            c->solve_smem = (((228 * 1024) / k - 1024) / 16) * 16;
            if (c->solve_smem > 227 * 1024) c->solve_smem = 227 * 1024;
        }
    }
    // L1 experiment knob: k resident solver warps per SM WITHOUT padding the request -- the shared-memory carve-out is set to what
    // k CTAs need and the rest of the SM's 256 KB stays L1 (12 CTAs leave 28 KB of it; 8 leave 92 KB, 10 leave 60 KB)
    int l1_ctas = 0;
    if (const char* ev = getenv("WBC_SOLVE_L1_CTAS")) {
        const int k = atoi(ev);
        if (k >= 1 && k <= SOLVE_CTAS_PER_SM) { l1_ctas = k; per_sm = k; c->occ_forced = 1; c->solve_smem = sl::BYTES; }
    }
    c->nblocks = c->sm_count * per_sm;
    // one scratch block per resident solver warp a launch can use (a launch never has more CTAs than instances)
    const long nteams = c->nblocks < max_batch ? c->nblocks : max_batch;
    cudaError_t e = cudaSuccess;
#define TRY(call) if (e == cudaSuccess) e = (call)
    TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    TRY(cudaEventCreate(&c->ev0)); TRY(cudaEventCreate(&c->ev1)); TRY(cudaEventCreate(&c->ev2));
    TRY(cudaMalloc(&c->recs, nb * QPREC_DOUBLES * sizeof(double)));
    TRY(cudaMalloc(&c->yd, nb * 6 * sizeof(double)));
    TRY(cudaMalloc(&c->yw, nb * 6 * sizeof(double)));
    TRY(cudaMalloc(&c->yg, nb * 6 * sizeof(double)));
    TRY(cudaMalloc(&c->w_dev, nb * 6 * sizeof(double)));
    TRY(cudaMalloc(&c->tau_prev, nb * 12 * sizeof(double)));
    TRY(cudaMemset(c->tau_prev, 0, nb * 12 * sizeof(double)));
    // Which solver kernel.  wbc_solve_kernel: one warp per solve.  wbc_solve_staged_kernel: stage tasks with SM roles -- the QQP
    // iteration (its hot code fits an SM's instruction cache) on three SM pairs of five, everything else on the other two.
    // Measured on B200 (profiles/README.md, round 2): the staged kernel was 19 % faster at 65 536 instances (37.1 against 44.1 ms) and
    // slower at 4 096 (4.0 against 3.3 ms: a solve is eleven hand-overs and the batch is only 2.3 solves per warp), so the choice
    // goes by batch size; WBC_SOLVER = mono | staged forces one, WBC_STAGED_MIN_N moves the threshold.  After the inlining of the
    // round's last step the one-warp-per-solve kernel gained more than the staged one and the crossover moved from 12 288 to
    // ~49 152 instances (profiles/r02_az_crossover.txt: 24 576: 13.33 against 13.98 ms, 49 152: 25.05 / 24.99, 65 536: 33.03 / 32.33).
    c->staged = 2; c->staged_min_n = 49152; c->m_period = (3 << 16) | (7 << 8) | 25; c->m_group = 2;     // of every 25 SM pairs: 3 SETUP, 7 POST, 15 QQP (0.5 % over 2 POST/SETUP in 5)
    if (const char* ev = getenv("WBC_SOLVER")) c->staged = strcmp(ev, "staged") == 0 ? 1 : (strcmp(ev, "mono") == 0 ? 0 : 2);
    if (const char* ev = getenv("WBC_STAGED_MIN_N")) c->staged_min_n = atoi(ev);
    c->front_leg = 1;
    // express lanes (ExpressLanes): WBC_EXPRESS = "period,keep,head multiplier,min n"; period 0 switches them off
    c->xl_period = 9; c->xl_keep = 4; c->xl_head_mult = 1.0; c->xl_min_n = 2048; c->xl_warps = 12; c->xl_time_scale = 0.0f;
    if (const char* ev = getenv("WBC_EXPRESS")) {
        int a = 9, b = 4, d = 2048, wps = 12; double m = 2.0, ts = 0.0;
        const int got = sscanf(ev, "%d,%d,%lf,%d,%d,%lf", &a, &b, &m, &d, &wps, &ts);
        if (got >= 6 && ts >= 0.0) c->xl_time_scale = (float)ts;
        if (got >= 5 && wps >= 4 && wps <= 12) c->xl_warps = wps;
        if (got >= 1 && a >= 0 && a < 75) c->xl_period = a;
        if (got >= 2 && b >= 1 && b <= 12) c->xl_keep = b;
        if (got >= 3 && m >= 0.0) c->xl_head_mult = m;
        if (got >= 4 && d >= 0) c->xl_min_n = d;
    }
    if (const char* ev = getenv("WBC_FRONT")) c->front_leg = strcmp(ev, "thread") != 0;
    if (const char* ev = getenv("WBC_STAGE_ROLES")) {        // "nS,nP/den"
        int a = 0, b = 2, d = 5;
        if (sscanf(ev, "%d,%d/%d", &a, &b, &d) == 3 && d > 0 && d < 256 && a >= 0 && b >= 0 && a + b <= d) c->m_period = (a << 16) | (b << 8) | d;
    }
    if (const char* ev = getenv("WBC_STAGE_M_GROUP")) c->m_group = atoi(ev) > 0 ? atoi(ev) : 1;
    double slots_per_warp = 2.0;     // measured at 65 536 instances: 1.0 -> 42.7 ms, 1.5 -> 39.2, 2.0 -> 39.1, 3.0 -> 38.9 (profiles/README.md)
    if (const char* ev = getenv("WBC_STAGE_SLOTS_PER_WARP")) slots_per_warp = atof(ev) >= 1.0 ? atof(ev) : 1.0;
    const long want_slots = (long)((double)nteams * slots_per_warp + 0.5);
    c->nslots = (int)(want_slots < (long)max_batch ? want_slots : (nteams > max_batch ? nteams : max_batch));
    if (c->nslots < nteams) c->nslots = (int)nteams;
    c->sq_rsize = 1;
    while (c->sq_rsize < c->nslots) c->sq_rsize <<= 1;
    TRY(cudaMalloc(&c->scratch, (size_t)c->nslots * gl::TOTAL * sizeof(double)));
    TRY(cudaMalloc(&c->kkt, (size_t)nteams * gl::KKT_DOUBLES * sizeof(double)));
    TRY(cudaMalloc(&c->sq_ctl, sizeof(StageCtl)));
    TRY(cudaMalloc(&c->sq_ring, (size_t)3 * c->sq_rsize * sizeof(int)));
    if (getenv("WBC_STAGE_PROF")) { TRY(cudaMalloc(&c->prof, (size_t)nteams * 12 * sizeof(unsigned long long))); TRY(cudaMemset(c->prof, 0, (size_t)nteams * 12 * sizeof(unsigned long long))); c->prof_rows = (int)nteams; }
    TRY(cudaMalloc(&c->queue, (1 + 3 * ORD_NB) * sizeof(int)));
    TRY(cudaMalloc(&c->lanes, LANES_INTS * sizeof(int)));
    TRY(cudaMemset(c->lanes, 0, LANES_INTS * sizeof(int)));
    TRY(cudaMemset(c->queue, 0, (1 + 3 * ORD_NB) * sizeof(int)));
    TRY(cudaMalloc(&c->cost, nb * sizeof(unsigned)));
    TRY(cudaMalloc(&c->aset, nb * 4 * sizeof(unsigned)));
    TRY(cudaMemset(c->aset, 0, nb * 4 * sizeof(unsigned)));
    TRY(cudaMalloc(&c->cycles, nb * sizeof(unsigned)));
    TRY(cudaMalloc(&c->order, nb * sizeof(int)));
    TRY(cudaMalloc(&c->d_in, nb * (kInDoublesNoTerrain + 41) * sizeof(double)));
    TRY(cudaMalloc(&c->d_out, nb * kOutDoubles * sizeof(double)));
    TRY(cudaMalloc(&c->d_mode, nb * sizeof(int)));
    TRY(cudaMalloc(&c->d_iout, nb * kOutInts * sizeof(int)));
    TRY(cudaMallocHost(&c->h_pin, nb * (kInDoublesNoTerrain + 41) * sizeof(double)));
    TRY(cudaMallocHost(&c->h_pin_i, nb * kOutInts * sizeof(int)));
    TRY(cudaMemset(c->yd, 0, nb * 6 * sizeof(double)));
    TRY(cudaMemset(c->yw, 0, nb * 6 * sizeof(double)));
    TRY(cudaMemset(c->yg, 0, nb * 6 * sizeof(double)));
    TRY(cudaMemset(c->scratch, 0, (size_t)c->nslots * gl::TOTAL * sizeof(double)));
    TRY(cudaMemset(c->kkt, 0, (size_t)nteams * gl::KKT_DOUBLES * sizeof(double)));
    TRY(cudaFuncSetAttribute(wbc_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));      // padded requests: see wbc_cycle
    TRY(cudaFuncSetAttribute(wbc_solve_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, c->solve_smem));
    TRY(cudaFuncSetAttribute(wbc_solve_staged_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TRY(cudaFuncSetAttribute(wbc_dense_qp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, c->solve_smem));
    TRY(cudaFuncSetAttribute(wbc_solve_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TRY(cudaFuncSetAttribute(wbc_dense_qp_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TRY(cudaFuncSetAttribute(wbc_solve_exact_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TRY(cudaFuncSetAttribute(wbc_solve_exact_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TRY(cudaFuncSetAttribute(wbc_solve_exact_kernel<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TRY(cudaFuncSetAttribute(wbc_solve_exact_kernel<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TRY(cudaFuncSetAttribute(wbc_dense_qp_exact_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    TRY(cudaFuncSetAttribute(wbc_dense_qp_exact_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    if (l1_ctas > 0) {
        const int pct = (int)((100L * l1_ctas * (sl::BYTES + 1024) + 228 * 1024 - 1) / (228 * 1024));
        TRY(cudaFuncSetAttribute(wbc_solve_staged_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct > 100 ? 100 : pct));
        TRY(cudaFuncSetAttribute(wbc_solve_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct > 100 ? 100 : pct));
    }
    if (e == cudaSuccess) {
        // the persistent grid is exactly the resident CTAs: more would queue behind whole solves
        int occ = 0;
        int occ2 = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, wbc_solve_staged_kernel, SOLVE_T, (size_t)c->solve_smem);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, wbc_solve_kernel, SOLVE_T, (size_t)c->solve_smem);
        if (occ2 < occ) occ = occ2;
        if (e == cudaSuccess && occ >= 1) {
            c->occ_per_sm = occ;
            if (c->nblocks > c->sm_count * occ) c->nblocks = c->sm_count * occ;
            if (l1_ctas > 0 && l1_ctas < occ) c->occ_per_sm = l1_ctas;
        }
    }
    if (e == cudaSuccess) {
        // exact mode: the scratch blocks of the DENSE-AUL kernels, carved into the exact solver's smaller ones
        int occ = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, wbc_solve_exact_kernel<false>, EXACT_T, (size_t)wbcdual::ds::BYTES);
        const long cap = (long)c->nslots * gl::TOTAL / wbcdual::SCRATCH_DOUBLES;
        c->exact_per_sm = occ > 0 ? occ : 1;
        const long want = (long)c->sm_count * c->exact_per_sm;
        c->exact_blocks = (int)(want < cap ? want : cap);
    }
#undef TRY
    if (e != cudaSuccess) {
        fail(e == cudaErrorMemoryAllocation ? WBC_ENOMEM : WBC_ECUDA, "wbc_create: %s", cudaGetErrorString(e));
        wbc_destroy(c);
        return e == cudaErrorMemoryAllocation ? WBC_ENOMEM : WBC_ECUDA;
    }
    *out = c;
    return WBC_OK;
}

int wbc_set_params(wbc_ctx* c, const wbc_params* p)
{
    if (!c || !p) return fail(WBC_EINVAL, "wbc_set_params: null argument");
    memcpy(&c->params, p, sizeof(Params));
    return WBC_OK;
}

int wbc_set_observer_state(wbc_ctx* c, int n, const double* yd, const double* yw, long ld)
{
    if (!c || !yd || !yw || n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "wbc_set_observer_state: bad arguments");
    if (n == 0) return WBC_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpy2D(c->yd, (size_t)c->max_batch * 8, yd, (size_t)ld * 8, (size_t)n * 8, 6, cudaMemcpyHostToDevice));
    CU(cudaMemcpy2D(c->yw, (size_t)c->max_batch * 8, yw, (size_t)ld * 8, (size_t)n * 8, 6, cudaMemcpyHostToDevice));
    return WBC_OK;
}

int wbc_set_observer_state2(wbc_ctx* c, int n, const double* yg, long ld)
{
    if (!c || !yg || n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "wbc_set_observer_state2: bad arguments");
    if (n == 0) return WBC_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpy2D(c->yg, (size_t)c->max_batch * 8, yg, (size_t)ld * 8, (size_t)n * 8, 6, cudaMemcpyHostToDevice));
    return WBC_OK;
}

int wbc_get_observer_state2(wbc_ctx* c, int n, double* yg, long ld)
{
    if (!c || !yg || n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "wbc_get_observer_state2: bad arguments");
    if (n == 0) return WBC_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpy2D(yg, (size_t)ld * 8, c->yg, (size_t)c->max_batch * 8, (size_t)n * 8, 6, cudaMemcpyDeviceToHost));
    return WBC_OK;
}

int wbc_get_observer_state(wbc_ctx* c, int n, double* yd, double* yw, long ld)
{
    if (!c || !yd || !yw || n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "wbc_get_observer_state: bad arguments");
    if (n == 0) return WBC_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpy2D(yd, (size_t)ld * 8, c->yd, (size_t)c->max_batch * 8, (size_t)n * 8, 6, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy2D(yw, (size_t)ld * 8, c->yw, (size_t)c->max_batch * 8, (size_t)n * 8, 6, cudaMemcpyDeviceToHost));
    return WBC_OK;
}

// Front kernel block size: small batches use small blocks so that every SM gets work.
static int front_threads(const wbc_ctx* c, int n)
{
    if (n >= c->sm_count * 64 * 4) return 64;
    return 32;
}

static int check_inputs(const wbc_inputs* in, int n, bool sampled_traj = false)
{
    if (!in) return fail(WBC_EINVAL, "null wbc_inputs");
    if (in->ld < n) return fail(WBC_EINVAL, "wbc_inputs.ld < n");
    const void* req[] = {in->base_pos, in->base_rot, in->base_rpy, in->base_vel, in->q, in->dq, in->com_des_pos, in->com_des_vel,
                         in->com_des_acc, in->sw_des_pos, in->sw_des_vel, in->sw_des_acc, in->foot_force, in->mode};
    for (int f = 0; f < 14; f++) {
        if (sampled_traj && f >= 6 && f <= 11) continue;      // com_des_*, sw_des_*: taken from the ctx's samples
        if (!req[f]) return fail(WBC_EINVAL, "wbc_inputs: a required array is NULL (only `terrain` may be)");
    }
    return WBC_OK;
}

// Page-locked host memory (cudaMallocHost / cudaHostRegister) can be the source or target of an asynchronous copy
// directly; pageable memory goes through the ctx's pinned bounce buffer.
static bool is_pinned_host(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// Stage host SoA inputs into the ctx's device buffers, one H2D copy per field so that the DMA of a field overlaps the
// host-side packing of the next: straight from the caller's arrays when they are page-locked, else through the
// pinned bounce buffer.
static int stage_inputs(wbc_ctx* c, int n, const wbc_inputs* in, cudaStream_t s, DevInputs* dev, bool slab, bool sampled_traj = false)
{
    const double* src[15] = {in->base_pos, in->base_rot, in->base_rpy, in->base_vel, in->q, in->dq, in->com_des_pos, in->com_des_vel,
                             in->com_des_acc, in->sw_des_pos, in->sw_des_vel, in->sw_des_acc, in->foot_force, in->terrain, in->obs_gain};
    const double** dst[15] = {&dev->base_pos, &dev->base_rot, &dev->base_rpy, &dev->base_vel, &dev->q, &dev->dq, &dev->com_des_pos,
                              &dev->com_des_vel, &dev->com_des_acc, &dev->sw_des_pos, &dev->sw_des_vel, &dev->sw_des_acc,
                              &dev->foot_force, &dev->terrain, &dev->obs_gain};
    size_t off = 0;
    const size_t row = (size_t)n * sizeof(double);
    // a run of page-locked fields that are adjacent in host memory in field order (one slab, ld == n) is one copy
    const double* run_src = nullptr;
    size_t run_off = 0, run_rows = 0;
    for (int f = 0; f < 15; f++) {
        const int K = kInFieldK[f];
        if (sampled_traj && f >= 6 && f <= 11) {
            // desired-trajectory rows: filled on the device from the ctx's samples (one strided D2D copy, below)
            if (run_src) { CU(cudaMemcpyAsync(c->d_in + run_off, run_src, run_rows * row, cudaMemcpyHostToDevice, s)); run_src = nullptr; }
            if (f == 6)
                CU(cudaMemcpy2DAsync(c->d_in + off, row, c->traj_s, (size_t)c->max_batch * sizeof(double), row, wbc::TRAJ_OUT_ROWS, cudaMemcpyDeviceToDevice, s));
            *dst[f] = c->d_in + off;
            off += (size_t)K * n;
            continue;
        }
        if (!src[f]) { *dst[f] = nullptr; continue; }
        const bool pinned = is_pinned_host(src[f]);
        if (run_src && !(slab && pinned && in->ld == n && src[f] == run_src + run_rows * n)) {
            CU(cudaMemcpyAsync(c->d_in + run_off, run_src, run_rows * row, cudaMemcpyHostToDevice, s));
            run_src = nullptr;
        }
        if (slab && pinned && in->ld == n) {
            if (!run_src) { run_src = src[f]; run_off = off; run_rows = 0; }
            run_rows += K;
        } else if (pinned) {
            CU(cudaMemcpy2DAsync(c->d_in + off, row, src[f], (size_t)in->ld * sizeof(double), row, K, cudaMemcpyHostToDevice, s));
        } else {
            for (int k = 0; k < K; k++) memcpy(c->h_pin + off + (size_t)k * n, src[f] + (size_t)k * in->ld, row);
            CU(cudaMemcpyAsync(c->d_in + off, c->h_pin + off, row * K, cudaMemcpyHostToDevice, s));
        }
        *dst[f] = c->d_in + off;
        off += (size_t)K * n;
    }
    if (run_src) CU(cudaMemcpyAsync(c->d_in + run_off, run_src, run_rows * row, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(c->d_mode, in->mode, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    dev->mode = c->d_mode;
    dev->ld = n;
    return WBC_OK;
}

static void to_dev_inputs(const wbc_inputs* in, DevInputs* d)
{
    d->base_pos = in->base_pos; d->base_rot = in->base_rot; d->base_rpy = in->base_rpy; d->base_vel = in->base_vel;
    d->q = in->q; d->dq = in->dq; d->com_des_pos = in->com_des_pos; d->com_des_vel = in->com_des_vel; d->com_des_acc = in->com_des_acc;
    d->sw_des_pos = in->sw_des_pos; d->sw_des_vel = in->sw_des_vel; d->sw_des_acc = in->sw_des_acc; d->foot_force = in->foot_force;
    d->terrain = in->terrain; d->mode = in->mode; d->obs_gain = in->obs_gain; d->ld = in->ld;
}

int wbc_cycle(wbc_ctx* c, int n, const wbc_inputs* in, const wbc_outputs* out, void* cuda_stream, unsigned flags)
{
    if (!c || !out) return fail(WBC_EINVAL, "wbc_cycle: null argument");
    if (n < 0 || n > c->max_batch) return fail(WBC_EINVAL, "wbc_cycle: n outside [0, max_batch]");
    if (n == 0) { c->launches = 0; return WBC_OK; }
    const bool sampled = (flags & WBC_SAMPLED_TRAJ) != 0;
    int rc = check_inputs(in, n, sampled);
    if (rc) return rc;
    if (!out->tau || out->ld < n) return fail(WBC_EINVAL, "wbc_cycle: outputs.tau is required and outputs.ld >= n");
    const bool dev_ptrs = (flags & WBC_DEVICE_PTRS) != 0;
    const bool exact = (flags & WBC_QP_EXACT) != 0;
    const bool warm = (flags & WBC_QP_WARM) != 0;
    if (warm && !exact) return fail(WBC_EINVAL, "wbc_cycle: WBC_QP_WARM is only valid together with WBC_QP_EXACT");
    if (sampled && c->traj_sampled_n < n) return fail(WBC_EINVAL, "wbc_cycle: WBC_SAMPLED_TRAJ without a wbc_sample_trajectory(out = NULL) covering n instances");
    if (sampled && dev_ptrs && in->ld != c->max_batch)
        return fail(WBC_EINVAL, "wbc_cycle: WBC_SAMPLED_TRAJ with device pointers needs inputs.ld == max_batch (or sample into your own arrays)");
    CU(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;

    DevInputs din;
    SolveOut so;
    double* w_ptr;
    long w_ld;
    double* w3_ptr;
    long w3_ld;
    if (dev_ptrs) {
        to_dev_inputs(in, &din);
        if (sampled) {
            const size_t blk = (size_t)6 * c->max_batch;
            din.com_des_pos = c->traj_s; din.com_des_vel = c->traj_s + blk; din.com_des_acc = c->traj_s + 2 * blk;
            din.sw_des_pos = c->traj_s + 3 * blk; din.sw_des_vel = c->traj_s + 4 * blk; din.sw_des_acc = c->traj_s + 5 * blk;
        }
        so.tau = out->tau; so.x = out->x; so.qp_obj = out->qp_obj; so.status = out->status; so.qp_info = out->qp_info;
        so.qp_flops = out->qp_flops; so.ld = out->ld;
        w_ptr = out->w ? out->w : c->w_dev;
        w_ld = out->w ? out->ld : c->max_batch;
        w3_ptr = out->w3; w3_ld = out->ld;
    } else {
        rc = stage_inputs(c, n, in, s, &din, (flags & WBC_HOST_SLAB) != 0, sampled);
        if (rc) return rc;
        so.tau = c->d_out; so.x = out->x ? c->d_out + 18L * n : nullptr; so.qp_obj = out->qp_obj ? c->d_out + 48L * n : nullptr;
        so.qp_flops = out->qp_flops ? c->d_out + 49L * n : nullptr;
        so.status = out->status ? c->d_iout : nullptr; so.qp_info = out->qp_info ? c->d_iout + n : nullptr; so.ld = n;
        w_ptr = c->d_out + 12L * n;
        w_ld = n;
        w3_ptr = out->w3 ? c->d_out + 50L * n : nullptr; w3_ld = n;
    }
    so.tau_prev = c->tau_prev; so.ld_prev = c->max_batch;
    FrontState st;
    st.yd = c->yd; st.yw = c->yw; st.yg = c->yg; st.ld = c->max_batch;
    st.w3 = w3_ptr; st.w3_ld = w3_ld;
    DevDebug nodbg;
    memset(&nodbg, 0, sizeof(nodbg));
    // dispatch order: longest solve first, predicted by each instance's previous solve (same batch size only)
    int* hist_ab[2] = {c->queue, c->queue + 2 * ORD_NB + 1};
    int* counter = c->queue + ORD_NB;
    int* hist_prev = hist_ab[c->hist_sel];
    int* hist_next = hist_ab[c->hist_sel ^ 1];
    const bool ordered = !(flags & WBC_FIFO_DISPATCH) && c->order_n == n && n > 1;
    DispatchOrder ord;
    ord.cost = ordered ? c->cost : nullptr; ord.hist = hist_prev; ord.cursor = counter + 1; ord.order = c->order;
    // express lanes for the one-warp-per-solve kernel on a batch of a few solves per warp (see ExpressLanes)
    const bool staged_sel = !exact && (c->staged == 1 || (c->staged == 2 && n >= c->staged_min_n));
    const bool express = !exact && !staged_sel && c->xl_period > 0 && !c->occ_forced && c->occ_per_sm >= 12 && n >= c->xl_min_n;
    ord.lanes = express ? c->lanes : nullptr;
    // one memset: counter, cursors and the histogram this cycle fills (A lies just before the counter, B just after the cursors)
    CU(cudaMemsetAsync((c->hist_sel ^ 1) == 0 ? c->queue : counter, 0, (1 + 2 * ORD_NB) * sizeof(int), s));
    CU(cudaEventRecord(c->ev0, s));
    const int fthreads = front_threads(c, n);
    StageReset sr;
    memset(&sr, 0, sizeof(sr));
    const bool staged_next = !exact && (c->staged == 1 || (c->staged == 2 && n >= c->staged_min_n));
    if (staged_next) {
        sr.ctl = reinterpret_cast<int*>(c->sq_ctl); sr.nctl = (int)(sizeof(StageCtl) / sizeof(int));
        sr.free_tail_index = (int)(offsetof(StageCtl, tail) / sizeof(int)) + SQ_FREE * 32;
        sr.free_avail_index = (int)(offsetof(StageCtl, avail) / sizeof(int)) + SQ_FREE * 32;
        sr.ring = c->sq_ring; sr.rsize = c->sq_rsize; sr.nslots = c->nslots;
    }
    if (c->front_leg) {
        // four lanes per instance; 64-thread CTAs (16 instances) keep a small batch spread over every SM
        const int lt = (4L * n >= (long)c->sm_count * 128 * 4) ? 128 : 64;
        wbc_front_leg_kernel<<<(unsigned)((4L * n + lt - 1) / lt), lt, 0, s>>>(c->params, din, st, n, c->recs, w_ptr, w_ld, ord, sr);
    } else {
        wbc_front_kernel<<<(n + fthreads - 1) / fthreads, fthreads, 0, s>>>(c->params, din, st, n, c->recs, w_ptr, w_ld, nodbg, 0, ord, sr);
    }
    CU(cudaEventRecord(c->ev1, s));
    // Resident solver warps for this batch.  Large batches take every warp that fits (12 per SM).  A batch of a few thousand is
    // only two or three solves per warp: its step ends with its longest solve, and every solve runs slower the more warps share
    // the SM's instruction supply.  From xl_min_n instances: 12 warps per SM with express lanes for the longest solves
    // (ExpressLanes; 3.05 ms against 3.25 at 4 096 instances).  Below, or with the lanes switched off: 8 warps per SM, which
    // beat a plain 12 by 3 % at 4 096 instances (profiles/README.md).
    int nblocks = c->nblocks;
    int smem = c->solve_smem;
    const bool staged = !exact && (c->staged == 1 || (c->staged == 2 && n >= c->staged_min_n));
    c->last_staged = exact ? 2 : (staged ? 1 : 0);
    ExpressLanes xl;
    xl.lanes = c->lanes; xl.head = 0; xl.period = 0; xl.keep = c->xl_keep; xl.cycles = c->cycles; xl.prof = c->prof; xl.time_scale = c->xl_time_scale;
    c->cycles_valid = 0;
    if (express) {
        // every resident warp (12 per SM); the express SM pairs keep xl_keep warps per SM and serve the head of the order
        int nexp = 0;
        for (int sm = 0; sm < c->sm_count; sm++) nexp += ((sm >> 1) % c->xl_period) == (c->xl_period >> 1);
        xl.period = c->xl_period;
        c->cycles_valid = 1;
        xl.head = (int)(c->xl_head_mult * nexp * c->xl_keep + 0.5);
        if (xl.head > n) xl.head = n;
        if (c->xl_warps < c->occ_per_sm) {         // fewer warps on the regular SMs (padded shared-memory request, as below)
            nblocks = c->xl_warps * c->sm_count;
            smem = (((228 * 1024) / c->xl_warps - 1024) / 16) * 16;
        }
    } else if (exact) {
        // the exact solver's own launch shape: every resident CTA, whatever the batch size
        nblocks = c->exact_blocks;
        smem = wbcdual::ds::BYTES;
    } else if (!staged && c->occ_per_sm > 8 && !c->occ_forced) {
        int per_sm = (int)((double)n / (3.4 * c->sm_count));
        per_sm = per_sm < 8 ? 8 : (per_sm > c->occ_per_sm ? c->occ_per_sm : per_sm);
        if (per_sm < c->occ_per_sm) {
            // the shared-memory request is padded so that exactly per_sm CTAs fit an SM: the block scheduler then spreads
            // the grid evenly instead of filling the first SMs with twelve
            nblocks = per_sm * c->sm_count;
            smem = (((228 * 1024) / per_sm - 1024) / 16) * 16;
        }
    }
    if (n < nblocks) nblocks = n;
    c->last_grid = nblocks;
    if (exact) {
        const int* ordp = ordered ? c->order : nullptr;
        const long mb = c->max_batch;
        if (c->prof && warm)
            wbc_solve_exact_kernel<true, true><<<nblocks, EXACT_T, smem, s>>>(c->params, n, c->recs, so, c->scratch, counter, ordp, c->cost, hist_next,
                                                                              c->prof, c->prof_rows, c->aset, mb);
        else if (c->prof)
            wbc_solve_exact_kernel<true><<<nblocks, EXACT_T, smem, s>>>(c->params, n, c->recs, so, c->scratch, counter, ordp, c->cost, hist_next,
                                                                        c->prof, c->prof_rows, c->aset, mb);
        else if (warm)
            wbc_solve_exact_kernel<false, true><<<nblocks, EXACT_T, smem, s>>>(c->params, n, c->recs, so, c->scratch, counter, ordp, c->cost, hist_next,
                                                                               nullptr, 0, c->aset, mb);
        else
            wbc_solve_exact_kernel<false><<<nblocks, EXACT_T, smem, s>>>(c->params, n, c->recs, so, c->scratch, counter, ordp, c->cost, hist_next,
                                                                         nullptr, 0, c->aset, mb);
    } else if (staged) {
        StageQueues sq;
        sq.ctl = c->sq_ctl; sq.ring = c->sq_ring; sq.rmask = c->sq_rsize - 1; sq.nslots = c->nslots;
        wbc_solve_staged_kernel<<<nblocks, c->threads, c->solve_smem, s>>>(c->params, n, c->recs, so, c->scratch, c->kkt, sq, ordered ? c->order : nullptr,
                                                                      c->cost, hist_next, c->m_period, c->m_group, c->prof);
    } else {
        wbc_solve_kernel<<<nblocks, c->threads, smem, s>>>(c->params, n, c->recs, so, c->scratch, c->kkt, counter, ordered ? c->order : nullptr,
                                                               c->cost, hist_next, xl);
    }
    CU(cudaEventRecord(c->ev2, s));
    CU(cudaGetLastError());
    c->launches = 2;
    c->last_n = n;
    c->hist_sel ^= 1;
    c->order_n = n;
    if (!dev_ptrs) {
        // results: straight into the caller's arrays where they are page-locked, else one D2H of the packed block
        // (tau 12 | w 6 | x 30 | obj 1 | flops 1) into the bounce buffer and a scatter after the synchronisation
        constexpr int NOF = 6;
        struct OutF { double* p; int k0, K; long ld; } of[NOF] = {{out->tau, 0, 12, out->ld}, {out->w, 12, 6, out->ld}, {out->x, 18, 30, out->ld},
                                                                  {out->qp_obj, 48, 1, n}, {out->qp_flops, 49, 1, n}, {out->w3, 50, 12, out->ld}};
        bool direct[NOF];
        const size_t row = (size_t)n * sizeof(double);
        int hi = 0;                                   // bounce prefix, in rows
        for (int f = 0; f < NOF; f++) {
            direct[f] = of[f].p && is_pinned_host(of[f].p);
            if (of[f].p && !direct[f]) hi = of[f].k0 + of[f].K;
        }
        for (int f = 0; f < NOF; f++)
            if (direct[f])
                CU(cudaMemcpy2DAsync(of[f].p, (size_t)of[f].ld * sizeof(double), c->d_out + (size_t)of[f].k0 * n, row, row, of[f].K, cudaMemcpyDeviceToHost, s));
        if (hi) CU(cudaMemcpyAsync(c->h_pin, c->d_out, (size_t)hi * row, cudaMemcpyDeviceToHost, s));
        if (out->status || out->qp_info) CU(cudaMemcpyAsync(c->h_pin_i, c->d_iout, (size_t)kOutInts * n * sizeof(int), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        for (int f = 0; f < NOF; f++)
            if (of[f].p && !direct[f])
                for (int k = 0; k < of[f].K; k++) memcpy(of[f].p + (size_t)k * of[f].ld, c->h_pin + (size_t)(of[f].k0 + k) * n, row);
        if (out->status) memcpy(out->status, c->h_pin_i, (size_t)n * 4);
        if (out->qp_info) for (int k = 0; k < 8; k++) memcpy(out->qp_info + (size_t)k * out->ld, c->h_pin_i + (size_t)(1 + k) * n, (size_t)n * 4);
    } else if (!(flags & WBC_NO_SYNC)) {
        CU(cudaStreamSynchronize(s));
    }
    return WBC_OK;
}

// ---- on-device trajectory sampling (SURVEY.md 8f-1; spline.cc:48-93, polynomial.cc:50-104, main.cpp:1004-1010, 1333-1368)
int wbc_set_trajectory(wbc_ctx* c, int n, const wbc_trajectory* tr, void* cuda_stream, unsigned flags)
{
    if (!c || !tr || !tr->durations || !tr->nodes) return fail(WBC_EINVAL, "wbc_set_trajectory: null argument");
    if (n <= 0 || n > c->max_batch || tr->ld < n) return fail(WBC_EINVAL, "wbc_set_trajectory: n outside (0, max_batch] or ld < n");
    if (tr->nseg < 1 || tr->nseg > wbc::TRAJ_MAX_SEG) return fail(WBC_EINVAL, "wbc_set_trajectory: nseg outside [1, WBC_TRAJ_MAX_SEG]");
    CU(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    const size_t mb = (size_t)c->max_batch;
    if (!c->traj_dur) {
        CU(cudaMalloc(&c->traj_dur, mb * wbc::traj_duration_rows(wbc::TRAJ_MAX_SEG) * sizeof(double)));
        CU(cudaMalloc(&c->traj_nodes, mb * wbc::traj_node_rows(wbc::TRAJ_MAX_SEG) * sizeof(double)));
        CU(cudaMalloc(&c->traj_s, mb * wbc::TRAJ_OUT_ROWS * sizeof(double)));
        CU(cudaMalloc(&c->traj_t, mb * sizeof(double)));
    }
    const cudaMemcpyKind kind = (flags & WBC_DEVICE_PTRS) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const size_t row = (size_t)n * sizeof(double);
    CU(cudaMemcpy2DAsync(c->traj_dur, mb * sizeof(double), tr->durations, (size_t)tr->ld * sizeof(double), row, wbc::traj_duration_rows(tr->nseg), kind, s));
    CU(cudaMemcpy2DAsync(c->traj_nodes, mb * sizeof(double), tr->nodes, (size_t)tr->ld * sizeof(double), row, wbc::traj_node_rows(tr->nseg), kind, s));
    CU(cudaStreamSynchronize(s));            // the caller may free or overwrite its tables on return
    c->traj_nseg = tr->nseg;
    c->traj_n = n;
    c->traj_sampled_n = 0;
    return WBC_OK;
}

int wbc_sample_trajectory(wbc_ctx* c, int n, const double* t, double t_all, const wbc_traj_samples* out, void* cuda_stream, unsigned flags)
{
    if (!c) return fail(WBC_EINVAL, "wbc_sample_trajectory: null ctx");
    if (c->traj_nseg == 0) return fail(WBC_EINVAL, "wbc_sample_trajectory: no plan uploaded (wbc_set_trajectory)");
    if (n <= 0 || n > c->traj_n) return fail(WBC_EINVAL, "wbc_sample_trajectory: n exceeds the uploaded plan");
    const bool dev_ptrs = (flags & WBC_DEVICE_PTRS) != 0;
    if (out) {
        if (out->ld < n) return fail(WBC_EINVAL, "wbc_traj_samples.ld < n");
        const double* req[6] = {out->com_des_pos, out->com_des_vel, out->com_des_acc, out->sw_des_pos, out->sw_des_vel, out->sw_des_acc};
        for (const double* p : req)
            if (!p) return fail(WBC_EINVAL, "wbc_traj_samples: an array is NULL");
    }
    CU(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    const double* dt = t;
    if (t && !dev_ptrs) {
        CU(cudaMemcpyAsync(c->traj_t, t, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, s));
        dt = c->traj_t;
    }
    wbc::TrajOut o;
    const bool to_caller = out && dev_ptrs;
    if (to_caller) {
        o.p[0] = out->com_des_pos; o.p[1] = out->com_des_vel; o.p[2] = out->com_des_acc;
        o.p[3] = out->sw_des_pos; o.p[4] = out->sw_des_vel; o.p[5] = out->sw_des_acc;
        o.ld = out->ld;
    } else {
        for (int b = 0; b < 6; b++) o.p[b] = c->traj_s + (size_t)b * 6 * c->max_batch;
        o.ld = c->max_batch;
    }
    wbc_traj_kernel<<<(n + 127) / 128, 128, 0, s>>>(n, c->traj_nseg, c->traj_dur, c->traj_nodes, c->max_batch, dt, t_all, o);
    CU(cudaGetLastError());
    c->launches = 1;
    if (!to_caller) c->traj_sampled_n = n;
    if (out && !dev_ptrs) {
        double* host[6] = {out->com_des_pos, out->com_des_vel, out->com_des_acc, out->sw_des_pos, out->sw_des_vel, out->sw_des_acc};
        for (int b = 0; b < 6; b++)
            CU(cudaMemcpy2DAsync(host[b], (size_t)out->ld * sizeof(double), c->traj_s + (size_t)b * 6 * c->max_batch, (size_t)c->max_batch * sizeof(double),
                                 (size_t)n * sizeof(double), 6, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    } else if (!(flags & WBC_NO_SYNC) && !dev_ptrs) {
        CU(cudaStreamSynchronize(s));
    }
    return WBC_OK;
}

int wbc_plant_step(wbc_ctx* c, int n, double* base_pos, double* base_vel, double* foot_force, const double* x, const double* push, long ld,
                   void* cuda_stream, unsigned flags)
{
    if (!c || !base_vel || !push) return fail(WBC_EINVAL, "wbc_plant_step: null argument");
    if (foot_force && !x) return fail(WBC_EINVAL, "wbc_plant_step: closed loop (foot_force) needs the QP solution x");
    if (n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "wbc_plant_step: n outside [0, max_batch] or ld < n");
    if (n != c->last_n) return fail(WBC_EINVAL, "wbc_plant_step: n differs from the last wbc_cycle on this ctx");
    if (n == 0) { c->launches = 0; return WBC_OK; }
    CU(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    const bool dev_ptrs = (flags & WBC_DEVICE_PTRS) != 0;
    double *dpos = base_pos, *dvel = base_vel, *dff = foot_force;
    const double *dpush = push, *dx = x;
    long dld = ld;
    if (!dev_ptrs) {
        // convenience path for small host-side rollouts: packed staging in the input buffer
        // layout (doubles per instance): pos 3 | vel 6 | foot_force 12 | push 6 | x[18:30] at rows 18..29 of a 30-row block
        double* h = c->h_pin;
        const size_t N = (size_t)n;
        for (int k = 0; k < 3; k++) memcpy(h + k * N, base_pos ? base_pos + (size_t)k * ld : base_vel, N * 8);
        for (int k = 0; k < 6; k++) memcpy(h + (3 + k) * N, base_vel + (size_t)k * ld, N * 8);
        for (int k = 0; k < 6; k++) memcpy(h + (21 + k) * N, push + (size_t)k * ld, N * 8);
        if (foot_force) for (int k = 0; k < 12; k++) memcpy(h + (45 + k) * N, x + (size_t)(18 + k) * ld, N * 8);
        CU(cudaMemcpyAsync(c->d_in, h, 57 * N * 8, cudaMemcpyHostToDevice, s));
        dpos = base_pos ? c->d_in : nullptr; dvel = c->d_in + 3 * N; dff = foot_force ? c->d_in + 9 * N : nullptr;
        dpush = c->d_in + 21 * N; dx = c->d_in + 27 * N; dld = n;
    }
    wbc_plant_kernel<<<(n + 127) / 128, 128, 0, s>>>(c->params, n, c->recs, dpos, dvel, dff, dx, dpush, dld);
    CU(cudaGetLastError());
    c->launches = 1;
    if (!dev_ptrs) {
        CU(cudaMemcpyAsync(c->h_pin, c->d_in, (size_t)21 * n * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        if (base_pos) for (int k = 0; k < 3; k++) memcpy(base_pos + (size_t)k * ld, c->h_pin + (size_t)k * n, (size_t)n * 8);
        for (int k = 0; k < 6; k++) memcpy(base_vel + (size_t)k * ld, c->h_pin + (size_t)(3 + k) * n, (size_t)n * 8);
        if (foot_force) for (int k = 0; k < 12; k++) memcpy(foot_force + (size_t)k * ld, c->h_pin + (size_t)(9 + k) * n, (size_t)n * 8);
    } else if (!(flags & WBC_NO_SYNC)) {
        CU(cudaStreamSynchronize(s));
    }
    return WBC_OK;
}

int wbc_plant_dynamics_step(wbc_ctx* c, int n, const wbc_plant_state* st, const double* tau, const double* push, long ld, int substeps,
                            double gamma, double* diag, void* cuda_stream, unsigned flags)
{
    if (!c || !st || !tau || !push) return fail(WBC_EINVAL, "wbc_plant_dynamics_step: null argument");
    if (!st->base_pos || !st->base_rot || !st->base_rpy || !st->base_vel || !st->q || !st->dq || !st->foot_force || !st->mode)
        return fail(WBC_EINVAL, "wbc_plant_dynamics_step: a state array is NULL");
    if (n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "wbc_plant_dynamics_step: n outside [0, max_batch] or ld < n");
    if (substeps < 1 || substeps > 1000) return fail(WBC_EINVAL, "wbc_plant_dynamics_step: substeps outside [1, 1000]");
    if (n == 0) { c->launches = 0; return WBC_OK; }
    CU(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    const bool dev_ptrs = (flags & WBC_DEVICE_PTRS) != 0;
    wbc::FdynIO io;
    static const int K[7] = {3, 9, 3, 6, 12, 12, 12};
    double* host[7] = {st->base_pos, st->base_rot, st->base_rpy, st->base_vel, st->q, st->dq, st->foot_force};
    const size_t N = (size_t)n;
    if (dev_ptrs) {
        io.base_pos = st->base_pos; io.base_rot = st->base_rot; io.base_rpy = st->base_rpy; io.base_vel = st->base_vel; io.q = st->q; io.dq = st->dq;
        io.foot_force = st->foot_force; io.mode = st->mode; io.tau = tau; io.push = push; io.diag = diag; io.ld = ld;
    } else {
        // packed staging in the ctx's input buffer: state 57 rows | tau 12 | push 6 | diag 2
        double* h = c->h_pin;
        size_t off = 0;
        for (int f = 0; f < 7; f++)
            for (int k = 0; k < K[f]; k++, off++) memcpy(h + off * N, host[f] + (size_t)k * ld, N * 8);
        for (int k = 0; k < 12; k++, off++) memcpy(h + off * N, tau + (size_t)k * ld, N * 8);
        for (int k = 0; k < 6; k++, off++) memcpy(h + off * N, push + (size_t)k * ld, N * 8);
        CU(cudaMemcpyAsync(c->d_in, h, off * N * 8, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(c->d_mode, st->mode, N * sizeof(int), cudaMemcpyHostToDevice, s));
        double* d = c->d_in;
        io.base_pos = d; io.base_rot = d + 3 * N; io.base_rpy = d + 12 * N; io.base_vel = d + 15 * N; io.q = d + 21 * N; io.dq = d + 33 * N;
        io.foot_force = d + 45 * N; io.tau = d + 57 * N; io.push = d + 69 * N; io.diag = d + 75 * N; io.mode = c->d_mode; io.ld = n;
    }
    wbc_fdyn_kernel<<<(n + 63) / 64, 64, 0, s>>>(c->params, io, n, substeps, gamma);
    CU(cudaGetLastError());
    c->launches = 1;
    if (!dev_ptrs) {
        CU(cudaMemcpyAsync(c->h_pin, c->d_in, (size_t)77 * N * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        size_t off = 0;
        for (int f = 0; f < 7; f++)
            for (int k = 0; k < K[f]; k++, off++) memcpy(host[f] + (size_t)k * ld, c->h_pin + off * N, N * 8);
        if (diag) for (int k = 0; k < 2; k++) memcpy(diag + (size_t)k * ld, c->h_pin + (size_t)(75 + k) * N, N * 8);
    } else if (!(flags & WBC_NO_SYNC)) {
        CU(cudaStreamSynchronize(s));
    }
    return WBC_OK;
}

// The host side of both contact-plant entry points; terrain == nullptr runs the flat kernel (ground_z, mu), otherwise the terrain
// kernel (ground_z then holds the plane offsets, mu is NULL).
static int contact_step(const char* fn, wbc_ctx* c, int n, const wbc_plant_state* st, const double* tau, const double* push,
                        const double* ground_z, const double* mu, const double* terrain, long ld, int substeps, const wbc_contact_params* cp,
                        int* contact, double* diag, int* status, void* cuda_stream, unsigned flags)
{
    if (!c || !st || !tau || !push) return fail(WBC_EINVAL, "%s: null argument", fn);
    if (!st->base_pos || !st->base_rot || !st->base_rpy || !st->base_vel || !st->q || !st->dq || !st->foot_force)
        return fail(WBC_EINVAL, "%s: a state array is NULL", fn);
    if (n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "%s: n outside [0, max_batch] or ld < n", fn);
    if (substeps < 1 || substeps > 1000) return fail(WBC_EINVAL, "%s: substeps outside [1, 1000]", fn);
    wbc_contact_params cpv;
    wbc_default_contact_params(&cpv);
    if (cp) cpv = *cp;
    if (!(cpv.beta >= 0.0 && cpv.beta <= 1.0) || !(cpv.eps >= 0.0 && cpv.eps < 1.0) || !(cpv.margin >= 0.0 && cpv.margin < 1.0e300) ||
        cpv.max_iter < 1)
        return fail(WBC_EINVAL, "%s: contact params outside beta in [0, 1], eps in [0, 1), finite margin >= 0, max_iter >= 1", fn);
    if (n == 0) { c->launches = 0; return WBC_OK; }
    CU(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    const bool dev_ptrs = (flags & WBC_DEVICE_PTRS) != 0;
    const wbc::ContactParams kp = {cpv.beta, cpv.eps, cpv.margin, cpv.max_iter};
    wbc::ContactIO io;
    const double* dterrain = terrain;
    static const int K[7] = {3, 9, 3, 6, 12, 12, 12};
    double* host[7] = {st->base_pos, st->base_rot, st->base_rpy, st->base_vel, st->q, st->dq, st->foot_force};
    const size_t N = (size_t)n;
    if (dev_ptrs) {
        io.base_pos = st->base_pos; io.base_rot = st->base_rot; io.base_rpy = st->base_rpy; io.base_vel = st->base_vel; io.q = st->q; io.dq = st->dq;
        io.foot_force = st->foot_force; io.tau = tau; io.push = push; io.ground_z = ground_z; io.mu = mu;
        io.contact = contact; io.diag = diag; io.status = status; io.ld = ld;
    } else {
        // packed staging in the ctx's input buffer: state 57 rows | tau 12 | push 6 | ground_z 4 | mu 1 | diag 4 | terrain 40;
        // contact 4 and status 1 in the integer output buffer
        double* h = c->h_pin;
        size_t off = 0;
        for (int f = 0; f < 7; f++)
            for (int k = 0; k < K[f]; k++, off++) memcpy(h + off * N, host[f] + (size_t)k * ld, N * 8);
        for (int k = 0; k < 12; k++, off++) memcpy(h + off * N, tau + (size_t)k * ld, N * 8);
        for (int k = 0; k < 6; k++, off++) memcpy(h + off * N, push + (size_t)k * ld, N * 8);
        if (ground_z) for (int k = 0; k < 4; k++) memcpy(h + (off + k) * N, ground_z + (size_t)k * ld, N * 8);
        if (mu) memcpy(h + (off + 4) * N, mu, N * 8);
        CU(cudaMemcpyAsync(c->d_in, h, (off + 5) * N * 8, cudaMemcpyHostToDevice, s));
        double* d = c->d_in;
        if (terrain) {
            for (int k = 0; k < 40; k++) memcpy(h + (84 + k) * N, terrain + (size_t)k * ld, N * 8);
            CU(cudaMemcpyAsync(d + 84 * N, h + 84 * N, 40 * N * 8, cudaMemcpyHostToDevice, s));
            dterrain = d + 84 * N;
        }
        io.base_pos = d; io.base_rot = d + 3 * N; io.base_rpy = d + 12 * N; io.base_vel = d + 15 * N; io.q = d + 21 * N; io.dq = d + 33 * N;
        io.foot_force = d + 45 * N; io.tau = d + 57 * N; io.push = d + 69 * N;
        io.ground_z = ground_z ? d + 75 * N : nullptr; io.mu = mu ? d + 79 * N : nullptr; io.diag = diag ? d + 80 * N : nullptr;
        io.contact = contact ? c->d_iout : nullptr; io.status = status ? c->d_iout + 4 * N : nullptr; io.ld = n;
    }
    if (terrain)
        wbc_contact_terrain_kernel<<<(n + 63) / 64, 64, 0, s>>>(c->params, kp, io, n, substeps, dterrain);
    else
        wbc_contact_kernel<<<(n + 63) / 64, 64, 0, s>>>(c->params, kp, io, n, substeps);
    CU(cudaGetLastError());
    c->launches = 1;
    if (!dev_ptrs) {
        CU(cudaMemcpyAsync(c->h_pin, c->d_in, (size_t)84 * N * 8, cudaMemcpyDeviceToHost, s));
        if (contact || status) CU(cudaMemcpyAsync(c->h_pin_i, c->d_iout, 5 * N * sizeof(int), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        size_t off = 0;
        for (int f = 0; f < 7; f++)
            for (int k = 0; k < K[f]; k++, off++) memcpy(host[f] + (size_t)k * ld, c->h_pin + off * N, N * 8);
        if (diag) for (int k = 0; k < 4; k++) memcpy(diag + (size_t)k * ld, c->h_pin + (size_t)(80 + k) * N, N * 8);
        if (contact) for (int k = 0; k < 4; k++) memcpy(contact + (size_t)k * ld, c->h_pin_i + (size_t)k * N, N * sizeof(int));
        if (status) memcpy(status, c->h_pin_i + 4 * N, N * sizeof(int));
    } else if (!(flags & WBC_NO_SYNC)) {
        CU(cudaStreamSynchronize(s));
    }
    return WBC_OK;
}

int wbc_plant_contact_step(wbc_ctx* c, int n, const wbc_plant_state* st, const double* tau, const double* push, const double* ground_z,
                           const double* mu, long ld, int substeps, const wbc_contact_params* cp, int* contact, double* diag, int* status,
                           void* cuda_stream, unsigned flags)
{
    return contact_step("wbc_plant_contact_step", c, n, st, tau, push, ground_z, mu, nullptr, ld, substeps, cp, contact, diag, status,
                        cuda_stream, flags);
}

int wbc_plant_contact_step_terrain(wbc_ctx* c, int n, const wbc_plant_state* st, const double* tau, const double* push, const double* terrain,
                                   const double* plane_d, long ld, int substeps, const wbc_contact_params* cp, int* contact, double* diag,
                                   int* status, void* cuda_stream, unsigned flags)
{
    if (!terrain) return fail(WBC_EINVAL, "wbc_plant_contact_step_terrain: terrain is NULL (flat ground is wbc_plant_contact_step)");
    return contact_step("wbc_plant_contact_step_terrain", c, n, st, tau, push, plane_d, nullptr, terrain, ld, substeps, cp, contact, diag,
                        status, cuda_stream, flags);
}

// The host side of wbc_gait_init (init = true: k0, no command, outputs or contact flags) and wbc_gait_step.
static int gait_call(const char* fn, bool init, wbc_ctx* c, int n, const wbc_gait_params* gp, wbc_gait_state* gs, const wbc_plant_state* st,
                     const int* k0, const double* cmd, const int* contact, const double* terrain, const double* plane_d, int* mode,
                     const wbc_traj_samples* out, int* status, long ld, void* cuda_stream, unsigned flags)
{
    if (!c || !gs || !st) return fail(WBC_EINVAL, "%s: null argument", fn);
    if (!st->base_pos || !st->base_rot || !st->base_rpy || !st->base_vel || !st->q)
        return fail(WBC_EINVAL, "%s: a state array (base_pos, base_rot, base_rpy, base_vel, q) is NULL", fn);
    if (!gs->phase || !gs->tick || !gs->landed || !gs->com_ref || !gs->v_ref || !gs->liftoff || !gs->target || !gs->offset)
        return fail(WBC_EINVAL, "%s: a gait state array is NULL", fn);
    if (!init && (!mode || !out || !out->com_des_pos || !out->com_des_vel || !out->com_des_acc || !out->sw_des_pos || !out->sw_des_vel ||
                  !out->sw_des_acc))
        return fail(WBC_EINVAL, "%s: mode or an output array is NULL", fn);
    if (plane_d && !terrain) return fail(WBC_EINVAL, "%s: plane_d needs terrain", fn);
    if (n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "%s: n outside [0, max_batch] or ld < n", fn);
    if (!init && out->ld < n) return fail(WBC_EINVAL, "%s: out->ld < n", fn);
    wbc_gait_params g;
    wbc_default_gait_params(&g);
    if (gp) g = *gp;
    const double fin[6] = {g.step_height, g.k_v, g.max_step, g.acc_lin, g.acc_yaw, g.leash};
    bool ok = g.stance_cycles >= 1 && g.swing_cycles >= 2 && g.stance_cycles <= (1 << 20) && g.swing_cycles <= (1 << 20) && g.leash > 0.0;
    for (int k = 0; k < 6; k++) ok = ok && fin[k] >= 0.0 && fin[k] < 1.0e300;
    if (!ok)
        return fail(WBC_EINVAL, "%s: gait params outside stance_cycles in [1, 2^20], swing_cycles in [2, 2^20], finite step_height, k_v, "
                                "max_step, acc_lin, acc_yaw >= 0 and leash > 0", fn);
    if (n == 0) { c->launches = 0; return WBC_OK; }
    CU(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    const bool dev_ptrs = (flags & WBC_DEVICE_PTRS) != 0;
    const wbc::GaitParams G = {g.stance_cycles, g.swing_cycles, g.step_height, g.k_v, g.max_step, g.acc_lin, g.acc_yaw, g.leash};
    wbc::GaitIO io;
    io.k0 = k0; io.cmd = cmd; io.contact = contact; io.terrain = terrain; io.plane_d = plane_d; io.status = status; io.mode = mode;
    io.base_pos = st->base_pos; io.base_rot = st->base_rot; io.base_rpy = st->base_rpy; io.base_vel = st->base_vel; io.q = st->q;
    io.phase = gs->phase; io.tick = gs->tick; io.landed = gs->landed;
    io.com_ref = gs->com_ref; io.v_ref = gs->v_ref; io.liftoff = gs->liftoff; io.target = gs->target; io.offset = gs->offset;
    double* const hout[6] = {init ? nullptr : out->com_des_pos, init ? nullptr : out->com_des_vel, init ? nullptr : out->com_des_acc,
                             init ? nullptr : out->sw_des_pos, init ? nullptr : out->sw_des_vel, init ? nullptr : out->sw_des_acc};
    for (int b = 0; b < 6; b++) io.des[b] = hout[b];
    io.out_ld = init ? ld : out->ld; io.ld = ld;
    // host path: packed staging.  Doubles in d_in: state 30 rows (base_pos 3, base_rot 9, base_rpy 3, base_vel[0:3], q 12) | gait
    // state 27 (com_ref 4, v_ref 3, liftoff 6, target 6, offset 8) | cmd 3 | plane_d 4 | terrain 40; the six outputs in d_out; ints in
    // d_iout: phase, tick, landed | contact 4 (k0 in its first row) | mode | status.  The gait state and the outputs are uploaded too,
    // since a refused robot keeps them as they were.
    static const int KS[5] = {3, 9, 3, 3, 12};
    static const int KG[5] = {4, 3, 6, 6, 8};
    const double* hst[5] = {st->base_pos, st->base_rot, st->base_rpy, st->base_vel, st->q};
    double* hgs[5] = {gs->com_ref, gs->v_ref, gs->liftoff, gs->target, gs->offset};
    int* hint[3] = {gs->phase, gs->tick, gs->landed};
    const size_t N = (size_t)n;
    if (!dev_ptrs) {
        double* h = c->h_pin;
        int* hi = c->h_pin_i;
        double* d = c->d_in;
        size_t off = 0;
        for (int f = 0; f < 5; f++)
            for (int k = 0; k < KS[f]; k++, off++) memcpy(h + off * N, hst[f] + (size_t)k * ld, N * 8);
        for (int f = 0; f < 5; f++)
            for (int k = 0; k < KG[f]; k++, off++) memcpy(h + off * N, hgs[f] + (size_t)k * ld, N * 8);
        if (cmd) for (int k = 0; k < 3; k++) memcpy(h + (57 + k) * N, cmd + (size_t)k * ld, N * 8);
        if (plane_d) for (int k = 0; k < 4; k++) memcpy(h + (60 + k) * N, plane_d + (size_t)k * ld, N * 8);
        if (terrain) for (int k = 0; k < 40; k++) memcpy(h + (64 + k) * N, terrain + (size_t)k * ld, N * 8);
        CU(cudaMemcpyAsync(d, h, (terrain ? 104 : 64) * N * 8, cudaMemcpyHostToDevice, s));
        for (int k = 0; k < 3; k++) memcpy(hi + k * N, hint[k], N * sizeof(int));
        if (k0) memcpy(hi + 3 * N, k0, N * sizeof(int));
        if (contact) for (int k = 0; k < 4; k++) memcpy(hi + (3 + k) * N, contact + (size_t)k * ld, N * sizeof(int));
        if (mode) memcpy(hi + 7 * N, mode, N * sizeof(int));
        CU(cudaMemcpyAsync(c->d_iout, hi, 8 * N * sizeof(int), cudaMemcpyHostToDevice, s));
        if (!init) {
            for (int b = 0; b < 6; b++)
                CU(cudaMemcpy2DAsync(c->d_out + (size_t)b * 6 * N, N * 8, hout[b], (size_t)out->ld * 8, N * 8, 6, cudaMemcpyHostToDevice, s));
            for (int b = 0; b < 6; b++) io.des[b] = c->d_out + (size_t)b * 6 * N;
        }
        io.base_pos = d; io.base_rot = d + 3 * N; io.base_rpy = d + 12 * N; io.base_vel = d + 15 * N; io.q = d + 18 * N;
        io.com_ref = d + 30 * N; io.v_ref = d + 34 * N; io.liftoff = d + 37 * N; io.target = d + 43 * N; io.offset = d + 49 * N;
        io.cmd = cmd ? d + 57 * N : nullptr; io.plane_d = plane_d ? d + 60 * N : nullptr; io.terrain = terrain ? d + 64 * N : nullptr;
        io.phase = c->d_iout; io.tick = c->d_iout + N; io.landed = c->d_iout + 2 * N;
        io.k0 = k0 ? c->d_iout + 3 * N : nullptr; io.contact = contact ? c->d_iout + 3 * N : nullptr;
        io.mode = mode ? c->d_iout + 7 * N : nullptr; io.status = status ? c->d_iout + 8 * N : nullptr;
        io.out_ld = n; io.ld = n;
    }
    const double dt = c->params.obs_dt;
    if (init)
        wbc_gait_init_kernel<<<(n + 127) / 128, 128, 0, s>>>(G, dt, io, n);
    else
        wbc_gait_kernel<<<(n + 127) / 128, 128, 0, s>>>(G, dt, io, n);
    CU(cudaGetLastError());
    c->launches = 1;
    if (!dev_ptrs) {
        CU(cudaMemcpyAsync(c->h_pin + 30 * N, c->d_in + 30 * N, 27 * N * 8, cudaMemcpyDeviceToHost, s));
        if (!init) CU(cudaMemcpyAsync(c->h_pin + 57 * N, c->d_out, 36 * N * 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(c->h_pin_i, c->d_iout, 9 * N * sizeof(int), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        size_t off = 30;
        for (int f = 0; f < 5; f++)
            for (int k = 0; k < KG[f]; k++, off++) memcpy(hgs[f] + (size_t)k * ld, c->h_pin + off * N, N * 8);
        if (!init)
            for (int b = 0; b < 6; b++)
                for (int k = 0; k < 6; k++) memcpy(hout[b] + (size_t)k * out->ld, c->h_pin + (57 + 6 * b + k) * N, N * 8);
        for (int k = 0; k < 3; k++) memcpy(hint[k], c->h_pin_i + k * N, N * sizeof(int));
        if (mode) memcpy(mode, c->h_pin_i + 7 * N, N * sizeof(int));
        if (status) memcpy(status, c->h_pin_i + 8 * N, N * sizeof(int));
    } else if (!(flags & WBC_NO_SYNC)) {
        CU(cudaStreamSynchronize(s));
    }
    return WBC_OK;
}

int wbc_gait_init(wbc_ctx* c, int n, const wbc_gait_params* gp, const wbc_plant_state* st, const int* k0, const double* terrain,
                  const double* plane_d, wbc_gait_state* gs, int* status, long ld, void* cuda_stream, unsigned flags)
{
    return gait_call("wbc_gait_init", true, c, n, gp, gs, st, k0, nullptr, nullptr, terrain, plane_d, nullptr, nullptr, status, ld,
                     cuda_stream, flags);
}

int wbc_gait_step(wbc_ctx* c, int n, const wbc_gait_params* gp, wbc_gait_state* gs, const wbc_plant_state* st, const double* cmd,
                  const int* contact, const double* terrain, const double* plane_d, int* mode, const wbc_traj_samples* out, int* status,
                  long ld, void* cuda_stream, unsigned flags)
{
    return gait_call("wbc_gait_step", false, c, n, gp, gs, st, nullptr, cmd, contact, terrain, plane_d, mode, out, status, ld, cuda_stream,
                     flags);
}

int wbc_last_timing(wbc_ctx* c, float* front_ms, float* solve_ms)
{
    if (!c) return fail(WBC_EINVAL, "null ctx");
    CU(cudaSetDevice(c->device));
    CU(cudaEventSynchronize(c->ev2));
    float a = 0, b = 0;
    CU(cudaEventElapsedTime(&a, c->ev0, c->ev1));
    CU(cudaEventElapsedTime(&b, c->ev1, c->ev2));
    if (front_ms) *front_ms = a;
    if (solve_ms) *solve_ms = b;
    return WBC_OK;
}

int wbc_last_solve_cycles(wbc_ctx* c, int n, unsigned long long* cycles)
{
    if (!c || !cycles || n < 0 || n > c->max_batch) return fail(WBC_EINVAL, "wbc_last_solve_cycles: bad arguments");
    if (n == 0) return WBC_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaDeviceSynchronize());
    unsigned* h = (unsigned*)malloc((size_t)n * sizeof(unsigned));
    if (!h) return fail(WBC_ENOMEM, "out of host memory");
    const cudaError_t e = cudaMemcpy(h, c->cycles_valid ? c->cycles : c->cost, (size_t)n * sizeof(unsigned), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess)
        for (int i = 0; i < n; i++) cycles[i] = (unsigned long long)h[i] << 10;     // stored >> 10
    free(h);
    if (e != cudaSuccess) return fail(WBC_ECUDA, "wbc_last_solve_cycles: %s", cudaGetErrorString(e));
    return WBC_OK;
}
int wbc_last_launches(wbc_ctx* c) { return c ? c->launches : 0; }

int wbc_stage_profile(wbc_ctx* c, unsigned long long* out, int max_rows)
{
    if (!c || !out) return fail(WBC_EINVAL, "wbc_stage_profile: null argument");
    if (!c->prof) return fail(WBC_EINVAL, "wbc_stage_profile: the ctx was created without WBC_STAGE_PROF=1");
    CU(cudaSetDevice(c->device));
    CU(cudaDeviceSynchronize());
    const int rows = max_rows < c->nblocks ? max_rows : c->nblocks;
    CU(cudaMemcpy(out, c->prof, (size_t)rows * 12 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return rows;
}

int wbc_solver_shape(wbc_ctx* c, int* ctas_per_sm, int* smem_bytes, int* grid, int* stage_tasks)
{
    if (!c) return fail(WBC_EINVAL, "null ctx");
    if (ctas_per_sm) *ctas_per_sm = c->last_staged == 2 ? c->exact_per_sm : c->occ_per_sm;
    if (smem_bytes) *smem_bytes = c->last_staged == 2 ? wbcdual::ds::BYTES : c->solve_smem;
    if (grid) *grid = c->last_grid > 0 ? c->last_grid : c->nblocks;
    if (stage_tasks) *stage_tasks = c->last_staged;
    return WBC_OK;
}

int wbc_host_alloc(void** p, size_t bytes)
{
    if (!p || bytes == 0) return fail(WBC_EINVAL, "wbc_host_alloc: bad arguments");
    const cudaError_t e = cudaMallocHost(p, bytes);
    if (e != cudaSuccess) { *p = nullptr; return fail(e == cudaErrorMemoryAllocation ? WBC_ENOMEM : WBC_ECUDA, "wbc_host_alloc: %s", cudaGetErrorString(e)); }
    return WBC_OK;
}
int wbc_host_free(void* p)
{
    if (!p) return WBC_OK;
    const cudaError_t e = cudaFreeHost(p);
    if (e != cudaSuccess) return fail(WBC_ECUDA, "wbc_host_free: %s", cudaGetErrorString(e));
    return WBC_OK;
}

int wbc_debug_update(wbc_ctx* c, int n, const wbc_inputs* in, const wbc_debug* dbg, unsigned flags)
{
    if (!c || !dbg) return fail(WBC_EINVAL, "wbc_debug_update: null argument");
    if (n <= 0 || n > c->max_batch) return fail(WBC_EINVAL, "wbc_debug_update: n outside (0, max_batch]");
    if (flags & WBC_DEVICE_PTRS) return fail(WBC_EINVAL, "wbc_debug_update takes host pointers only");
    int rc = check_inputs(in, n);
    if (rc) return rc;
    if (dbg->ld < n) return fail(WBC_EINVAL, "wbc_debug.ld < n");
    CU(cudaSetDevice(c->device));
    cudaStream_t s = c->stream;
    DevInputs din;
    rc = stage_inputs(c, n, in, s, &din, (flags & WBC_HOST_SLAB) != 0);
    if (rc) return rc;
    static const int K[17] = {324, 18, 18, 216, 12, 3, 3, 36, 144, 18, 18, 216, 12, 12, 12, 12, 6};
    double* host[17] = {dbg->M, dbg->h, dbg->g, dbg->Jac_lin, dbg->Jdqd_lin, dbg->com, dbg->com_vel, dbg->Mcom_b, dbg->Mcom_j, dbg->hcom,
                        dbg->gcom, dbg->Jcom_lin, dbg->Jdqdcom_lin, dbg->foot_pos, dbg->foot_vel, dbg->Fgrf, dbg->Wcom_des};
    size_t tot = 0;
    for (int f = 0; f < 17; f++) tot += K[f];
    double* dbuf = nullptr;
    CU(cudaMalloc(&dbuf, tot * (size_t)n * sizeof(double)));
    DevDebug dd;
    double** dp[17] = {&dd.M, &dd.h, &dd.g, &dd.Jac_lin, &dd.Jdqd_lin, &dd.com, &dd.com_vel, &dd.Mcom_b, &dd.Mcom_j, &dd.hcom, &dd.gcom,
                       &dd.Jcom_lin, &dd.Jdqdcom_lin, &dd.foot_pos, &dd.foot_vel, &dd.Fgrf, &dd.Wcom_des};
    size_t off = 0;
    for (int f = 0; f < 17; f++) { *dp[f] = dbuf + off * n; off += K[f]; }
    dd.ld = n;
    // The observer state must not advance and the ctx's QP records must stay those of the last wbc_cycle (wbc_plant_step
    // reads them): run on a scratch copy of yd/yw and into scratch records.
    double* ytmp = nullptr;
    double* rtmp = nullptr;
    cudaError_t e = cudaMalloc(&ytmp, (size_t)24 * n * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&rtmp, (size_t)n * QPREC_DOUBLES * sizeof(double));
    if (e != cudaSuccess) { cudaFree(dbuf); cudaFree(ytmp); return fail(WBC_ENOMEM, "wbc_debug_update: %s", cudaGetErrorString(e)); }
    e = cudaMemcpy2DAsync(ytmp, (size_t)n * 8, c->yd, (size_t)c->max_batch * 8, (size_t)n * 8, 6, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(ytmp + 6L * n, (size_t)n * 8, c->yw, (size_t)c->max_batch * 8, (size_t)n * 8, 6, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(ytmp + 18L * n, (size_t)n * 8, c->yg, (size_t)c->max_batch * 8, (size_t)n * 8, 6, cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) {
        FrontState st;
        st.yd = ytmp; st.yw = ytmp + 6L * n; st.yg = ytmp + 18L * n; st.ld = n; st.w3 = nullptr; st.w3_ld = 0;
        const int fthreads = front_threads(c, n);
        wbc_front_kernel<<<(n + fthreads - 1) / fthreads, fthreads, 0, s>>>(c->params, din, st, n, rtmp, ytmp + 12L * n, n, dd, 1, DispatchOrder{nullptr, nullptr, nullptr, nullptr, nullptr}, StageReset{nullptr, 0, 0, 0, nullptr, 0, 0});
        e = cudaStreamSynchronize(s);
        if (e == cudaSuccess) e = cudaGetLastError();
    }
    off = 0;
    for (int f = 0; f < 17 && e == cudaSuccess; f++) {
        if (host[f]) e = cudaMemcpy2D(host[f], (size_t)dbg->ld * 8, dbuf + off * n, (size_t)n * 8, (size_t)n * 8, K[f], cudaMemcpyDeviceToHost);
        off += K[f];
    }
    cudaFree(dbuf);
    cudaFree(ytmp);
    cudaFree(rtmp);
    c->launches = 1;
    if (e != cudaSuccess) return fail(WBC_ECUDA, "wbc_debug_update: %s", cudaGetErrorString(e));
    return WBC_OK;
}

int wbc_debug_qp_records(wbc_ctx* c, int n, double* recs, int* doubles_per_record)
{
    if (!c) return fail(WBC_EINVAL, "wbc_debug_qp_records: null ctx");
    if (doubles_per_record) *doubles_per_record = QPREC_DOUBLES;
    if (!recs) return WBC_OK;
    if (n < 0 || n > c->last_n) return fail(WBC_EINVAL, "wbc_debug_qp_records: n exceeds the last wbc_cycle's batch");
    if (n == 0) return WBC_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpy(recs, c->recs, (size_t)n * QPREC_DOUBLES * sizeof(double), cudaMemcpyDeviceToHost));
    return WBC_OK;
}

// wbc_qp_solve, and wbc_qp_solve_warm (active != NULL: the exact solver's warm instantiation, active [n][3] in/out)
static int qp_solve_impl(wbc_ctx* c, int n, const double* Q, const double* cvec, const double* L, int nrows, int neq, double* x, int* status,
                         int* info, double* flops, unsigned* active, void* cuda_stream, unsigned flags)
{
    if (!c || !Q || !cvec || !L || !x) return fail(WBC_EINVAL, "wbc_qp_solve: null argument");
    if (n < 0 || n > c->max_batch) return fail(WBC_EINVAL, "wbc_qp_solve: n outside [0, max_batch]");
    if (nrows < 0 || nrows > 86 || neq < 0 || neq > nrows || nrows - neq > MAXNIC)
        return fail(WBC_EINVAL, "wbc_qp_solve: constraint counts outside the controller's shapes (nrows <= 86)");
    if (n == 0) { c->launches = 0; return WBC_OK; }
    CU(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? (cudaStream_t)cuda_stream : c->stream;
    const bool dev_ptrs = (flags & WBC_DEVICE_PTRS) != 0;
    const size_t nq = (size_t)n * 900, nc = (size_t)n * 30, nl = (size_t)n * nrows * 31, nx = (size_t)n * 30;
    const double *dQ = Q, *dc = cvec, *dL = L;
    double* dx = x;
    int *dstatus = status, *dinfo = info;
    double* dflops = flops;
    unsigned* dactive = active;
    if (!dev_ptrs) {
        const size_t need = (nq + nc + nl + nx + n) * sizeof(double) + (size_t)n * (active ? 12 : 9) * sizeof(int);
        if (need > c->dense_cap) {
            CU(cudaStreamSynchronize(s));
            cudaFree(c->d_dense);
            c->d_dense = nullptr; c->dense_cap = 0;
            CU(cudaMalloc(&c->d_dense, need));
            c->dense_cap = need;
        }
        double* p = c->d_dense;
        CU(cudaMemcpyAsync(p, Q, nq * 8, cudaMemcpyHostToDevice, s)); dQ = p; p += nq;
        CU(cudaMemcpyAsync(p, cvec, nc * 8, cudaMemcpyHostToDevice, s)); dc = p; p += nc;
        if (nl) CU(cudaMemcpyAsync(p, L, nl * 8, cudaMemcpyHostToDevice, s));
        dL = p; p += nl;
        dx = p; p += nx;
        dflops = flops ? p : nullptr; p += n;
        int* ip = reinterpret_cast<int*>(p);
        dstatus = status ? ip : nullptr;
        dinfo = info ? ip + n : nullptr;
        if (active) {
            dactive = reinterpret_cast<unsigned*>(ip + 9L * n);
            CU(cudaMemcpyAsync(dactive, active, (size_t)n * 3 * sizeof(unsigned), cudaMemcpyHostToDevice, s));
        }
    }
    CU(cudaMemsetAsync(c->queue + ORD_NB, 0, sizeof(int), s));
    const bool exact = active || (flags & WBC_QP_EXACT) != 0;
    const int nblocks = exact ? (n < c->exact_blocks ? n : c->exact_blocks) : (n < c->nblocks ? n : c->nblocks);
    CU(cudaEventRecord(c->ev0, s));
    CU(cudaEventRecord(c->ev1, s));
    if (active)
        wbc_dense_qp_exact_kernel<true><<<nblocks, EXACT_T, wbcdual::ds::BYTES, s>>>(n, dQ, dc, dL, nrows, neq, dx, dstatus, dinfo, dflops, c->scratch,
                                                                                      c->queue + ORD_NB, dactive);
    else if (exact)
        wbc_dense_qp_exact_kernel<<<nblocks, EXACT_T, wbcdual::ds::BYTES, s>>>(n, dQ, dc, dL, nrows, neq, dx, dstatus, dinfo, dflops, c->scratch,
                                                                                c->queue + ORD_NB);
    else
        wbc_dense_qp_kernel<<<nblocks, c->threads, c->solve_smem, s>>>(c->params, n, dQ, dc, dL, nrows, neq, dx, dstatus, dinfo, dflops, c->scratch, c->kkt, c->queue + ORD_NB);
    CU(cudaEventRecord(c->ev2, s));
    CU(cudaGetLastError());
    c->launches = 1;
    if (!dev_ptrs) {
        CU(cudaMemcpyAsync(x, dx, nx * 8, cudaMemcpyDeviceToHost, s));
        if (flops) CU(cudaMemcpyAsync(flops, dflops, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
        if (status) CU(cudaMemcpyAsync(status, dstatus, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        if (info) CU(cudaMemcpyAsync(info, dinfo, (size_t)n * 8 * 4, cudaMemcpyDeviceToHost, s));
        if (active) CU(cudaMemcpyAsync(active, dactive, (size_t)n * 3 * sizeof(unsigned), cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
    } else if (!(flags & WBC_NO_SYNC)) {
        CU(cudaStreamSynchronize(s));
    }
    return WBC_OK;
}

int wbc_qp_solve(wbc_ctx* c, int n, const double* Q, const double* cvec, const double* L, int nrows, int neq, double* x, int* status,
                 int* info, double* flops, void* cuda_stream, unsigned flags)
{
    return qp_solve_impl(c, n, Q, cvec, L, nrows, neq, x, status, info, flops, nullptr, cuda_stream, flags);
}

int wbc_qp_solve_warm(wbc_ctx* c, int n, const double* Q, const double* cvec, const double* L, int nrows, int neq, double* x, int* status,
                      int* info, double* flops, unsigned* active, void* cuda_stream, unsigned flags)
{
    if (!active) return fail(WBC_EINVAL, "wbc_qp_solve_warm: null argument");
    return qp_solve_impl(c, n, Q, cvec, L, nrows, neq, x, status, info, flops, active, cuda_stream, flags);
}

int wbc_set_active_set(wbc_ctx* c, int n, const unsigned* sets, long ld)
{
    if (!c || !sets || n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "wbc_set_active_set: bad arguments");
    if (n == 0) return WBC_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpy2D(c->aset, (size_t)c->max_batch * 4, sets, (size_t)ld * 4, (size_t)n * 4, 4, cudaMemcpyHostToDevice));
    return WBC_OK;
}

int wbc_get_active_set(wbc_ctx* c, int n, unsigned* sets, long ld)
{
    if (!c || !sets || n < 0 || n > c->max_batch || ld < n) return fail(WBC_EINVAL, "wbc_get_active_set: bad arguments");
    if (n == 0) return WBC_OK;
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemcpy2D(sets, (size_t)ld * 4, c->aset, (size_t)c->max_batch * 4, (size_t)n * 4, 4, cudaMemcpyDeviceToHost));
    return WBC_OK;
}

int wbc_measure_dfma_peak(wbc_ctx* c, double* flops_per_s)
{
    if (!c || !flops_per_s) return fail(WBC_EINVAL, "null argument");
    CU(cudaSetDevice(c->device));
    const int blocks = c->sm_count * 8, threads = 256, iters = 2048;
    double* d = nullptr;
    CU(cudaMalloc(&d, (size_t)blocks * threads * sizeof(double)));
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(c->ev0, c->stream);
        wbc_dfma_peak_kernel<<<blocks, threads, 0, c->stream>>>(d, iters);
        cudaEventRecord(c->ev1, c->stream);
        cudaError_t e = cudaEventSynchronize(c->ev1);
        if (e != cudaSuccess) { cudaFree(d); return fail(WBC_ECUDA, "dfma peak: %s", cudaGetErrorString(e)); }
        float ms = 0;
        cudaEventElapsedTime(&ms, c->ev0, c->ev1);
        if (rep > 0 && ms < best) best = ms;
    }
    cudaFree(d);
    const double fl = 2.0 * 8 * 16 * (double)iters * blocks * threads;
    *flops_per_s = fl / (best * 1e-3);
    return WBC_OK;
}

}  // extern "C"
