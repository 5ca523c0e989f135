// wbc_dogctrl.hpp -- header-only C++ host layer above the C ABI (wbc_b200.h).
//
// It mirrors, name for name, the two interfaces the reference's control thread talks to on the hot path, so that
// ctrl_loop() (dogbot_controller/src/client/main.cpp:836-1955) can call the B200 path without being rewritten:
//
//   reference                                              here
//   -----------------------------------------------------  -----------------------------------------------------------
//   class OPT                      lopt.h:5-36             wbc_b200::OPT        setQ/setc/setL_stance/setL_swing/
//     OPT(30,86,82) main.cpp:266                                                opt_stance/opt_swing (one dense QP)
//   DOGCTRL::update(H, q, dq, v, g) main.cpp:63, 572-660   wbc_b200::DogCtrl::update(...)   same five arguments
//   DOGCTRL::estimate()            main.cpp:692-725        folded into DogCtrl::cycle_stance()/cycle_swing()
//   stance / swing cycle bodies    main.cpp:984-1127,      DogCtrl::cycle_stance(), DogCtrl::cycle_swing(first_half)
//                                  1163-1397
//   (no batched form exists)                               wbc_b200::Batch      SoA host buffers for n instances
//
// No Eigen is needed (none is installed here): every matrix/vector argument is a template parameter that only has
// to offer `operator()(i, j)` / `operator()(i)` (Eigen::Matrix4d, Eigen::Matrix<double,12,1>, Eigen::VectorXd,
// Eigen::MatrixXd all do), or a plain `const double*`.  Errors are reported as wbc_b200::Error (the reference swallows
// solver failures, lopt.cpp:114-116, and leaves x_ untouched; `OPT::opt_*` keeps that behaviour when
// `swallow_failures` is set, and throws otherwise).  There is no CPU fallback: constructing any of these classes on
// a machine without an sm_100 GPU throws with WBC_ENODEV.
#ifndef WBC_DOGCTRL_HPP
#define WBC_DOGCTRL_HPP

#include <cstddef>
#include <stdexcept>
#include <string>
#include <vector>

#include "wbc_b200.h"

namespace wbc_b200 {

class Error : public std::runtime_error {
public:
    Error(int code, const std::string& what) : std::runtime_error(what), code_(code) {}
    int code() const { return code_; }

private:
    int code_;
};

inline void check(int rc, const char* what)
{
    if (rc != WBC_OK) throw Error(rc, std::string(what) + ": " + wbc_last_error());
}

// RAII owner of one wbc_ctx (one GPU).  Not copyable.
class Context {
public:
    explicit Context(int max_batch, int device = 0, const wbc_params* params = nullptr) : ctx_(nullptr)
    {
        check(wbc_create(&ctx_, device, max_batch, params), "wbc_create");
    }
    ~Context() { wbc_destroy(ctx_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;
    wbc_ctx* get() const { return ctx_; }

private:
    wbc_ctx* ctx_;
};

// ---------------------------------------------------------------------------------------------------------------
// OPT: the reference's solver operator (lopt.h:5-36).  Row-major dense copies are taken in the setters exactly as
// the reference copies Eigen -> alglib arrays element by element (lopt.cpp:22-66).
class OPT {
public:
    OPT(int control_variables, int stance_constraint, int swing_constraint, int device = 0)
        : swallow_failures(false), last_status(0), ctx_(1, device), Q_(900, 0.0), c_(30, 0.0), Ls_(86 * 31, 0.0), Lw_(82 * 31, 0.0)
    {
        for (int i = 0; i < 8; i++) last_info[i] = 0;
        if (control_variables != 30 || stance_constraint != 86 || swing_constraint != 82)
            throw Error(WBC_EINVAL, "OPT is specialised to the controller's shapes OPT(30, 86, 82) (main.cpp:266)");
    }
    template <class Mat> void setQ(const Mat& Q)
    {
        for (int i = 0; i < 30; i++)
            for (int j = 0; j < 30; j++) Q_[i * 30 + j] = Q(i, j);
    }
    template <class Vec> void setc(const Vec& c)
    {
        for (int i = 0; i < 30; i++) c_[i] = c(i);
    }
    template <class Mat> void setL_stance(const Mat& L)
    {
        for (int i = 0; i < 86; i++)
            for (int j = 0; j < 31; j++) Ls_[i * 31 + j] = L(i, j);
    }
    template <class Mat> void setL_swing(const Mat& L)
    {
        for (int i = 0; i < 82; i++)
            for (int j = 0; j < 31; j++) Lw_[i * 31 + j] = L(i, j);
    }
    // first 18 rows "=" (lopt.cpp:40-47); x_ must hold 30 entries (main.cpp:1122-1123)
    template <class Vec> void opt_stance(Vec& x_) { solve(Ls_.data(), 86, 18, x_, active_stance_); }
    // first 12 rows "=" (lopt.cpp:57-64)
    template <class Vec> void opt_swing(Vec& x_) { solve(Lw_.data(), 82, 12, x_, active_swing_); }

    bool swallow_failures;   // true: behave like lopt.cpp:114-116 (x_ untouched, nothing reported)
    bool exact_qp = false;   // true: solve to the exact optimum (WBC_QP_EXACT, dual active-set) instead of DENSE-AUL at the
                             // reference's settings; last_info then holds the exact-mode counters (wbc_b200.h)
    bool warm_start = false; // with exact_qp: opt_stance and opt_swing each start from the active set of their own previous solve
                             // (wbc_qp_solve_warm) -- for a control loop that solves almost the same QP every cycle
    int last_status;         // 0 ok, <0 solver failure of the last opt_* call
    int last_info[8];        // ncholesky, outer its, QQP calls, working set, max KKT dim, flags, 0, 0

private:
    template <class Vec> void solve(const double* L, int nrows, int neq, Vec& x_, unsigned* active)
    {
        double x[30];
        for (int i = 0; i < 30; i++) x[i] = x_(i);
        if (warm_start && !exact_qp) throw Error(WBC_EINVAL, "OPT: warm_start needs exact_qp");
        if (warm_start)
            check(wbc_qp_solve_warm(ctx_.get(), 1, Q_.data(), c_.data(), L, nrows, neq, x, &last_status, last_info, nullptr, active, nullptr,
                                    WBC_HOST_PTRS),
                  "wbc_qp_solve_warm");
        else
            check(wbc_qp_solve(ctx_.get(), 1, Q_.data(), c_.data(), L, nrows, neq, x, &last_status, last_info, nullptr, nullptr,
                               WBC_HOST_PTRS | (exact_qp ? WBC_QP_EXACT : 0u)),
                  "wbc_qp_solve");
        if (last_status != 0) {
            if (swallow_failures) return;
            throw Error(last_status, exact_qp ? "OPT: the exact QP solver reported failure" : "OPT: the DENSE-AUL solver reported failure");
        }
        for (int i = 0; i < 30; i++) x_(i) = x[i];
    }
    Context ctx_;
    std::vector<double> Q_, c_, Ls_, Lw_;
    unsigned active_stance_[3] = {0u, 0u, 0u}, active_swing_[3] = {0u, 0u, 0u};   // warm_start: the last final active sets
};

// ---------------------------------------------------------------------------------------------------------------
// Batch: n instances in host SoA buffers (component-major, leading dimension n), one wbc_cycle per call.
class Batch {
public:
    explicit Batch(int n, int device = 0, const wbc_params* params = nullptr)
        : n_(n), ctx_(n > 0 ? n : 1, device, params), base_pos(3 * n), base_rot(9 * n), base_rpy(3 * n), base_vel(6 * n), q(12 * n), dq(12 * n),
          com_des_pos(6 * n), com_des_vel(6 * n), com_des_acc(6 * n), sw_des_pos(6 * n), sw_des_vel(6 * n), sw_des_acc(6 * n),
          foot_force(12 * n), terrain(), mode(n, WBC_MODE_STANCE), tau(12 * n), w(6 * n), x(30 * n), qp_obj(n), status(n), w3(12 * n)
    {
    }
    int size() const { return n_; }
    wbc_ctx* ctx() const { return ctx_.get(); }
    // element k of instance i of an SoA array
    double& at(std::vector<double>& a, int k, int i) { return a[(size_t)k * n_ + i]; }
    void enable_terrain() { terrain.assign((size_t)40 * n_, 0.0); }
    void set_observer_state(const double* yd, const double* yw) { check(wbc_set_observer_state(ctx_.get(), n_, yd, yw, n_), "wbc_set_observer_state"); }
    void get_observer_state(double* yd, double* yw) { check(wbc_get_observer_state(ctx_.get(), n_, yd, yw, n_), "wbc_get_observer_state"); }
    // ygamma, the second-order observer's extra integrator (wbc_params::obs_order == 2; main.cpp:243, estimator_sem.cpp:20)
    void set_observer_state2(const double* yg) { check(wbc_set_observer_state2(ctx_.get(), n_, yg, n_), "wbc_set_observer_state2"); }
    void get_observer_state2(double* yg) { check(wbc_get_observer_state2(ctx_.get(), n_, yg, n_), "wbc_get_observer_state2"); }
    bool want_w3 = false;   // also compute ESTIMATOR_SEM::getw3 (estimator_sem.cpp:64-70) into w3
    bool exact_qp = false;  // solve each QP to its exact optimum (WBC_QP_EXACT) instead of DENSE-AUL at the reference's settings
    bool warm_qp = false;   // with exact_qp: start each instance from its previous exact-mode active set (WBC_QP_WARM)
    // Planner hand-over (once per plan): the node tables of the four towr splines of every instance, see wbc_trajectory.
    // durations [4*nseg][n], nodes [4*(nseg+1)*6][n].  Replaces keeping `SplineHolder solution` on the host (main.cpp:900-960).
    void set_trajectory(int nseg, const double* durations, const double* nodes)
    {
        wbc_trajectory tr;
        tr.nseg = nseg; tr.durations = durations; tr.nodes = nodes; tr.ld = n_;
        check(wbc_set_trajectory(ctx_.get(), n_, &tr, nullptr, WBC_HOST_PTRS), "wbc_set_trajectory");
    }
    // solution.base_linear_->GetPoint(t) ... ee_motion_.at(k)->GetPoint(t) of every instance, evaluated on the GPU
    // (main.cpp:1004-1010, 1333-1368); the samples stay on the device for cycle(true).
    void sample_trajectory(double t) { check(wbc_sample_trajectory(ctx_.get(), n_, nullptr, t, nullptr, nullptr, WBC_HOST_PTRS), "wbc_sample_trajectory"); }
    // One control cycle for all n instances: host buffers in, host buffers out (H2D + 2 kernels + D2H).
    // sampled_trajectory: take com_des_* / sw_des_* from the last sample_trajectory() instead of the host vectors.
    void cycle(bool sampled_trajectory = false)
    {
        wbc_inputs in;
        in.base_pos = base_pos.data(); in.base_rot = base_rot.data(); in.base_rpy = base_rpy.data(); in.base_vel = base_vel.data();
        in.q = q.data(); in.dq = dq.data(); in.com_des_pos = com_des_pos.data(); in.com_des_vel = com_des_vel.data();
        in.com_des_acc = com_des_acc.data(); in.sw_des_pos = sw_des_pos.data(); in.sw_des_vel = sw_des_vel.data();
        in.sw_des_acc = sw_des_acc.data(); in.foot_force = foot_force.data(); in.terrain = terrain.empty() ? nullptr : terrain.data();
        in.mode = mode.data(); in.ld = n_; in.obs_gain = nullptr;
        wbc_outputs out;
        out.tau = tau.data(); out.w = w.data(); out.x = x.data(); out.qp_obj = qp_obj.data(); out.status = status.data();
        out.qp_info = nullptr; out.qp_flops = nullptr; out.ld = n_; out.w3 = want_w3 ? w3.data() : nullptr;
        check(wbc_cycle(ctx_.get(), n_, &in, &out, nullptr, WBC_HOST_PTRS | (sampled_trajectory ? WBC_SAMPLED_TRAJ : 0u) | (exact_qp ? WBC_QP_EXACT : 0u) |
                                                     (warm_qp ? WBC_QP_WARM : 0u)),
              "wbc_cycle");
    }

private:
    int n_;
    Context ctx_;

public:
    std::vector<double> base_pos, base_rot, base_rpy, base_vel, q, dq, com_des_pos, com_des_vel, com_des_acc, sw_des_pos, sw_des_vel, sw_des_acc,
        foot_force, terrain;
    std::vector<int> mode;
    std::vector<double> tau, w, x, qp_obj;
    std::vector<int> status;
    std::vector<double> w3;   // [12][n] when want_w3
};

// ---------------------------------------------------------------------------------------------------------------
// DogCtrl: the N = 1 drop-in for the members of DOGCTRL that the control thread uses each cycle.
//
//   dc.update(_world_H_base, _jnt_pos, _jnt_vel, _base_vel, gravity);      // main.cpp:980 -- same call
//   dc.set_base_rpy(_base_pos[3], _base_pos[4], _base_pos[5]);            // the member update() reads at main.cpp:596
//   dc.set_com_desired(CoMPosD, CoMVelD, CoMAccD);                         // main.cpp:1005-1010
//   dc.set_foot_forces(force_br, force_bl, force_fl, force_fr);            // main.cpp:1022-1026 (sensor frames)
//   dc.cycle_stance();                                                     // main.cpp:984-1127 incl. estimate() at :1029
//   publish_cmd(dc.tau()); ... dc.w()                                      // main.cpp:1127, 1129-1144
//
// Joint order of jointPos/jointVel/tau() is the controller's DoF order (roll BL,BR,FL,FR, then pitch,knee of BL,BR,FL,FR,
// main.cpp:612-613); gravity is accepted for signature compatibility and forwarded to the ctx parameters.
class DogCtrl {
public:
    explicit DogCtrl(int device = 0) : b_(1, device)
    {
        wbc_default_params(&p_);
    }
    wbc_params& params() { return p_; }
    void apply_params() { check(wbc_set_params(b_.ctx(), &p_), "wbc_set_params"); }

    template <class M4, class V12a, class V12b, class V6, class V3>
    void update(const M4& eigenWorld_H_base, const V12a& eigenJointPos, const V12b& eigenJointVel, const V6& eigenBasevel, const V3& eigenGravity)
    {
        for (int i = 0; i < 3; i++) {
            b_.base_pos[i] = eigenWorld_H_base(i, 3);
            for (int j = 0; j < 3; j++) b_.base_rot[3 * i + j] = eigenWorld_H_base(i, j);
        }
        for (int i = 0; i < 12; i++) { b_.q[i] = eigenJointPos(i); b_.dq[i] = eigenJointVel(i); }
        for (int i = 0; i < 6; i++) b_.base_vel[i] = eigenBasevel(i);
        bool changed = false;
        for (int i = 0; i < 3; i++) {
            if (p_.gravity[i] != eigenGravity(i)) changed = true;
            p_.gravity[i] = eigenGravity(i);
        }
        if (changed) apply_params();
    }
    void set_base_rpy(double roll, double pitch, double yaw) { b_.base_rpy[0] = roll; b_.base_rpy[1] = pitch; b_.base_rpy[2] = yaw; }
    template <class V6a, class V6b, class V6c> void set_com_desired(const V6a& pos, const V6b& vel, const V6c& acc)
    {
        for (int i = 0; i < 6; i++) { b_.com_des_pos[i] = pos(i); b_.com_des_vel[i] = vel(i); b_.com_des_acc[i] = acc(i); }
    }
    // stacked order BR, BL, FL, FR (main.cpp:1022-1026)
    template <class V3> void set_foot_forces(const V3& f_br, const V3& f_bl, const V3& f_fl, const V3& f_fr)
    {
        for (int i = 0; i < 3; i++) { b_.foot_force[i] = f_br(i); b_.foot_force[3 + i] = f_bl(i); b_.foot_force[6 + i] = f_fl(i); b_.foot_force[9 + i] = f_fr(i); }
    }
    // the two swing feet in Jsw row order (first half-cycle BR then FL, main.cpp:1164-1167; second BL then FR, 1711-1714)
    template <class V6a, class V6b, class V6c> void set_swing_desired(const V6a& pos, const V6b& vel, const V6c& acc)
    {
        for (int i = 0; i < 6; i++) { b_.sw_des_pos[i] = pos(i); b_.sw_des_vel[i] = vel(i); b_.sw_des_acc[i] = acc(i); }
    }
    // Planner hand-over (after get_trajectory(), main.cpp:900-960): the four solution splines of this robot -- base_linear_,
    // base_angular_, ee_motion_ of the two swing feet -- as `nseg` cubic-Hermite polynomials each.  durations [4][nseg],
    // nodes [4][nseg+1][6] (position 3, velocity 3).  Then sample_trajectory(t) + cycle_*(true) replace set_com_desired /
    // set_swing_desired: solution.*->GetPoint(t) is evaluated on the GPU (main.cpp:1004-1010, 1333-1368).
    void set_trajectory(int nseg, const double* durations, const double* nodes) { b_.set_trajectory(nseg, durations, nodes); }
    void sample_trajectory(double t) { b_.sample_trajectory(t); }
    void cycle_stance(bool sampled_trajectory = false)
    {
        b_.mode[0] = WBC_MODE_STANCE;
        b_.exact_qp = exact_qp;
        b_.warm_qp = warm_qp;
        b_.cycle(sampled_trajectory);
    }
    void cycle_swing(bool first_half, bool sampled_trajectory = false)
    {
        b_.mode[0] = first_half ? WBC_MODE_SWING_BR_FL : WBC_MODE_SWING_BL_FR;
        b_.exact_qp = exact_qp;
        b_.warm_qp = warm_qp;
        b_.cycle(sampled_trajectory);
    }

    const double* tau() const { return b_.tau.data(); }     // [12]  main.cpp:1126, 1396
    const double* w() const { return b_.w.data(); }         // [6]   main.cpp:718; ESTIMATOR_SEM::getwext (estimator_sem.cpp:98-104)
    // ESTIMATOR_SEM::getw3 (estimator_sem.cpp:64-70): the estimate as foot forces, stacked BR, BL, FL, FR; set batch().want_w3 first
    const double* getw3() const { return b_.w3.data(); }    // [12]
    const double* x() const { return b_.x.data(); }         // [30]  QP solution
    double qp_objective() const { return b_.qp_obj[0]; }
    int status() const { return b_.status[0]; }
    Batch& batch() { return b_; }
    bool exact_qp = false;  // cycles solve each QP to its exact optimum (WBC_QP_EXACT) instead of DENSE-AUL
    bool warm_qp = false;   // with exact_qp: warm-start each cycle's QP from the previous exact-mode cycle's active set (WBC_QP_WARM)

private:
    Batch b_;
    wbc_params p_;
};

}  // namespace wbc_b200
#endif
