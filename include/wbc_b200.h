/* wbc_b200.h -- C ABI of the B200-native batched whole-body-control cycle.
 *
 * Drop-in boundary for the per-control-cycle hot path of prisma-lab/WBC-quadruped-DOB's
 * dogbot_controller (reference paths are relative to /root/reference/dogbot_controller/src):
 *
 *   reference interface                                   replaced by
 *   ----------------------------------------------------  ---------------------------------------
 *   DOGCTRL::update(world_H_base, jointPos, jointVel,     wbc_cycle()  (state in: wbc_inputs)
 *       baseVel, gravity)            client/main.cpp:63, 572-660
 *   DOGCTRL::estimate()              client/main.cpp:692-725     wbc_cycle()  (w out; yd/yw state kept in the ctx,
 *                                                                wbc_get/set_observer_state)
 *   stance / swing QP assembly + tau client/main.cpp:984-1127,   wbc_cycle()  (tau out)
 *                                    1163-1397
 *   OPT::OPT(30,86,82), setQ, setc,  lopt.h:5-36,                wbc_qp_solve()  (dense Q, c, L in; x out)
 *   setL_stance/_swing, opt_stance/  lopt.cpp:4-154
 *   opt_swing
 *
 * Conventions
 *   - plain C, no exceptions; every entry point returns 0 on success or a negative WBC_E* code, and
 *     wbc_last_error() returns a message for the calling thread's last failure;
 *   - all batched arrays are SoA "component-major": element k of instance i is at ptr[k*ld + i];
 *   - DoF order (12): roll BL, BR, FL, FR, then (pitch, knee) of BL, BR, FL, FR -- the order of the
 *     controller's qmin/qmax tables (main.cpp:612-613); torques use the same order;
 *   - stacked foot order (forces, terrain, contact Jacobian rows): BR, BL, FL, FR (main.cpp:674-686);
 *   - a ctx is bound to one GPU; calls on one ctx must be serialised by the caller, different ctxs
 *     are independent (one ctx per GPU / per rank);
 *   - there is no CPU fallback: every call fails with WBC_ENODEV when no sm_100 device is usable.
 */
#ifndef WBC_B200_H
#define WBC_B200_H

#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

#define WBC_OK 0
#define WBC_EINVAL (-1)     /* bad argument */
#define WBC_ENODEV (-2)     /* no usable CUDA device */
#define WBC_ECUDA (-3)      /* CUDA runtime error (see wbc_last_error) */
#define WBC_ENOMEM (-4)
/* per-instance status words (wbc_outputs.status) for inputs the cycle refuses to process */
#define WBC_ST_BAD_MODE (-20)    /* contact mode outside {0, 1, 2} */
#define WBC_ST_NONFINITE (-21)   /* a NaN or infinity among the inputs, or produced from them before the QP */
#define WBC_ST_INFEASIBLE (-22)  /* exact mode (WBC_QP_EXACT): the constraints admit no point (row-scaled residuals) */
#define WBC_ST_NOT_PD (-23)      /* exact mode: H (the lower triangle of Q mirrored) is not positive definite */
#define WBC_ST_BAD_TERRAIN (-24) /* wbc_plant_contact_step_terrain: a foot frame not orthonormal to 1e-9, or mu < 0 */

/* contact modes: which feet swing */
#define WBC_MODE_STANCE 0        /* main.cpp:979-1148, 1516-1675 */
#define WBC_MODE_SWING_BR_FL 1   /* main.cpp:1155-1424 */
#define WBC_MODE_SWING_BL_FR 2   /* main.cpp:1703-1949 */

/* wbc_cycle / wbc_qp_solve flags */
#define WBC_HOST_PTRS 0u         /* in/out pointers are host memory: H2D + D2H copies are part of the call */
#define WBC_DEVICE_PTRS 1u       /* in/out pointers are device memory on the ctx's GPU: launch only */
#define WBC_NO_SYNC 2u           /* (device pointers only) return after enqueueing on the stream */
#define WBC_FIFO_DISPATCH 4u     /* wbc_cycle: hand instances to the solver warps in index order.  Default: longest solve first,
                                    predicted from each instance's previous cycle on this ctx with the same n (the ctx keeps a
                                    per-instance cost: the solve's duration, or its flop count where small batches run with
                                    express lanes, DESIGN.md 4.2); the order never changes a result, only when the batch's tail ends. */
#define WBC_SAMPLED_TRAJ 16u     /* wbc_cycle: com_des_* and sw_des_* come from the last wbc_sample_trajectory(out = NULL) on this ctx;
                                  * those six wbc_inputs pointers are ignored (may be NULL) and are not copied from the host */
#define WBC_QP_EXACT 32u         /* wbc_cycle / wbc_qp_solve: solve each QP to its exact optimum with a Goldfarb-Idnani dual active-set
                                  * solver (one warp per QP, wbc_solve_exact_kernel) instead of the DENSE-AUL restatement at the
                                  * reference's settings; qp_epsx, qp_rho, qp_outerits and qp_literal_kkt are ignored.  Status 0 means
                                  * every row is satisfied to 1e-12 row-scaled and every active inequality multiplier is >= 0;
                                  * WBC_ST_INFEASIBLE, WBC_ST_NOT_PD, or -100 (iteration cap 2 nrows + 30) otherwise, with x = 0.
                                  * qp_info in this mode: [0] factorisations (1), [1] rows added to the active set (equalities
                                  * included), [2] rows dropped, [3] active inequality rows, [4] active-set size, [5] flags: 256 always
                                  * (exact mode), | 512 a dependent consistent equality was skipped, | 1024 a violated row depended on
                                  * the active set and dual steps were taken, | 4096 a violated row depended on the active set, was
                                  * implied by it and violated only by rounding, and was held out; [6], [7] 0.  qp_flops: the exact
                                  * solver's own count. */
#define WBC_QP_WARM 64u          /* wbc_cycle, only together with WBC_QP_EXACT (else WBC_EINVAL, nothing done): warm-start each instance
                                  * from the active set the ctx stored for its index (wbc_get_active_set) when that set was solved in
                                  * the instance's current contact mode; any other instance starts cold.  Every exact-mode cycle, warm
                                  * or cold, stores each instance's final active inequality rows (none when it failed or was refused).
                                  * x is the same unique optimum as in cold exact mode, to the solver's precision but not bit for bit:
                                  * it depends on the ctx's history.  qp_info in this mode: [1], [2] include the warm-start phase's
                                  * additions and drops, [6] warm rows added before the GI loop, [7] warm rows dropped before it (a
                                  * negative multiplier), [5] | 2048 when the instance was warm-started. */
#define WBC_HOST_SLAB 8u         /* (host pointers) the input arrays are carved, in wbc_inputs field order, from ONE page-locked
                                  * allocation with ld == n: adjacent fields are moved with a single copy */

typedef struct wbc_ctx wbc_ctx;

/* Gains, limits and solver settings; wbc_default_params() fills the reference's literals. */
typedef struct wbc_params {
    double kcom, dcom;        /* 2500, 50          main.cpp:1019-1020 */
    double q1_weight;         /* 50                main.cpp:997       */
    double slack_weight;      /* 1e8               main.cpp:1187      */
    double mu;                /* 0.6               main.cpp:1062      */
    double tau_max;           /* 60                main.cpp:1090-1091 */
    double joint_dt;          /* 0.025             main.cpp:1098      */
    double kp_sw, kd_sw;      /* 300, 20           main.cpp:1371-1373 */
    double g_acc;             /* 9.81              main.cpp:702, 1016 */
    double obs_gain;          /* 10                main.cpp:708       */
    double obs_dt;            /* 0.0025            main.cpp:715       */
    double gravity[3];        /* (0,0,-9.8)        main.cpp:855       */
    double qp_epsx, qp_rho;   /* 1e-2, 1e4         lopt.cpp:101, 138  */
    double obs_gain2;         /* 1                 second entry of the coefficient vector {10, 1} (main.cpp:707-708,
                                                   estimator_sem.cpp:47-48); only read when obs_order == 2 */
    int qp_outerits;          /* 5                 lopt.cpp:101, 138  */
    int observer_enabled;     /* 1: call estimate() at main.cpp:1029/1220/1569/1767 (reference ships 0) */
    int fix_swing_rhs;        /* 0: keep the reference's zero swing-equality rhs (main.cpp:1238-1241) */
    int qp_literal_kkt;       /* 0 (default): reduced multiplier update with the literal form as fallback; 1: always the literal stacked-KKT QR (opt.cpp:41803-42032) */
    int hold_tau_on_failure;  /* 0 (default): a failed instance gets tau from x = 0 (tau = 0 when its inputs are invalid);
                                 1: it gets the last good tau this ctx produced for that instance index -- the reference
                                 keeps publishing its `tau` member when the QP throws (lopt.cpp:114-116, main.cpp:242, 1126) */
    int obs_order;            /* 1 (default): the first-order observer DOGCTRL::estimate() runs (main.cpp:692-725).
                                 2: second-order recursion (SURVEY.md 8f-3) through the `ygamma` state both the controller and the
                                 dead ESTIMATOR_SEM carry but never advance (main.cpp:243, 724; estimator_sem.cpp:17-20):
                                     gamma1 = k1 (rho - yw - yd),  ygamma' = gamma1 - w,  w = k2 ygamma,
                                 k1 = obs_gain (or the per-instance gain), k2 = obs_gain2, i.e. w = k1 k2 / (s^2 + k2 s + k1 k2) w_true. */
    int obs_form;             /* 0 (default): backward-Euler gain of main.cpp:716-718, w = (I + k T)^-1 k (rho - yw_prev - yd);
                                 1: the explicit gain of ESTIMATOR_SEM::estimate, w = k (rho - yw_prev - yd) (estimator_sem.cpp:55-57,
                                 which also uses T = 0.001: set obs_dt). */
} wbc_params;

/* One control cycle's inputs for n instances (what update() receives plus the members it reads). */
typedef struct wbc_inputs {
    const double* base_pos;     /* [3]  base position, world                          main.cpp:440-446 */
    const double* base_rot;     /* [9]  world_R_base row-major (_world_H_base block)  main.cpp:447-451 */
    const double* base_rpy;     /* [3]  roll pitch yaw (_base_pos[3:6])               main.cpp:596     */
    const double* base_vel;     /* [6]  linear, angular velocity, world (MIXED)       main.cpp:453     */
    const double* q;            /* [12] joint positions                               main.cpp:388-433 */
    const double* dq;           /* [12] joint velocities                                               */
    const double* com_des_pos;  /* [6]  desired CoM pose sample                       main.cpp:1005-1010 */
    const double* com_des_vel;  /* [6]                                                                  */
    const double* com_des_acc;  /* [6]                                                                  */
    const double* sw_des_pos;   /* [6]  two swing feet, Jsw row order                 main.cpp:1333-1368 */
    const double* sw_des_vel;   /* [6]                                                                  */
    const double* sw_des_acc;   /* [6]                                                                  */
    const double* foot_force;   /* [12] contact-sensor forces, foot frames            main.cpp:794-834 */
    const double* terrain;      /* [40] per foot n(3) t1(3) t2(3) mu(1); NULL = flat  main.cpp:1062-1078 */
    const int* mode;            /* [1]  WBC_MODE_*                                                      */
    long ld;                    /* leading dimension (>= n) of every array above                       */
    const double* obs_gain;     /* [1]  per-instance observer gain k0 (main.cpp:708); NULL = params.obs_gain.
                                        Extension for BASELINE config 5's gain sweep (the reference hard-codes 10). */
} wbc_inputs;

typedef struct wbc_outputs {
    double* tau;        /* [12] joint torques                               main.cpp:1126, 1396 */
    double* w;          /* [6]  estimated disturbance wrench w[0]           main.cpp:718        */
    double* x;          /* [30] QP solution, may be NULL                    lopt.cpp:108-110    */
    double* qp_obj;     /* [1]  0.5 x'Qx + c'x, may be NULL                                     */
    int* status;        /* [1]  0 ok; <0 failure (the reference swallows these, lopt.cpp:114), may be NULL:
                               WBC_ST_BAD_MODE / WBC_ST_NONFINITE = invalid inputs (nothing is solved, the observer state of the
                               instance is left as it was), -9 = non-positive diagonal of Q (opt.cpp:48178), -100 = other */
    int* qp_info;       /* [8]  ncholesky, outer its, QQP calls, working set, max KKT dim, flags, factorisations reused (of ncholesky), 0; may be NULL */
    double* qp_flops;   /* [1]  instrumented algorithmic flop count of the solve, may be NULL */
    long ld;
    double* w3;         /* [12] the estimate mapped onto the feet, w3 = pinv(J)' w with J = JacCOM_lin[:, 0:6], stacked foot order
                               (ESTIMATOR_SEM::getw3, estimator_sem.cpp:64-70): the least-norm foot forces whose CoM wrench is w.
                               May be NULL (then nothing is computed). */
} wbc_outputs;

/* Intermediates of update() for stage-by-stage validation (all may be NULL individually). */
typedef struct wbc_debug {
    double* M;            /* [324] getFreeFloatingMassMatrix        main.cpp:620 */
    double* h;            /* [18]  generalizedBiasForces            main.cpp:622 */
    double* g;            /* [18]  generalizedGravityForces         main.cpp:628 */
    double* Jac_lin;      /* [216] linear rows of Jac               main.cpp:632, 727-737 */
    double* Jdqd_lin;     /* [12]  linear rows of Jdqd              main.cpp:634 */
    double* com;          /* [3] */
    double* com_vel;      /* [3] */
    double* Mcom_b;       /* [36]  MassMatrixCOM[0:6,0:6]           main.cpp:645 */
    double* Mcom_j;       /* [144] MassMatrixCOM[6:18,6:18] */
    double* hcom;         /* [18]  BiasCOM                          main.cpp:648 */
    double* gcom;         /* [18]  GravMatrixCOM                    main.cpp:651 */
    double* Jcom_lin;     /* [216] JacCOM_lin                       main.cpp:655 */
    double* Jdqdcom_lin;  /* [12]  JdqdCOM_lin                      main.cpp:659 */
    double* foot_pos;     /* [12] */
    double* foot_vel;     /* [12] */
    double* Fgrf;         /* [12]                                   main.cpp:1022-1026 */
    double* Wcom_des;     /* [6]                                    main.cpp:1032 */
    long ld;
} wbc_debug;

void wbc_default_params(wbc_params* p);
const char* wbc_last_error(void);
const char* wbc_version(void);

/* ctx lifetime.  max_batch bounds n of every later call; device is the CUDA ordinal. */
int wbc_create(wbc_ctx** out, int device, int max_batch, const wbc_params* params);
int wbc_destroy(wbc_ctx* ctx);
int wbc_set_params(wbc_ctx* ctx, const wbc_params* params);

/* Observer state yd, yw (main.cpp:243, 721-724): SoA [6][ld], host pointers.  The ctx zero-initialises it. */
int wbc_set_observer_state(wbc_ctx* ctx, int n, const double* yd, const double* yw, long ld);
int wbc_get_observer_state(wbc_ctx* ctx, int n, double* yd, double* yw, long ld);
/* The second-order observer's extra integrator state ygamma (main.cpp:243; estimator_sem.cpp:20), same layout; zero-initialised. */
int wbc_set_observer_state2(wbc_ctx* ctx, int n, const double* ygamma, long ld);
int wbc_get_observer_state2(wbc_ctx* ctx, int n, double* ygamma, long ld);

/* One control cycle for n instances: update() -> Fgrf -> estimate() -> QP assembly -> solve -> tau.
 * `cuda_stream` is a cudaStream_t (NULL = the ctx's own stream). */
int wbc_cycle(wbc_ctx* ctx, int n, const wbc_inputs* in, const wbc_outputs* out, void* cuda_stream, unsigned flags);

/* update() only, with intermediates dumped.  Runs on a copy of the ctx's observer state (so Fgrf / Wcom_des are what the next
 * wbc_cycle would compute) and changes neither that state nor the records wbc_plant_step reads. */
int wbc_debug_update(wbc_ctx* ctx, int n, const wbc_inputs* in, const wbc_debug* dbg, unsigned flags);

/* The QP records the front kernel of the last wbc_cycle on this ctx left for the solver (internal layout, wbc_types.h: the
 * non-redundant content of Q, c, L): recs [n][*doubles_per_record], host pointer; recs == NULL only reports the record size.
 * Validation only: the tests compare the two front kernels (four lanes per instance, the default; a thread per instance,
 * WBC_FRONT=thread in the environment when the ctx is created) record by record. */
int wbc_debug_qp_records(wbc_ctx* ctx, int n, double* recs, int* doubles_per_record);

/* The OPT operator (lopt.h:5-36): n dense QPs of the controller's shape, instance-major:
 *   Q [n][30*30] row-major (lower triangle used, opt.cpp:4962), c [n][30], L [n][nrows*31] row-major,
 *   first neq rows "=", the rest "<=" (lopt.cpp:35-66); x [n][30].  nrows <= 86.
 *   info [n][8] (ncholesky, outer its, QQP calls, working-set size, KKT dimension, flags, Newton factorisations reused, 0)
 *   and flops [n] may be NULL.  A failed instance (status < 0) returns x = 0. */
int wbc_qp_solve(wbc_ctx* ctx, int n, const double* Q, const double* c, const double* L, int nrows, int neq, double* x,
                 int* status, int* info, double* flops, void* cuda_stream, unsigned flags);
/* wbc_qp_solve with the exact solver (WBC_QP_EXACT implied), warm-started: active [n][3] (host or device per flags, like x) is read
 * as each instance's warm set -- bit r of word r / 32 is inequality row r; bits at equality rows or beyond nrows are ignored, an
 * all-zero set is a cold start -- and overwritten with the instance's final active inequality rows (all zero when it failed).
 * Feeding the output back on the next call warm-starts a QP that changes little from call to call.  info[6], info[7] as for
 * WBC_QP_WARM. */
int wbc_qp_solve_warm(wbc_ctx* ctx, int n, const double* Q, const double* c, const double* L, int nrows, int neq, double* x,
                      int* status, int* info, double* flops, unsigned* active, void* cuda_stream, unsigned flags);
/* The exact-mode active sets the ctx stores per instance index (see WBC_QP_WARM): sets [4][ld], host pointer; rows 0..2 the active
 * inequality rows as bit masks, row 3 the contact mode they were solved in + 1 (0: no set).  The ctx zero-initialises them.
 * Restore them with the observer state after a checkpoint, or after moving instances to other indices or ctxs (re-sharding). */
int wbc_set_active_set(wbc_ctx* ctx, int n, const unsigned* sets, long ld);
int wbc_get_active_set(wbc_ctx* ctx, int n, unsigned* sets, long ld);

/* Synthetic plant of BASELINE config 5 (disturbance-rejection sweep).  Stands in for Gazebo + the ModelPush plugin
 * (force_plugin/src/force_plugin.cpp:124-491), which cannot run here: a CoM momentum integrator with locked joints,
 *     rho' = rho + T (-m g_acc e3 + Jc' Fgrf + push),  CoM_vel' = Mc^-1 rho',  T = params.obs_dt,
 * using the momentum balance the LAST wbc_cycle on this ctx computed for the same n instances (the balance
 * DOGCTRL::estimate() inverts, main.cpp:692-725).  Updates the base twist in place (omega' = CoM_vel'[3:6],
 * v' = CoM_vel'[0:3] - omega' x (com - base)) and, when base_pos is not NULL, base_pos += T v'.
 * Open loop (foot_force == NULL): Fgrf is what the last cycle measured.  Closed loop (foot_force != NULL, stance only):
 * the ground reacts with the commanded forces f* = x[18:30] of the last cycle's QP solution `x` [30][ld], and
 * foot_force [12][ld] is overwritten with R_foot' f* -- what the contact sensors report to the next cycle
 * (main.cpp:794-834, 1022-1026).
 * base_pos [3][ld], base_vel [6][ld], push [6][ld] (world wrench at the CoM); host or device pointers per flags. */
int wbc_plant_step(wbc_ctx* ctx, int n, double* base_pos, double* base_vel, double* foot_force, const double* x, const double* push,
                   long ld, void* cuda_stream, unsigned flags);

/* Forward-dynamics plant (SURVEY.md 8f-2): one control period (params.obs_dt) of every robot as an articulated body under the
 * joint torques `tau` [12][ld] (held over the period, like main.cpp's 400 Hz loop over Gazebo's 1 ms steps), a world wrench `push`
 * [6][ld] at the CoM and rigid bilateral point contacts at the stance feet of its contact mode:
 *     M nu_dot + h = S'tau + push_gen + Js' f,      Js nu_dot = -Jdqd_s - gamma Js nu,
 * `substeps` semi-implicit Euler substeps.  Stands in for Gazebo + the ModelPush plugin (force_plugin.cpp:124-491), which
 * cannot run here; the reference for this stage is a physics engine, so its parity is unpinned (checked against the oracle's
 * dense formulation and physics identities).  The state arrays are advanced IN PLACE; foot_force receives the contact forces in
 * the sensor frames (swing feet: 0), i.e. the next cycle's measured forces.  diag [2][ld] (may be NULL): contact-constraint
 * residual, smallest normal force (unilaterality is not enforced).  Host or device pointers per flags. */
typedef struct wbc_plant_state {
    double* base_pos;    /* [3]  */
    double* base_rot;    /* [9]  world_R_base, row-major */
    double* base_rpy;    /* [3]  */
    double* base_vel;    /* [6]  */
    double* q;           /* [12] */
    double* dq;          /* [12] */
    double* foot_force;  /* [12] out */
    const int* mode;     /* [1]  in  */
} wbc_plant_state;
int wbc_plant_dynamics_step(wbc_ctx* ctx, int n, const wbc_plant_state* st, const double* tau, const double* push, long ld, int substeps,
                            double gamma, double* diag, void* cuda_stream, unsigned flags);

/* Contact plant: forward dynamics with unilateral, frictional point contacts at the feet (DESIGN.md 4.5).  One control period
 * (params.obs_dt) of every robot under the joint torques `tau` [12][ld] and the world wrench `push` [6][ld] at the CoM, in `substeps`
 * steps of dt.  Each foot point k (stacked order) has its own horizontal ground plane z = ground_z[k] ([4][ld], NULL = 0) and friction
 * coefficient mu ([1][ld], NULL = params.mu; mu >= 0).  Per step: nu_free = nu + dt M^-1 (S'tau + push_gen - h); the candidate feet
 * are those whose gap phi_k = p_k,z - ground_z[k] <= margin (geometry only: st->mode is not read and may be NULL); the contact
 * impulses lambda (3 per candidate foot, world axes) are the unique minimiser of
 *     min 1/2 lambda'(G + eps D) lambda + lambda'(J nu_free - b),   G = J M^-1 J', D = diag(G),
 * over every candidate foot's friction pyramid (lambda_z >= 0, |lambda_x|, |lambda_y| <= mu lambda_z), with b = 0 tangentially and
 * -phi/dt (phi >= 0) or -beta phi/dt (phi < 0) along the normal; nu+ = nu_free + M^-1 J' lambda, then semi-implicit Euler.  This is
 * the convex (Anitescu-type) relaxation of Coulomb contact: a sticking foot is exact; a sliding foot drifts off the plane at a normal
 * velocity of at most mu times its slip speed.  Each QP is solved to its KKT optimum (a Goldfarb-Idnani dual active-set method,
 * warm-started from the previous step's active rows, at most max_iter dual steps).
 * The state advances in place; foot_force receives the last step's contact forces lambda/dt in the sensor frames (R_foot' lambda / dt,
 * 0 off contact), as from wbc_plant_dynamics_step.  contact [4][ld] (may be NULL), last step: 0 no contact force, 1 sticking,
 * 2 sliding (a friction row active) -- a gait loop can end a swing phase on touchdown.  diag [4][ld] (may be NULL): largest
 * penetration over the steps (gaps at each step's start), smallest normal force of a candidate foot, largest scaled KKT residual of
 * the contact QPs, total dual active-set steps.  status [ld] (may be NULL): 0; WBC_ST_NONFINITE for a NaN or infinity among the
 * inputs or produced from them; -100 when a contact QP reaches max_iter.  A failed instance's state (foot_force included) is left
 * as it was at the start of the call, and its contact flags are 0.  Host or device pointers per flags, like wbc_plant_dynamics_step. */
typedef struct wbc_contact_params {
    double beta;     /* 0.2:  Baumgarte factor of the push-out of a penetrating foot          */
    double eps;      /* 1e-8: regularisation of the Delassus matrix, G + eps diag(G)           */
    double margin;   /* 2e-3: a foot is a contact candidate when its gap is <= margin (m)     */
    int max_iter;    /* 64:   dual active-set steps per contact QP before status -100          */
} wbc_contact_params;
void wbc_default_contact_params(wbc_contact_params* cp);
int wbc_plant_contact_step(wbc_ctx* ctx, int n, const wbc_plant_state* st, const double* tau, const double* push, const double* ground_z,
                           const double* mu, long ld, int substeps, const wbc_contact_params* cp, int* contact, double* diag, int* status,
                           void* cuda_stream, unsigned flags);
/* Contact plant on inclined ground: wbc_plant_contact_step with each foot's plane, contact frame and friction coefficient taken
 * from the controller's terrain layout (wbc_inputs.terrain), so that the plant's ground is the ground the controller is told about.
 * terrain [40][ld] (required; flat ground is wbc_plant_contact_step): for stacked foot k, rows 10k..10k+2 the unit normal n,
 * +3..+5 the tangent t1, +6..+8 the tangent t2, +9 mu.  plane_d [4][ld] (NULL = 0): foot k's plane is {p : n . p = d_k}.  Per step
 * the gap is measured along the normal, phi_k = n . p_k - d_k (candidates, speculative and Baumgarte targets, diag[0]); each
 * candidate foot's impulse is expressed in its frame, lambda = (lambda_t1, lambda_t2, lambda_n) with Jacobian rows F' J, F = [t1 t2 n],
 * over the pyramid |lambda_t1|, |lambda_t2| <= mu lambda_n, lambda_n >= 0 -- the controller's cone rows.  foot_force gets
 * R_foot' F lambda / dt; contact flags, diag (diag[1]: smallest lambda_n / dt) and status as in wbc_plant_contact_step.  An
 * instance whose frame is not orthonormal to 1e-9 or whose mu < 0 is refused with WBC_ST_BAD_TERRAIN, one with a non-finite terrain
 * or plane_d entry with WBC_ST_NONFINITE; its state is untouched and its flags are 0.  A foot keeps its plane for the whole call. */
int wbc_plant_contact_step_terrain(wbc_ctx* ctx, int n, const wbc_plant_state* st, const double* tau, const double* push,
                                   const double* terrain, const double* plane_d, long ld, int substeps, const wbc_contact_params* cp,
                                   int* contact, double* diag, int* status, void* cuda_stream, unsigned flags);

/* Device-side timing of the last wbc_cycle on this ctx (CUDA events on the launching stream), ms. */
int wbc_last_timing(wbc_ctx* ctx, float* front_ms, float* solve_ms);
/* Per-instance solve duration of the last wbc_cycle on this ctx, in SM clock cycles (clock64 around the instance's
 * set-up + DENSE-AUL solve + torque map; the figure that orders the next cycle's longest-first dispatch -- except for small batches
 * on the one-warp-per-solve kernel with express lanes, where the order goes by the solve's flop count, see DESIGN.md).
 * cycles [n], host pointer; synchronises the ctx's last launch stream work via a blocking copy. */
int wbc_last_solve_cycles(wbc_ctx* ctx, int n, unsigned long long* cycles);
/* Number of kernels launched by the last wbc_cycle / wbc_qp_solve. */
int wbc_last_launches(wbc_ctx* ctx);
/* Launch shape of the persistent solver kernel: resident CTAs (= warps) per SM as the occupancy calculator reports them
 * for this device, dynamic shared memory per CTA in bytes, and the grid of the last wbc_cycle (before any: SMs x resident
 * CTAs; small batches are launched with fewer CTAs per SM), and which solver kernel the last wbc_cycle ran (0: one warp per
 * solve, 1: stage tasks with SM roles -- chosen by batch size, see DESIGN.md; 2: the exact-mode kernel of WBC_QP_EXACT, whose
 * resident CTAs per SM and shared memory are then reported).  Any pointer may be NULL.
 * Measurement only (bench.py reports it beside the roofline); the reference has no counterpart. */
int wbc_solver_shape(wbc_ctx* ctx, int* ctas_per_sm, int* smem_bytes, int* grid, int* stage_tasks);
/* Per-warp profile of the last solver launch when the ctx was created with WBC_STAGE_PROF=1 in the environment: rows of 12
 * counters (cycles in QLOOP / UPDATE / SETUP tasks, their counts, cycles looking for a task, cycles in fences and queue
 * operations, tasks taken from the other role's queue, cycles in the kernel, role, SM id).  Returns the rows written (<= max_rows)
 * or a negative error.  Measurement only. */
int wbc_stage_profile(wbc_ctx* ctx, unsigned long long* out, int max_rows);

/* ---- On-device trajectory sampling (SURVEY.md 8f-1) -------------------------------------------------------------
 * The reference samples four towr::Spline objects at wall-clock time t on the host every cycle: base_linear_ and
 * base_angular_ (main.cpp:1004-1010) and ee_motion_ of the two swing feet (main.cpp:1333-1368); towr::Spline::GetPoint
 * is spline.cc:48-93, the cubic-Hermite coefficients polynomial.cc:98-104.  wbc_set_trajectory uploads the node tables
 * of a plan once; wbc_sample_trajectory evaluates them on the GPU for every instance, so a cycle needs only t. */
#define WBC_TRAJ_SPLINES 4   /* 0 base_linear, 1 base_angular, 2 first swing foot, 3 second swing foot (Jsw row order) */
#define WBC_TRAJ_MAX_SEG 8
typedef struct wbc_trajectory {
    int nseg;                  /* cubic-Hermite polynomials per spline, 1..WBC_TRAJ_MAX_SEG                              */
    const double* durations;   /* [4*nseg][ld]        row s*nseg + j: duration of polynomial j of spline s               */
    const double* nodes;       /* [4*(nseg+1)*6][ld]  row (s*(nseg+1) + k)*6 + c: node k, c = 0..2 position, 3..5 velocity */
    long ld;
} wbc_trajectory;
typedef struct wbc_traj_samples {   /* the six desired-trajectory arrays of wbc_inputs, each [6][ld] */
    double *com_des_pos, *com_des_vel, *com_des_acc, *sw_des_pos, *sw_des_vel, *sw_des_acc;
    long ld;
} wbc_traj_samples;
/* Upload (host pointers) or copy (WBC_DEVICE_PTRS) the plan of n instances into the ctx. */
int wbc_set_trajectory(wbc_ctx* ctx, int n, const wbc_trajectory* tr, void* cuda_stream, unsigned flags);
/* Sample the ctx's plan at time t[i] per instance (t == NULL: t_all for every instance).  One kernel launch.
 * out == NULL: the samples stay in the ctx, for a following wbc_cycle(..., WBC_SAMPLED_TRAJ);
 * out != NULL: written to the caller's arrays -- device arrays with WBC_DEVICE_PTRS (e.g. the ones handed to
 * wbc_cycle as device inputs), else host arrays (a D2H copy; for inspection and tests).  t follows the same flag.
 * The sampling and the cycle that consumes it must be ordered: pass both the same stream (NULL = the ctx's own). */
int wbc_sample_trajectory(wbc_ctx* ctx, int n, const double* t, double t_all, const wbc_traj_samples* out, void* cuda_stream, unsigned flags);

/* ---- On-device trot gait generator (DESIGN.md 4.8) --------------------------------------------------------------
 * A per-robot trot (phases 0 stance, 1 swing{BR,FL}, 2 stance, 3 swing{BL,FR}) that turns a velocity command, the robot's state
 * and the contact plant's flags into the contact mode and the six desired-trajectory arrays of wbc_inputs, once per control cycle
 * (dt = params.obs_dt), so that wbc_gait_step -> wbc_cycle -> wbc_plant_contact_step runs without a host round trip.  It stands in
 * for the reference's TOWR plan: the CoM reference integrates the (ramped) command and is held within `leash` of the measured CoM;
 * a swing foot follows a quintic from its lift-off point to a Raibert-style touchdown target with a sin^2 lift of step_height, and
 * its swing ends early when both swing feet are in contact past half of the phase. */
typedef struct wbc_gait_params {
    int stance_cycles;    /* 46:   control cycles of each stance phase                                               */
    int swing_cycles;     /* 46:   control cycles of each swing phase (>= 2)                                         */
    double step_height;   /* 0.03: foot lift (m), the apex of the sin^2 profile at mid-swing                          */
    double k_v;           /* 0.1:  touchdown target correction per m/s of measured minus reference velocity (s)        */
    double max_step;      /* 0.1:  largest distance of a touchdown target from its neutral point (m)                   */
    double acc_lin;       /* 1.0:  largest change of the reference (vx, vy) per second (m/s^2)                         */
    double acc_yaw;       /* 2.0:  largest change of the reference yaw rate per second (rad/s^2)                       */
    double leash;         /* 0.05: largest distance of the CoM reference from the measured CoM in xy (m, > 0)          */
} wbc_gait_params;
void wbc_default_gait_params(wbc_gait_params* gp);
/* Gait state, caller-owned SoA arrays [k][ld] (a checkpoint is a copy of them). */
typedef struct wbc_gait_state {
    int* phase;        /* [1] 0..3                                                                                      */
    int* tick;         /* [1] cycles into the phase, 0 .. phase length - 1                                              */
    int* landed;       /* [1] 1 once the current swing has touched down (the robot is then in stance until the phase ends) */
    double* com_ref;   /* [4] CoM reference x, y (world), clearance of the CoM above the ground, reference yaw            */
    double* v_ref;     /* [3] reference velocity vx, vy (heading frame, i.e. rotated by the reference yaw) and yaw rate   */
    double* liftoff;   /* [6] lift-off points of the current (or next) swing pair, Jsw row order: first foot xyz, second  */
    double* target;    /* [6] their touchdown targets (equal to liftoff outside a swing phase at init)                   */
    double* offset;    /* [8] xy of each stacked foot from its hip in the heading frame, captured at init                 */
} wbc_gait_state;
/* Capture the gait state of n robots from the plant state: start offset k0 [ld] (NULL = 0; taken modulo the gait period
 * 2 (stance_cycles + swing_cycles)) gives phase and tick, landed = 0; com_ref = (measured CoM xy, CoM height above the ground,
 * base yaw), v_ref = 0, the foot offsets; a robot that starts in a swing phase gets its lift-off points and targets from the current
 * state.  terrain [40][ld] / plane_d [4][ld] (NULL: flat ground z = 0) as in wbc_plant_contact_step_terrain: the ground height under
 * a point is the mean of the four feet's plane heights there.  gp NULL = the defaults.  status [ld] (may be NULL): 0;
 * WBC_ST_NONFINITE for a non-finite input; WBC_ST_BAD_TERRAIN for a foot frame that is not orthonormal to 1e-9 or whose normal has
 * n_z < 0.5.  A refused robot's gait state is left untouched.  Host or device pointers per flags (st->foot_force, st->dq and
 * st->mode are not read). */
int wbc_gait_init(wbc_ctx* ctx, int n, const wbc_gait_params* gp, const wbc_plant_state* st, const int* k0, const double* terrain,
                  const double* plane_d, wbc_gait_state* gs, int* status, long ld, void* cuda_stream, unsigned flags);
/* One gait step of n robots (DESIGN.md 4.8): touchdown from contact [4][ld] (the flags of the previous wbc_plant_contact_step; NULL:
 * a swing lasts its whole phase), lift-off, the ramp of v_ref toward cmd [3][ld] (vx, vy in the heading frame, yaw rate; NULL = 0,
 * a trot in place), the CoM reference; writes mode [ld] and the six desired arrays of `out` (com_des_* [6][out->ld]: x, y, z, roll 0,
 * pitch 0, yaw on the measured base_rpy branch; sw_des_* in Jsw row order), then advances the state.  terrain / plane_d as in
 * wbc_gait_init.  Bad params (non-finite, stance_cycles < 1, swing_cycles < 2, a negative step_height, k_v, max_step, acc_lin or
 * acc_yaw, leash <= 0) return WBC_EINVAL with nothing done.  status [ld] (may be NULL): as wbc_gait_init, plus WBC_ST_BAD_MODE for a
 * phase outside 0..3 or a tick outside its phase; a refused robot's state, mode and outputs are left untouched.  st->mode is not
 * read.  Host or device pointers per flags, WBC_NO_SYNC with device pointers. */
int wbc_gait_step(wbc_ctx* ctx, int n, const wbc_gait_params* gp, wbc_gait_state* gs, const wbc_plant_state* st, const double* cmd,
                  const int* contact, const double* terrain, const double* plane_d, int* mode, const wbc_traj_samples* out, int* status,
                  long ld, void* cuda_stream, unsigned flags);

/* Page-locked host memory for the SoA arrays handed to wbc_cycle with WBC_HOST_PTRS.  Arrays that are page-locked
 * (from here, cudaMallocHost or cudaHostRegister) are copied to and from the device directly; pageable arrays go
 * through the ctx's pinned bounce buffer (one extra host-side pass over the data). */
int wbc_host_alloc(void** p, size_t bytes);
int wbc_host_free(void* p);

/* FP64 DFMA peak microbenchmark (roofline denominator): returns achieved FLOP/s on the ctx's device. */
int wbc_measure_dfma_peak(wbc_ctx* ctx, double* flops_per_s);

#ifdef __cplusplus
}
#endif
#endif
