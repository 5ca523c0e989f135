"""TEST INFRASTRUCTURE ONLY -- ctypes bindings for the CPU oracle.

  libwbc_oracle.so            our plain-C restatement of the reference control cycle (oracle/wbc_oracle.c)
  _ref/libref_alglib_qp.so    the reference's own vendored ALGLIB, compiled from /root/reference
                              (oracle/Makefile `make ref`); the pinned QP oracle.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module (the product package never does).
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "libwbc_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libref_alglib_qp.so")

MODE_STANCE, MODE_SWING_BR_FL, MODE_SWING_BL_FR = 0, 1, 2


class Params(C.Structure):
    _fields_ = [(n, C.c_double) for n in
                ("kcom", "dcom", "q1_weight", "slack_weight", "mu", "tau_max", "joint_dt", "kp_sw", "kd_sw",
                 "g_acc", "obs_gain", "obs_dt")] + [("observer_enabled", C.c_int), ("fix_swing_rhs", C.c_int),
                                                    ("obs_gain2", C.c_double), ("obs_order", C.c_int), ("obs_form", C.c_int)]


class In(C.Structure):
    _fields_ = [("base_pos", C.c_double * 3), ("base_R", C.c_double * 9), ("rpy", C.c_double * 3),
                ("base_vel", C.c_double * 6), ("q", C.c_double * 12), ("dq", C.c_double * 12),
                ("gravity", C.c_double * 3),
                ("com_des_pos", C.c_double * 6), ("com_des_vel", C.c_double * 6), ("com_des_acc", C.c_double * 6),
                ("mode", C.c_int),
                ("sw_des_pos", C.c_double * 6), ("sw_des_vel", C.c_double * 6), ("sw_des_acc", C.c_double * 6),
                ("foot_force", C.c_double * 12), ("terrain", C.c_double * 40), ("has_terrain", C.c_int),
                ("yd_prev", C.c_double * 6), ("yw_prev", C.c_double * 6), ("yg_prev", C.c_double * 6)]


class Out(C.Structure):
    _fields_ = [("tau", C.c_double * 12), ("w", C.c_double * 6), ("yd", C.c_double * 6), ("yw", C.c_double * 6),
                ("x", C.c_double * 30), ("qp_obj", C.c_double), ("status", C.c_int), ("ncholesky", C.c_int),
                ("yg", C.c_double * 6)]


class Dyn(C.Structure):
    _fields_ = [("M", C.c_double * 324), ("h", C.c_double * 18), ("g", C.c_double * 18),
                ("Jac_lin", C.c_double * 216), ("Jdqd_lin", C.c_double * 12),
                ("com", C.c_double * 3), ("com_vel", C.c_double * 3),
                ("foot_pos", C.c_double * 12), ("foot_vel", C.c_double * 12), ("foot_R", C.c_double * 36),
                ("T", C.c_double * 324), ("T_inv_dot", C.c_double * 324),
                ("Mcom", C.c_double * 324), ("hcom", C.c_double * 18), ("gcom", C.c_double * 18),
                ("Jcom_lin", C.c_double * 216), ("Jdqdcom_lin", C.c_double * 12)]


class Qp(C.Structure):
    _fields_ = [("Q", C.c_double * 900), ("c", C.c_double * 30), ("L", C.c_double * (86 * 31)),
                ("nrows", C.c_int), ("neq", C.c_int), ("Fgrf", C.c_double * 12), ("Wcom_des", C.c_double * 6)]


QP_FN = C.CFUNCTYPE(C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, C.c_int,
                    C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_int))


def build(ref=True, quiet=True):
    """Compile the oracle (always) and oracle/_ref (only when /root/reference is present)."""
    kw = dict(stdout=subprocess.DEVNULL, stderr=subprocess.STDOUT) if quiet else {}
    subprocess.check_call(["make", "-C", HERE, "oracle"], **kw)
    if ref and os.path.isdir("/root/reference") and not os.path.exists(REF_SO):
        subprocess.check_call(["make", "-C", HERE, "ref", "-j6"], **kw)


_oracle = None
_ref = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        if not os.path.exists(ORACLE_SO):
            build(ref=False)
        lib = C.CDLL(ORACLE_SO)
        lib.wbc_oracle_default_params.argtypes = [C.POINTER(Params)]
        lib.wbc_oracle_update.argtypes = [C.POINTER(In), C.POINTER(Dyn)]
        lib.wbc_oracle_cycle.argtypes = [C.POINTER(Params), C.POINTER(In), C.c_void_p, C.POINTER(Out),
                                         C.POINTER(Dyn), C.POINTER(Qp)]
        lib.wbc_oracle_cycle.restype = C.c_int
        lib.wbc_oracle_batch.argtypes = [C.POINTER(Params), C.POINTER(In), C.c_int, C.c_int, C.c_void_p,
                                         C.POINTER(Out)]
        lib.wbc_oracle_batch.restype = C.c_double
        _oracle = lib
    return _oracle


def ref_lib():
    """The compiled reference ALGLIB.  Raises FileNotFoundError if oracle/_ref was never built."""
    global _ref
    if _ref is None:
        if not os.path.exists(REF_SO):
            raise FileNotFoundError(REF_SO + " (run `make -C oracle ref` where /root/reference exists)")
        lib = C.CDLL(REF_SO)
        dp = C.POINTER(C.c_double)
        lib.ref_qp_solve.argtypes = [dp, dp, dp, C.c_int, C.c_int, dp, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        lib.ref_qp_solve.restype = C.c_int
        lib.ref_qp_solve_ex.argtypes = [C.c_int, dp, dp, dp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, dp,
                                        C.POINTER(C.c_int), C.POINTER(C.c_int)]
        lib.ref_qp_solve_ex.restype = C.c_int
        lib.ref_qp_solve_exact.argtypes = [C.c_int, dp, dp, dp, C.c_int, C.c_int, dp]
        lib.ref_qp_solve_exact.restype = C.c_int
        _ref = lib
    return _ref


def have_ref():
    return os.path.exists(REF_SO)


def default_params(observer_enabled=1):
    p = Params()
    oracle_lib().wbc_oracle_default_params(C.byref(p))
    p.observer_enabled = observer_enabled
    return p


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def ref_qp_solve(Q, c, L, neq, exact=False):
    """Solve one QP with the compiled reference ALGLIB (reference settings). Returns (x, ncholesky, rc)."""
    Q = np.ascontiguousarray(Q, dtype=np.float64)
    c = np.ascontiguousarray(c, dtype=np.float64)
    L = np.ascontiguousarray(L, dtype=np.float64)
    x = np.zeros(Q.shape[0])
    if exact:
        rc = ref_lib().ref_qp_solve_exact(Q.shape[0], _dp(Q), _dp(c), _dp(L), L.shape[0], neq, _dp(x))
        return x, 0, rc
    nch, tt = C.c_int(0), C.c_int(0)
    rc = ref_lib().ref_qp_solve(_dp(Q), _dp(c), _dp(L), L.shape[0], neq, _dp(x), C.byref(nch), C.byref(tt))
    return x, nch.value, rc


# ---------------------------------------------------------------------------------------------
# SoA numpy scenario dict (wbc_quadruped_dob_b200.scenarios) -> array of oracle `In` structs
_FIELDS = [("base_pos", 3), ("base_R", 9), ("rpy", 3), ("base_vel", 6), ("q", 12), ("dq", 12),
           ("com_des_pos", 6), ("com_des_vel", 6), ("com_des_acc", 6),
           ("sw_des_pos", 6), ("sw_des_vel", 6), ("sw_des_acc", 6), ("foot_force", 12),
           ("yd_prev", 6), ("yw_prev", 6)]
_SOA_NAME = {"base_R": "base_rot", "rpy": "base_rpy", "yd_prev": "obs_yd", "yw_prev": "obs_yw"}


def to_structs(sc, gravity=(0.0, 0.0, -9.8)):
    n = sc["mode"].shape[0]
    arr = (In * n)()
    view = np.frombuffer(arr, dtype=np.dtype(In))
    for name, k in _FIELDS:
        src = sc[_SOA_NAME.get(name, name)]          # [k][n]
        view[name][:] = np.ascontiguousarray(src.T)
    view["mode"][:] = sc["mode"]
    view["yg_prev"][:] = np.ascontiguousarray(sc["obs_yg"].T) if sc.get("obs_yg") is not None else 0.0
    view["gravity"][:] = np.asarray(gravity, dtype=np.float64)[None, :]
    if sc.get("terrain") is not None:
        view["terrain"][:] = np.ascontiguousarray(sc["terrain"].T)
        view["has_terrain"][:] = 1
    else:
        view["has_terrain"][:] = 0
    return arr


def qp_solver(solver):
    """The oracle's QP solver as a C function pointer: "ref" is the compiled reference ALGLIB; otherwise a ctypes function of the
    wbc_qp_fn signature (QP_FN), for tests that must run where the reference ALGLIB is not built."""
    if isinstance(solver, C._CFuncPtr):
        return C.cast(solver, C.c_void_p)
    if solver == "ref":
        return C.cast(ref_lib().ref_qp_solve, C.c_void_p)
    raise ValueError("the oracle's QP solver is the compiled reference ALGLIB or a wbc_qp_fn C function")


def run_cycle_batch(sc, params=None, nthreads=1, solver="ref", gravity=(0.0, 0.0, -9.8)):
    """Full oracle control cycle on every instance.  Returns (dict of [n][k] arrays, wall seconds).  solver: see qp_solver."""
    params = params or default_params()
    n = sc["mode"].shape[0]
    arr = to_structs(sc, gravity)
    out = (Out * n)()
    fn = qp_solver(solver)
    secs = oracle_lib().wbc_oracle_batch(C.byref(params), arr, n, nthreads, fn, out)
    v = np.frombuffer(out, dtype=np.dtype(Out))
    res = {k: np.array(v[k]) for k in ("tau", "w", "yd", "yw", "yg", "x", "qp_obj", "status", "ncholesky")}
    return res, secs


def run_cycle_one(sc, i, params=None, gravity=(0.0, 0.0, -9.8), solver="ref"):
    """One instance with all intermediates (Out, Dyn, Qp ctypes structs)."""
    params = params or default_params()
    one = {k: (v[..., i:i + 1] if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    arr = to_structs(one, gravity)
    out, dyn, qp = Out(), Dyn(), Qp()
    fn = qp_solver(solver)
    oracle_lib().wbc_oracle_cycle(C.byref(params), C.byref(arr[0]), fn, C.byref(out), C.byref(dyn), C.byref(qp))
    return out, dyn, qp


def update_only(sc, i, gravity=(0.0, 0.0, -9.8)):
    one = {k: (v[..., i:i + 1] if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    arr = to_structs(one, gravity)
    dyn = Dyn()
    oracle_lib().wbc_oracle_update(C.byref(arr[0]), C.byref(dyn))
    return dyn


def assemble_only(sc, i, params=None, w=None, gravity=(0.0, 0.0, -9.8)):
    """update() + QP assembly without solving; returns (Dyn, Qp)."""
    params = params or default_params()
    lib = oracle_lib()
    lib.wbc_oracle_assemble.argtypes = [C.POINTER(Params), C.POINTER(In), C.POINTER(Dyn), C.POINTER(C.c_double),
                                        C.POINTER(Qp)]
    one = {k: (v[..., i:i + 1] if isinstance(v, np.ndarray) else v) for k, v in sc.items()}
    arr = to_structs(one, gravity)
    dyn, qp = Dyn(), Qp()
    lib.wbc_oracle_update(C.byref(arr[0]), C.byref(dyn))
    wv = (C.c_double * 6)(*(w if w is not None else [0.0] * 6))
    lib.wbc_oracle_assemble(C.byref(params), C.byref(arr[0]), C.byref(dyn), wv, C.byref(qp))
    return dyn, qp


def run_cycle_batch_gains(sc, params=None, nthreads=1, solver="ref"):
    """run_cycle_batch for a scenario with a per-instance observer gain sc["obs_gain"] (BASELINE config 5):
    the oracle's gain is a scalar parameter like the reference's literal (main.cpp:708), so instances are grouped."""
    gains = sc.get("obs_gain")
    if gains is None:
        return run_cycle_batch(sc, params, nthreads, solver)
    n = sc["mode"].shape[0]
    res, secs = None, 0.0
    for gval in np.unique(gains):
        idx = np.nonzero(gains == gval)[0]
        sub = {k: (np.ascontiguousarray(v[..., idx]) if isinstance(v, np.ndarray) else v) for k, v in sc.items() if k != "obs_gain"}
        p = default_params() if params is None else params
        p2 = Params.from_buffer_copy(p)
        p2.obs_gain = float(gval)
        r, s = run_cycle_batch(sub, p2, nthreads, solver)
        secs += s
        if res is None:
            res = {k: np.zeros((n,) + v.shape[1:], dtype=v.dtype) for k, v in r.items()}
        for k, v in r.items():
            res[k][idx] = v
    return res, secs


def plant_step(sc, push, x=None, params=None, gravity=(0.0, 0.0, -9.8)):
    """Synthetic plant of BASELINE config 5 (wbc_oracle_plant_step) on every instance; push [6][n]; x [n][30] (the
    oracle's QP solutions) closes the loop.  Returns (base_pos [3][n], base_vel [6][n], foot_force [12][n] or None)."""
    params = params or default_params()
    lib = oracle_lib()
    pd = C.POINTER(C.c_double)
    lib.wbc_oracle_plant_step.argtypes = [C.POINTER(Params), C.POINTER(In), pd, pd, pd, pd, pd]
    lib.wbc_oracle_plant_step.restype = None
    n = sc["mode"].shape[0]
    arr = to_structs(sc, gravity)
    pos, vel, ff = np.zeros((n, 3)), np.zeros((n, 6)), np.zeros((n, 12))
    pt = np.ascontiguousarray(np.asarray(push, dtype=np.float64).T)
    xs = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
    for i in range(n):
        lib.wbc_oracle_plant_step(C.byref(params), C.byref(arr[i]), _dp(pt[i]), _dp(xs[i]) if xs is not None else None, _dp(pos[i]),
                                  _dp(vel[i]), _dp(ff[i]))
    return np.ascontiguousarray(pos.T), np.ascontiguousarray(vel.T), (np.ascontiguousarray(ff.T) if xs is not None else None)


def fdyn_step(sc, tau, push, params=None, nsub=5, gamma=100.0, gravity=(0.0, 0.0, -9.8)):
    """Forward dynamics with hard contacts (wbc_oracle_fdyn_step) on every instance: tau [12][n], push [6][n] (world wrench at
    the CoM).  Returns (next-state dict with base_pos, base_rot, base_rpy, base_vel, q, dq, foot_force in SoA layout, diag [n][2])."""
    params = params or default_params()
    lib = oracle_lib()
    pd = C.POINTER(C.c_double)
    lib.wbc_oracle_fdyn_step.argtypes = [C.POINTER(Params), C.POINTER(In), pd, pd, C.c_int, C.c_double, C.POINTER(In), pd, pd]
    lib.wbc_oracle_fdyn_step.restype = None
    n = sc["mode"].shape[0]
    arr = to_structs(sc, gravity)
    tt = np.ascontiguousarray(np.asarray(tau, dtype=np.float64).T)
    pt = np.ascontiguousarray(np.asarray(push, dtype=np.float64).T)
    nxt = {"base_pos": np.zeros((3, n)), "base_rot": np.zeros((9, n)), "base_rpy": np.zeros((3, n)), "base_vel": np.zeros((6, n)),
           "q": np.zeros((12, n)), "dq": np.zeros((12, n)), "foot_force": np.zeros((12, n))}
    diag = np.zeros((n, 2))
    ff = np.zeros(12)
    o = In()
    for i in range(n):
        lib.wbc_oracle_fdyn_step(C.byref(params), C.byref(arr[i]), _dp(tt[i]), _dp(pt[i]), int(nsub), float(gamma), C.byref(o), _dp(ff), _dp(diag[i]))
        nxt["base_pos"][:, i] = o.base_pos; nxt["base_rot"][:, i] = o.base_R; nxt["base_rpy"][:, i] = o.rpy
        nxt["base_vel"][:, i] = o.base_vel; nxt["q"][:, i] = o.q; nxt["dq"][:, i] = o.dq; nxt["foot_force"][:, i] = ff
    return nxt, diag


def spline_point(durations, nodes, t):
    """towr::Spline::GetPoint (oracle restatement): durations [nseg], nodes [nseg+1, 6] -> (id, p, v, a)."""
    lib = oracle_lib()
    pd = C.POINTER(C.c_double)
    lib.wbc_oracle_spline_point.argtypes = [C.c_int, pd, pd, C.c_double, pd, pd, pd]
    lib.wbc_oracle_spline_point.restype = C.c_int
    d = np.ascontiguousarray(durations, dtype=np.float64)
    nd = np.ascontiguousarray(nodes, dtype=np.float64)
    p, v, a = np.zeros(3), np.zeros(3), np.zeros(3)
    sid = lib.wbc_oracle_spline_point(d.shape[0], d.ctypes.data_as(pd), nd.ctypes.data_as(pd), float(t), p.ctypes.data_as(pd),
                                      v.ctypes.data_as(pd), a.ctypes.data_as(pd))
    return sid, p, v, a


def sample_trajectory(traj, t):
    """All instances of a plan (scenarios.make_trajectory layout) at times t [n] -> dict of the six [6, n] arrays."""
    nseg, dur, nodes = traj["nseg"], traj["durations"], traj["nodes"]
    n = dur.shape[1]
    out = {k: np.zeros((6, n)) for k in ("com_des_pos", "com_des_vel", "com_des_acc", "sw_des_pos", "sw_des_vel", "sw_des_acc")}
    for i in range(n):
        for s in range(4):
            d = dur[s * nseg:(s + 1) * nseg, i]
            nd = nodes[s * (nseg + 1) * 6:(s + 1) * (nseg + 1) * 6, i].reshape(nseg + 1, 6)
            sid, p, v, a = spline_point(d, nd, t[i])
            assert sid >= 0, "time outside the plan"
            pre, r0 = ("com_des_" if s < 2 else "sw_des_"), (s & 1) * 3
            out[pre + "pos"][r0:r0 + 3, i] = p
            out[pre + "vel"][r0:r0 + 3, i] = v
            out[pre + "acc"][r0:r0 + 3, i] = a
    return out


def foot_wrench_map(Jcom_lin, w):
    """ESTIMATOR_SEM::getw3 (estimator_sem.cpp:64-70): w3 = pinv(J)' w with J = JacCOM_lin[:, 0:6] (12 x 6).  The reference takes the
    pseudo-inverse from Eigen's complete orthogonal decomposition; numpy's SVD-based pinv is the same Moore-Penrose matrix."""
    J = np.asarray(Jcom_lin, dtype=np.float64).reshape(12, 18)[:, :6]
    return np.linalg.pinv(J).T @ np.asarray(w, dtype=np.float64)
