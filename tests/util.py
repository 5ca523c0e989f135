"""Shared helpers for the tests (test infrastructure only)."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
EMU_DIR = os.path.join(ROOT, "tests", "host_emu")
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)

IN_NAMES = ("base_pos base_rot base_rpy base_vel q dq com_des_pos com_des_vel com_des_acc sw_des_pos sw_des_vel "
            "sw_des_acc foot_force").split()

# north_star tolerances
TOL_TAU = 1e-6      # torques, relative to max |tau| of the instance
TOL_OBJ = 1e-8      # QP objective, relative
TOL_OBS = 1e-9      # observer estimates


def rel_rows(a, b):
    """Per-instance relative error: max_k |a-b| / max(1e-30, max_k |b|); arrays are [n, k]."""
    return np.max(np.abs(a - b), axis=1) / np.maximum(1e-30, np.max(np.abs(b), axis=1))


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    sc = {k[3:]: z[k] for k in z.files if k.startswith("in_")}
    out = {k[4:]: z[k] for k in z.files if k.startswith("out_")}
    sc.setdefault("terrain", None)
    return sc, out


def _build_emu(src, so):
    if not os.path.exists(so) or os.path.getmtime(so) < max(
            os.path.getmtime(os.path.join(ROOT, "wbc_quadruped_dob_b200", "csrc", f))
            for f in os.listdir(os.path.join(ROOT, "wbc_quadruped_dob_b200", "csrc"))) or \
            os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", so, src])


class EmuParams(C.Structure):
    _fields_ = [(n, C.c_double) for n in
                "kcom dcom q1_weight slack_weight mu tau_max joint_dt kp_sw kd_sw g_acc obs_gain obs_dt".split()] + \
               [("gravity", C.c_double * 3), ("qp_epsx", C.c_double), ("qp_rho", C.c_double), ("obs_gain2", C.c_double),
                ("qp_outerits", C.c_int), ("observer_enabled", C.c_int), ("fix_swing_rhs", C.c_int), ("qp_literal_kkt", C.c_int),
                ("hold_tau_on_failure", C.c_int), ("obs_order", C.c_int), ("obs_form", C.c_int)]


class _EmuIO(C.Structure):
    _fields_ = [(n, _dp) for n in IN_NAMES + ["terrain"]] + \
               [("mode", _ip), ("ld", C.c_long), ("yd", _dp), ("yw", _dp), ("tau", _dp), ("w", _dp), ("x", _dp),
                ("qp_obj", _dp), ("status", _ip), ("info", _ip), ("rec", _dp), ("yg", _dp), ("w3", _dp)]


def emu_default_params():
    return EmuParams(2500, 50, 50, 1e8, 0.6, 60, 0.025, 300, 20, 9.81, 10, 0.0025, (C.c_double * 3)(0, 0, -9.8),
                     1e-2, 1e4, 1.0, 5, 1, 0, 0, 0, 1, 0)


class Emu:
    """g++ build of the DEVICE headers with the single-lane executor (tests/host_emu): checks the device code's
    arithmetic and decisions on a machine without a GPU.  Never part of the product path."""

    def __init__(self):
        so = os.path.join(EMU_DIR, "libwbc_emu.so")
        _build_emu(os.path.join(EMU_DIR, "wbc_emu.cpp"), so)
        self.lib = C.CDLL(so)
        assert self.lib.emu_sizeof_params() == C.sizeof(EmuParams)
        so2 = os.path.join(EMU_DIR, "libqp_emu.so")
        _build_emu(os.path.join(EMU_DIR, "qp_emu.cpp"), so2)
        self.qp = C.CDLL(so2)
        self.qp.emu_qp_solve.argtypes = [_dp, _dp, _dp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, _dp,
                                         _ip, _dp]

    def cycle(self, sc, params=None):
        P = params or emu_default_params()
        n = int(sc["mode"].shape[0])
        keep = []

        def p_(a):
            a = np.ascontiguousarray(a, dtype=np.float64)
            keep.append(a)
            return a.ctypes.data_as(_dp)
        io = _EmuIO()
        for k in IN_NAMES:
            setattr(io, k, p_(sc[k]))
        io.terrain = p_(sc["terrain"]) if sc.get("terrain") is not None else None
        mode = np.ascontiguousarray(sc["mode"], dtype=np.int32)
        io.mode = mode.ctypes.data_as(_ip)
        io.ld = n
        out = dict(yd=np.array(sc["obs_yd"], dtype=np.float64, order="C"), yw=np.array(sc["obs_yw"], dtype=np.float64, order="C"),
                   tau=np.zeros((12, n)), w=np.zeros((6, n)), x=np.zeros((30, n)), qp_obj=np.zeros(n),
                   status=np.zeros(n, dtype=np.int32), qp_info=np.zeros((8, n), dtype=np.int32),
                   rec=np.zeros((n, self.lib.emu_qprec_doubles())),
                   yg=np.array(sc.get("obs_yg", np.zeros((6, n))), dtype=np.float64, order="C"), w3=np.zeros((12, n)))
        io.yd, io.yw = out["yd"].ctypes.data_as(_dp), out["yw"].ctypes.data_as(_dp)
        io.yg, io.w3 = out["yg"].ctypes.data_as(_dp), out["w3"].ctypes.data_as(_dp)
        io.tau, io.w, io.x = out["tau"].ctypes.data_as(_dp), out["w"].ctypes.data_as(_dp), out["x"].ctypes.data_as(_dp)
        io.qp_obj, io.status, io.info = out["qp_obj"].ctypes.data_as(_dp), out["status"].ctypes.data_as(_ip), out["qp_info"].ctypes.data_as(_ip)
        io.rec = out["rec"].ctypes.data_as(_dp)
        self.lib.emu_cycle(C.byref(P), C.byref(io), n)
        return out

    def fdyn_step(self, sc, tau, push, nsub=5, gamma=100.0, params=None):
        """The device code's forward-dynamics plant step on the host; returns (next-state dict, diag [2, n])."""
        P = params or emu_default_params()
        n = int(sc["mode"].shape[0])
        st = {k: np.array(sc[k], dtype=np.float64, order="C") for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq")}
        st["foot_force"] = np.zeros((12, n))
        mode = np.ascontiguousarray(sc["mode"], dtype=np.int32)
        tau = np.ascontiguousarray(tau, dtype=np.float64); push = np.ascontiguousarray(push, dtype=np.float64)
        diag = np.zeros((2, n))
        self.lib.emu_fdyn_step.argtypes = [C.POINTER(EmuParams), C.c_int, C.c_long] + [_dp] * 7 + [_ip, _dp, _dp, _dp, C.c_int, C.c_double]
        self.lib.emu_fdyn_step.restype = None
        d = lambda a: a.ctypes.data_as(_dp)
        self.lib.emu_fdyn_step(C.byref(P), n, n, d(st["base_pos"]), d(st["base_rot"]), d(st["base_rpy"]), d(st["base_vel"]), d(st["q"]), d(st["dq"]),
                               d(st["foot_force"]), mode.ctypes.data_as(_ip), d(tau), d(push), d(diag), int(nsub), float(gamma))
        return st, diag

    def sample_trajectory(self, traj, t):
        dur = np.ascontiguousarray(traj["durations"], dtype=np.float64)
        nodes = np.ascontiguousarray(traj["nodes"], dtype=np.float64)
        t = np.ascontiguousarray(t, dtype=np.float64)
        n = dur.shape[1]
        out = np.zeros((36, n))
        self.lib.emu_sample_trajectory.argtypes = [C.c_int, C.c_int, _dp, _dp, C.c_long, _dp, _dp]
        self.lib.emu_sample_trajectory.restype = None
        self.lib.emu_sample_trajectory(n, int(traj["nseg"]), dur.ctypes.data_as(_dp), nodes.ctypes.data_as(_dp), n, t.ctypes.data_as(_dp),
                                       out.ctypes.data_as(_dp))
        names = ["com_des_pos", "com_des_vel", "com_des_acc", "sw_des_pos", "sw_des_vel", "sw_des_acc"]
        return {k: out[6 * b:6 * b + 6] for b, k in enumerate(names)}

    def qp_solve(self, Q, c, L, neq, epsx=1e-2, rho=1e4, outerits=5, kkt_mode=1):
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        c = np.ascontiguousarray(c, dtype=np.float64)
        L = np.ascontiguousarray(L, dtype=np.float64)
        x = np.zeros(30)
        ist = (C.c_int * 8)()
        ds = (C.c_double * 2)()
        self.qp.emu_qp_solve(Q.ctypes.data_as(_dp), c.ctypes.data_as(_dp), L.ctypes.data_as(_dp), L.shape[0], int(neq),
                             epsx, rho, outerits, kkt_mode, x.ctypes.data_as(_dp), ist, ds)
        return x, list(ist), ds[0]

    def oracle_qp_fn(self):
        """The solver restatement as the oracle's QP solver (emu_qp_solve_oracle: reference settings, literal multiplier update),
        a C function the oracle calls from all its threads.  Its parity with the reference ALGLIB is pinned by
        tests/golden/qp_*.npz (test_emulation.py)."""
        return self.qp.emu_qp_solve_oracle


def check_cycle_parity(got, ref, n=None, what=""):
    """got: dict of SoA [k, n] arrays from the CUDA path / emulation; ref: oracle dict of [n, k] arrays."""
    tau, w = got["tau"].T, got["w"].T
    et = rel_rows(tau, ref["tau"])
    assert et.max() <= TOL_TAU, "%s torque parity: worst rel err %.3e at instance %d" % (what, et.max(), int(et.argmax()))
    ew = np.abs(w - ref["w"]).max()
    assert ew <= TOL_OBS * max(1.0, np.abs(ref["w"]).max()), "%s observer parity: %.3e" % (what, ew)
    if "qp_obj" in got:
        eo = np.abs(got["qp_obj"] - ref["qp_obj"]) / np.maximum(1e-30, np.abs(ref["qp_obj"]))
        assert eo.max() <= TOL_OBJ, "%s QP objective parity: %.3e at %d" % (what, eo.max(), int(eo.argmax()))
    if "status" in got:
        assert (got["status"] == 0).all(), "%s: solver failure flagged" % what
    return et.max()
