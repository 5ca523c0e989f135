"""Host-side mirror of the reference controller's per-cycle interface, on top of the C ABI.

    reference (dogbot_controller/src)                         here
    --------------------------------------------------------  ----------------------------------------
    DOGCTRL::update(...) + estimate() + QP + tau              WbcBatch.cycle(inputs) -> tau, w, x, ...
        client/main.cpp:572-660, 692-725, 984-1127, 1163-1397
    OPT(30, 86, 82); setQ; setc; setL_stance; opt_stance      OPT(...).setQ(...).setc(...).setL_stance(...).opt_stance()
        lopt.h:5-36, lopt.cpp:4-154

Everything numeric happens inside libwbc_b200.so (hand-written sm_100a CUDA behind include/wbc_b200.h).
This module only marshals pointers: numpy arrays for host buffers, torch CUDA tensors (or raw device
pointers) for device-resident buffers.  There is no CPU fallback: loading fails loudly when the
library is missing, and every call fails when no B200-class GPU is present.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

MODE_STANCE, MODE_SWING_BR_FL, MODE_SWING_BL_FR = 0, 1, 2
HOST_PTRS, DEVICE_PTRS, NO_SYNC, FIFO_DISPATCH, HOST_SLAB, SAMPLED_TRAJ, QP_EXACT, QP_WARM = 0, 1, 2, 4, 8, 16, 32, 64
FL_WARM_STARTED = 2048       # qp_info[5] of an instance that a WBC_QP_WARM cycle started from its stored active set
ST_BAD_MODE, ST_NONFINITE, ST_INFEASIBLE, ST_NOT_PD = -20, -21, -22, -23
SOLVER_KERNELS = {0: "wbc_solve_kernel", 1: "wbc_solve_staged_kernel", 2: "wbc_solve_exact_kernel"}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)

IN_FIELDS = [("base_pos", 3), ("base_rot", 9), ("base_rpy", 3), ("base_vel", 6), ("q", 12), ("dq", 12),
             ("com_des_pos", 6), ("com_des_vel", 6), ("com_des_acc", 6),
             ("sw_des_pos", 6), ("sw_des_vel", 6), ("sw_des_acc", 6), ("foot_force", 12), ("terrain", 40)]
OUT_FIELDS = [("tau", 12), ("w", 6), ("x", 30), ("qp_obj", 1)]
DEBUG_FIELDS = [("M", 324), ("h", 18), ("g", 18), ("Jac_lin", 216), ("Jdqd_lin", 12), ("com", 3), ("com_vel", 3),
                ("Mcom_b", 36), ("Mcom_j", 144), ("hcom", 18), ("gcom", 18), ("Jcom_lin", 216), ("Jdqdcom_lin", 12),
                ("foot_pos", 12), ("foot_vel", 12), ("Fgrf", 12), ("Wcom_des", 6)]


class Params(C.Structure):
    _fields_ = [(n, C.c_double) for n in
                ("kcom", "dcom", "q1_weight", "slack_weight", "mu", "tau_max", "joint_dt", "kp_sw", "kd_sw", "g_acc",
                 "obs_gain", "obs_dt")] + [("gravity", C.c_double * 3), ("qp_epsx", C.c_double), ("qp_rho", C.c_double),
                                           ("obs_gain2", C.c_double),
                                           ("qp_outerits", C.c_int), ("observer_enabled", C.c_int),
                                           ("fix_swing_rhs", C.c_int), ("qp_literal_kkt", C.c_int),
                                           ("hold_tau_on_failure", C.c_int), ("obs_order", C.c_int), ("obs_form", C.c_int)]


class _Inputs(C.Structure):
    _fields_ = [(n, C.c_void_p) for n, _ in IN_FIELDS] + [("mode", C.c_void_p), ("ld", C.c_long), ("obs_gain", C.c_void_p)]


class _Outputs(C.Structure):
    _fields_ = [("tau", C.c_void_p), ("w", C.c_void_p), ("x", C.c_void_p), ("qp_obj", C.c_void_p), ("status", C.c_void_p),
                ("qp_info", C.c_void_p), ("qp_flops", C.c_void_p), ("ld", C.c_long), ("w3", C.c_void_p)]


class _Debug(C.Structure):
    _fields_ = [(n, C.c_void_p) for n, _ in DEBUG_FIELDS] + [("ld", C.c_long)]


class _PlantState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq", "foot_force", "mode")]


class ContactParams(C.Structure):
    """wbc_contact_params: Baumgarte factor, Delassus regularisation, candidate margin (m), dual steps per contact QP."""
    _fields_ = [("beta", C.c_double), ("eps", C.c_double), ("margin", C.c_double), ("max_iter", C.c_int)]


CONTACT_NONE, CONTACT_STICK, CONTACT_SLIDE = 0, 1, 2


class _Trajectory(C.Structure):
    _fields_ = [("nseg", C.c_int), ("durations", C.c_void_p), ("nodes", C.c_void_p), ("ld", C.c_long)]


TRAJ_FIELDS = ["com_des_pos", "com_des_vel", "com_des_acc", "sw_des_pos", "sw_des_vel", "sw_des_acc"]


class _TrajSamples(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in TRAJ_FIELDS] + [("ld", C.c_long)]


class GaitParams(C.Structure):
    """wbc_gait_params: phase lengths (control cycles), foot lift (m), touchdown-target velocity gain (s) and step limit (m), command
    ramp limits (m/s^2, rad/s^2), leash of the CoM reference (m)."""
    _fields_ = [("stance_cycles", C.c_int), ("swing_cycles", C.c_int)] + \
               [(n, C.c_double) for n in ("step_height", "k_v", "max_step", "acc_lin", "acc_yaw", "leash")]


GAIT_INT_FIELDS = [("phase", 1), ("tick", 1), ("landed", 1)]
GAIT_FIELDS = [("com_ref", 4), ("v_ref", 3), ("liftoff", 6), ("target", 6), ("offset", 8)]


class _GaitState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n, _ in GAIT_INT_FIELDS + GAIT_FIELDS]


class WbcError(RuntimeError):
    pass


_lib = None

EXPORTS = ["wbc_default_params", "wbc_last_error", "wbc_version", "wbc_create", "wbc_destroy", "wbc_set_params",
           "wbc_set_observer_state", "wbc_get_observer_state", "wbc_set_observer_state2", "wbc_get_observer_state2", "wbc_cycle", "wbc_debug_update", "wbc_debug_qp_records", "wbc_qp_solve",
           "wbc_qp_solve_warm", "wbc_set_active_set", "wbc_get_active_set",
           "wbc_plant_step", "wbc_plant_dynamics_step", "wbc_default_contact_params", "wbc_plant_contact_step", "wbc_plant_contact_step_terrain", "wbc_last_timing", "wbc_last_solve_cycles", "wbc_last_launches", "wbc_solver_shape", "wbc_stage_profile", "wbc_host_alloc",
           "wbc_host_free",
           "wbc_set_trajectory", "wbc_sample_trajectory",
           "wbc_default_gait_params", "wbc_gait_init", "wbc_gait_step",
           "wbc_measure_dfma_peak"]


def lib_path():
    return _build.LIB


def load():
    """dlopen libwbc_b200.so (building it in-tree first if a compiler is at hand).  Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("WBC_B200_LIB") or _build.LIB          # A/B experiments: a variant build of the same library
    if path == _build.LIB:
        # rebuild when the library is missing or older than its sources (a no-op otherwise); on a box without nvcc the
        # shipped library is used as it is, and a missing one is an error: there is no CPU fallback
        if _build.have_nvcc() or not os.path.exists(_build.LIB):
            _build.build()
    lib = C.CDLL(path)
    lib.wbc_default_params.argtypes = [C.POINTER(Params)]
    lib.wbc_last_error.restype = C.c_char_p
    lib.wbc_version.restype = C.c_char_p
    lib.wbc_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.POINTER(Params)]
    lib.wbc_destroy.argtypes = [C.c_void_p]
    lib.wbc_set_params.argtypes = [C.c_void_p, C.POINTER(Params)]
    lib.wbc_set_observer_state.argtypes = [C.c_void_p, C.c_int, _dp, _dp, C.c_long]
    lib.wbc_get_observer_state.argtypes = [C.c_void_p, C.c_int, _dp, _dp, C.c_long]
    lib.wbc_debug_qp_records.argtypes = [C.c_void_p, C.c_int, _dp, C.POINTER(C.c_int)]
    lib.wbc_set_observer_state2.argtypes = [C.c_void_p, C.c_int, _dp, C.c_long]
    lib.wbc_get_observer_state2.argtypes = [C.c_void_p, C.c_int, _dp, C.c_long]
    lib.wbc_cycle.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Inputs), C.POINTER(_Outputs), C.c_void_p, C.c_uint]
    lib.wbc_debug_update.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Inputs), C.POINTER(_Debug), C.c_uint]
    lib.wbc_qp_solve.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
    lib.wbc_qp_solve_warm.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
    lib.wbc_set_active_set.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_long]
    lib.wbc_get_active_set.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_long]
    lib.wbc_plant_step.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_void_p,
                                   C.c_uint]
    lib.wbc_plant_dynamics_step.argtypes = [C.c_void_p, C.c_int, C.POINTER(_PlantState), C.c_void_p, C.c_void_p, C.c_long, C.c_int, C.c_double,
                                            C.c_void_p, C.c_void_p, C.c_uint]
    lib.wbc_default_contact_params.argtypes = [C.POINTER(ContactParams)]
    lib.wbc_plant_contact_step.argtypes = [C.c_void_p, C.c_int, C.POINTER(_PlantState), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long,
                                           C.c_int, C.POINTER(ContactParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint]
    lib.wbc_plant_contact_step_terrain.argtypes = lib.wbc_plant_contact_step.argtypes
    lib.wbc_last_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    lib.wbc_last_solve_cycles.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_ulonglong)]
    lib.wbc_last_launches.argtypes = [C.c_void_p]
    lib.wbc_solver_shape.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.wbc_stage_profile.argtypes = [C.c_void_p, C.POINTER(C.c_ulonglong), C.c_int]
    lib.wbc_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    lib.wbc_host_free.argtypes = [C.c_void_p]
    lib.wbc_set_trajectory.argtypes = [C.c_void_p, C.c_int, C.POINTER(_Trajectory), C.c_void_p, C.c_uint]
    lib.wbc_sample_trajectory.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.POINTER(_TrajSamples), C.c_void_p, C.c_uint]
    lib.wbc_default_gait_params.argtypes = [C.POINTER(GaitParams)]
    lib.wbc_gait_init.argtypes = [C.c_void_p, C.c_int, C.POINTER(GaitParams), C.POINTER(_PlantState), C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.POINTER(_GaitState), C.c_void_p, C.c_long, C.c_void_p, C.c_uint]
    lib.wbc_gait_step.argtypes = [C.c_void_p, C.c_int, C.POINTER(GaitParams), C.POINTER(_GaitState), C.POINTER(_PlantState), C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(_TrajSamples), C.c_void_p, C.c_long, C.c_void_p,
                                  C.c_uint]
    lib.wbc_measure_dfma_peak.argtypes = [C.c_void_p, _dp]
    _lib = lib
    return lib


def default_params():
    p = Params()
    load().wbc_default_params(C.byref(p))
    return p


def default_contact_params():
    cp = ContactParams()
    load().wbc_default_contact_params(C.byref(cp))
    return cp


def default_gait_params():
    gp = GaitParams()
    load().wbc_default_gait_params(C.byref(gp))
    return gp


def _warm_needs_exact(warm, exact):
    if warm and not exact:
        raise WbcError("warm start (WBC_QP_WARM) is only available with the exact solver: pass exact=True as well")


def _check(rc, what):
    if rc != 0:
        raise WbcError("%s failed (%d): %s" % (what, rc, load().wbc_last_error().decode()))


def _ptr(a):
    """numpy array -> host pointer; torch tensor -> data_ptr(); int -> itself; None -> NULL."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    return int(a)


class WbcBatch:
    """One ctx = one GPU.  Holds the per-instance observer state across cycles (main.cpp:243, 721-724)."""

    def __init__(self, max_batch, device=0, params=None):
        self.lib = load()
        self.params = params or default_params()
        self.max_batch = int(max_batch)
        self.device = int(device)
        h = C.c_void_p()
        _check(self.lib.wbc_create(C.byref(h), self.device, self.max_batch, C.byref(self.params)), "wbc_create")
        self.h = h
        self._pinned = []
        self.fifo_dispatch = False      # True: WBC_FIFO_DISPATCH (index-order work queue instead of longest-first)

    def close(self):
        if getattr(self, "h", None):
            self.lib.wbc_destroy(self.h)
            self.h = None
        for p in getattr(self, "_pinned", []):
            self.lib.wbc_host_free(p)
        self._pinned = []

    __del__ = close

    def set_params(self, params):
        self.params = params
        _check(self.lib.wbc_set_params(self.h, C.byref(params)), "wbc_set_params")

    def set_observer_state(self, yd, yw):
        yd = np.ascontiguousarray(yd, dtype=np.float64)
        yw = np.ascontiguousarray(yw, dtype=np.float64)
        n = yd.shape[1]
        _check(self.lib.wbc_set_observer_state(self.h, n, yd.ctypes.data_as(_dp), yw.ctypes.data_as(_dp), n),
               "wbc_set_observer_state")

    def get_observer_state(self, n):
        yd, yw = np.zeros((6, n)), np.zeros((6, n))
        _check(self.lib.wbc_get_observer_state(self.h, n, yd.ctypes.data_as(_dp), yw.ctypes.data_as(_dp), n),
               "wbc_get_observer_state")
        return yd, yw

    def set_observer_state2(self, yg):
        """ygamma, the extra integrator of the second-order observer (params.obs_order == 2)."""
        yg = np.ascontiguousarray(yg, dtype=np.float64)
        n = yg.shape[1]
        _check(self.lib.wbc_set_observer_state2(self.h, n, yg.ctypes.data_as(_dp), n), "wbc_set_observer_state2")

    def get_observer_state2(self, n):
        yg = np.zeros((6, n))
        _check(self.lib.wbc_get_observer_state2(self.h, n, yg.ctypes.data_as(_dp), n), "wbc_get_observer_state2")
        return yg

    def set_active_set(self, sets):
        """The exact-mode active sets stored per instance index, uint32 [4, n] (rows 0..2 bit masks of the active inequality rows,
        row 3 the contact mode + 1, 0 = none): restore them with the observer state after a checkpoint or a re-sharding."""
        sets = np.ascontiguousarray(sets, dtype=np.uint32)
        n = sets.shape[1]
        _check(self.lib.wbc_set_active_set(self.h, n, sets.ctypes.data, n), "wbc_set_active_set")

    def get_active_set(self, n):
        sets = np.zeros((4, n), dtype=np.uint32)
        _check(self.lib.wbc_get_active_set(self.h, n, sets.ctypes.data, n), "wbc_get_active_set")
        return sets

    @staticmethod
    def _inputs_struct(sc, n, keep, skip=()):
        ins = _Inputs()
        ld = None
        for name, k in IN_FIELDS:
            a = None if name in skip else sc.get(name)
            if a is None:
                if name != "terrain" and name not in skip:
                    raise WbcError("missing input array '%s'" % name)
                setattr(ins, name, None)
                continue
            if isinstance(a, np.ndarray):
                a = np.ascontiguousarray(a, dtype=np.float64)
                keep.append(a)
            if tuple(a.shape)[0] != k:
                raise WbcError("input '%s' must have shape [%d, ld]" % (name, k))
            ld = int(a.shape[1]) if ld is None else ld
            if int(a.shape[1]) != ld:
                raise WbcError("all inputs must share the same leading dimension")
            setattr(ins, name, _ptr(a))
        m = sc["mode"]
        if isinstance(m, np.ndarray):
            m = np.ascontiguousarray(m, dtype=np.int32)
            keep.append(m)
        ins.mode = _ptr(m)
        ins.ld = ld
        g = sc.get("obs_gain")                       # optional per-instance observer gain [n] (config 5's sweep)
        if g is not None:
            g = np.ascontiguousarray(g, dtype=np.float64).reshape(-1)
            if g.shape[0] != ld:
                raise WbcError("obs_gain must have one entry per instance")
            keep.append(g)
        ins.obs_gain = _ptr(g)
        if n > ld:
            raise WbcError("n exceeds the arrays' leading dimension")
        return ins

    def pinned(self, shape, dtype=np.float64):
        """A numpy array in page-locked host memory (wbc_host_alloc): wbc_cycle copies such arrays to / from the device
        directly instead of through its bounce buffer.  Freed with the batch."""
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _check(self.lib.wbc_host_alloc(C.byref(p), max(nbytes, 8)), "wbc_host_alloc")
        self._pinned.append(p)
        buf = (C.c_char * max(nbytes, 8)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def pinned_copy(self, a):
        out = self.pinned(a.shape, a.dtype)
        out[...] = a
        return out

    def set_trajectory(self, traj):
        """Upload a plan (scenarios.make_trajectory layout: nseg, durations [4*nseg, n], nodes [4*(nseg+1)*6, n])."""
        d = np.ascontiguousarray(traj["durations"], dtype=np.float64)
        nd = np.ascontiguousarray(traj["nodes"], dtype=np.float64)
        n = d.shape[1]
        tr = _Trajectory(int(traj["nseg"]), d.ctypes.data, nd.ctypes.data, n)
        _check(self.lib.wbc_set_trajectory(self.h, n, C.byref(tr), None, HOST_PTRS), "wbc_set_trajectory")

    def sample_trajectory(self, n, t=None, t_all=0.0, fetch=False):
        """Sample the uploaded plan on the GPU at per-instance times t [n] (or t_all for everyone).  The samples stay on
        the device for cycle(..., sampled_traj=True); fetch=True also returns them as a dict of [6, n] host arrays."""
        tp = None
        if t is not None:
            t = np.ascontiguousarray(t, dtype=np.float64)
            tp = t.ctypes.data
        _check(self.lib.wbc_sample_trajectory(self.h, n, tp, float(t_all), None, None, HOST_PTRS), "wbc_sample_trajectory")
        if not fetch:
            return None
        out = {k: np.zeros((6, n)) for k in TRAJ_FIELDS}
        o = _TrajSamples(*[out[k].ctypes.data for k in TRAJ_FIELDS], n)
        _check(self.lib.wbc_sample_trajectory(self.h, n, tp, float(t_all), C.byref(o), None, HOST_PTRS), "wbc_sample_trajectory")
        return out

    def pinned_inputs(self, sc):
        """Copy a scenario's input arrays into ONE page-locked slab laid out in wbc_inputs field order, so that
        wbc_cycle moves them with a single host-to-device copy.  Returns a dict of views (other keys passed through)."""
        n = int(sc["mode"].shape[0])
        fields = [(name, k) for name, k in IN_FIELDS if sc.get(name) is not None]
        rows = sum(k for _, k in fields) + (1 if sc.get("obs_gain") is not None else 0)
        slab = self.pinned((rows, n))
        out, r = dict(sc), 0
        for name, k in fields:
            out[name] = slab[r:r + k]
            out[name][...] = sc[name]
            r += k
        if sc.get("obs_gain") is not None:
            out["obs_gain"] = slab[r]
            out["obs_gain"][...] = sc["obs_gain"]
        out["mode"] = self.pinned_copy(np.ascontiguousarray(sc["mode"], dtype=np.int32))
        out["_slab"] = True          # cycle() passes WBC_HOST_SLAB
        return out

    def cycle(self, sc, n=None, want=("x", "qp_obj", "status", "qp_info", "qp_flops"), out=None, sampled_traj=False, exact=False,
              warm=False):
        """One control cycle on HOST (numpy) SoA inputs; returns a dict of numpy arrays [k, n].  `out`: preallocated
        result arrays to fill (e.g. page-locked ones from pinned()); its keys decide what is returned.  exact=True: solve each
        QP to its exact optimum (WBC_QP_EXACT, the dual active-set solver) instead of DENSE-AUL at the reference's settings.
        warm=True (needs exact=True): start each instance from the active set of its previous exact-mode cycle (WBC_QP_WARM)."""
        _warm_needs_exact(warm, exact)
        keep = []
        n = int(sc["mode"].shape[0]) if n is None else int(n)
        ins = self._inputs_struct(sc, n, keep, skip=TRAJ_FIELDS if sampled_traj else ())
        if out is None:
            out = {"tau": np.zeros((12, n)), "w": np.zeros((6, n))}
            if "x" in want: out["x"] = np.zeros((30, n))
            if "qp_obj" in want: out["qp_obj"] = np.zeros(n)
            if "status" in want: out["status"] = np.zeros(n, dtype=np.int32)
            if "qp_info" in want: out["qp_info"] = np.zeros((8, n), dtype=np.int32)
            if "qp_flops" in want: out["qp_flops"] = np.zeros(n)
            if "w3" in want: out["w3"] = np.zeros((12, n))
        o = _Outputs()
        for k in ("tau", "w", "x", "qp_obj", "status", "qp_info", "qp_flops", "w3"):
            setattr(o, k, _ptr(out.get(k)))
        o.ld = max(n, 1)
        _check(self.lib.wbc_cycle(self.h, n, C.byref(ins), C.byref(o), None, HOST_PTRS | (FIFO_DISPATCH if self.fifo_dispatch else 0) | (HOST_SLAB if sc.get("_slab") else 0) | (SAMPLED_TRAJ if sampled_traj else 0) | (QP_EXACT if exact else 0) | (QP_WARM if warm else 0)), "wbc_cycle")
        return out

    def cycle_device(self, dev_in, dev_out, n, ld, stream=None, sync=True, out_ld=None, exact=False, warm=False):
        """One control cycle on DEVICE-resident SoA buffers (dicts of torch CUDA tensors or raw pointers).
        `ld` is the leading dimension of the input arrays, `out_ld` that of the output arrays (default: the outputs' own
        second dimension when they are tensors, else `ld`).  exact, warm: as in cycle()."""
        _warm_needs_exact(warm, exact)
        if out_ld is None:
            t = dev_out.get("tau")
            out_ld = int(t.stride(0)) if hasattr(t, "stride") and t.dim() == 2 else ld
        # element (k, i) of an array is read or written at k * ld + i: refuse tensors whose row stride is not the leading
        # dimension they are passed with, or that are narrower than the batch (out-of-bounds accesses otherwise)
        for d, want_ld in ((dev_in, ld), (dev_out, out_ld)):
            for k, v in d.items():
                if hasattr(v, "stride") and hasattr(v, "dim"):
                    if v.dim() == 2 and (int(v.shape[1]) < n or (int(v.shape[0]) > 1 and int(v.stride(0)) != want_ld)):
                        raise WbcError("cycle_device: array %r has shape %s / row stride %d, expected >= %d columns and leading dimension %d"
                                       % (k, tuple(v.shape), int(v.stride(0)), n, want_ld))
                    if v.dim() == 1 and int(v.shape[0]) < n:
                        raise WbcError("cycle_device: array %r has %d entries, batch is %d" % (k, int(v.shape[0]), n))
        ins = _Inputs()
        for name, _ in IN_FIELDS:
            setattr(ins, name, _ptr(dev_in.get(name)))
        ins.mode = _ptr(dev_in["mode"])
        ins.obs_gain = _ptr(dev_in.get("obs_gain"))
        ins.ld = ld
        o = _Outputs()
        for k in ("tau", "w", "x", "qp_obj", "status", "qp_info", "qp_flops", "w3"):
            setattr(o, k, _ptr(dev_out.get(k)))
        o.ld = out_ld
        flags = DEVICE_PTRS | (0 if sync else NO_SYNC) | (FIFO_DISPATCH if self.fifo_dispatch else 0) | (QP_EXACT if exact else 0) | (QP_WARM if warm else 0)
        _check(self.lib.wbc_cycle(self.h, n, C.byref(ins), C.byref(o), stream, flags), "wbc_cycle")

    def qp_records(self, n):
        """The QP records of the last cycle [n, doubles per record] (wbc_debug_qp_records; validation only)."""
        k = C.c_int(0)
        _check(self.lib.wbc_debug_qp_records(self.h, 0, None, C.byref(k)), "wbc_debug_qp_records")
        out = np.zeros((n, k.value))
        _check(self.lib.wbc_debug_qp_records(self.h, n, out.ctypes.data_as(_dp), None), "wbc_debug_qp_records")
        return out

    def debug_update(self, sc, n=None):
        """update() intermediates (wbc_debug_update) for stage-by-stage validation."""
        keep = []
        n = int(sc["mode"].shape[0]) if n is None else int(n)
        ins = self._inputs_struct(sc, n, keep)
        d = _Debug()
        out = {}
        for name, k in DEBUG_FIELDS:
            out[name] = np.zeros((k, n))
            setattr(d, name, out[name].ctypes.data)
        d.ld = n
        _check(self.lib.wbc_debug_update(self.h, n, C.byref(ins), C.byref(d), HOST_PTRS), "wbc_debug_update")
        return out

    def qp_solve(self, Q, c, L, neq, exact=False, warm=False, active=None):
        """n dense QPs, instance-major numpy arrays Q [n,30,30], c [n,30], L [n,nrows,31] (the OPT operator).  exact=True: the
        exact-mode solver (WBC_QP_EXACT); info then holds its counters (include/wbc_b200.h).
        warm=True (needs exact=True; wbc_qp_solve_warm): `active` uint32 [n,3] is each instance's warm set (bit r of word r // 32:
        inequality row r; None or zeros: a cold start); returns (x, status, info, flops, active) with the final active sets."""
        _warm_needs_exact(warm, exact)
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        c = np.ascontiguousarray(c, dtype=np.float64)
        L = np.ascontiguousarray(L, dtype=np.float64)
        n, nrows = Q.shape[0], L.shape[1]
        x = np.zeros((n, 30))
        status = np.zeros(n, dtype=np.int32)
        info = np.zeros((n, 8), dtype=np.int32)
        flops = np.zeros(n)
        if warm:
            act = np.zeros((n, 3), np.uint32) if active is None else np.array(active, dtype=np.uint32).reshape(n, 3)
            _check(self.lib.wbc_qp_solve_warm(self.h, n, Q.ctypes.data, c.ctypes.data, L.ctypes.data, nrows, int(neq), x.ctypes.data,
                                              status.ctypes.data, info.ctypes.data, flops.ctypes.data, act.ctypes.data, None, HOST_PTRS),
                   "wbc_qp_solve_warm")
            return x, status, info, flops, act
        _check(self.lib.wbc_qp_solve(self.h, n, Q.ctypes.data, c.ctypes.data, L.ctypes.data, nrows, int(neq), x.ctypes.data,
                                     status.ctypes.data, info.ctypes.data, flops.ctypes.data, None, HOST_PTRS | (QP_EXACT if exact else 0)), "wbc_qp_solve")
        return x, status, info, flops

    def plant_step(self, base_pos, base_vel, push, foot_force=None, x=None, n=None, ld=None, stream=None, sync=True):
        """Synthetic plant of BASELINE config 5 (wbc_plant_step): advances base_pos [3,n] / base_vel [6,n] in place from the
        momentum balance of the last cycle and the world push wrench `push` [6,n]; with foot_force [12,n] and the last QP
        solution x [30,n] the loop is closed through the commanded ground-reaction forces.  numpy arrays (host), or torch
        CUDA tensors / raw device pointers (then pass n and ld)."""
        host = isinstance(base_vel, np.ndarray)
        if host:
            for a in (base_pos, base_vel, foot_force):
                assert a is None or (a.flags.c_contiguous and a.dtype == np.float64)
            n = int(base_vel.shape[1]); ld = n
            push = np.ascontiguousarray(push, dtype=np.float64)
            x = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
            flags = HOST_PTRS
        else:
            flags = DEVICE_PTRS | (0 if sync else NO_SYNC)
        _check(self.lib.wbc_plant_step(self.h, int(n), _ptr(base_pos), _ptr(base_vel), _ptr(foot_force), _ptr(x), _ptr(push), int(ld),
                                       stream, flags), "wbc_plant_step")

    def plant_dynamics_step(self, state, tau, push, n=None, ld=None, substeps=5, gamma=100.0, diag=None, stream=None, sync=True):
        """Forward-dynamics plant (wbc_plant_dynamics_step): `state` is a dict with base_pos, base_rot, base_rpy, base_vel, q, dq,
        foot_force, mode (numpy arrays: host path, advanced in place; torch CUDA tensors: device path)."""
        host = isinstance(state["q"], np.ndarray)
        n = int(state["mode"].shape[0]) if n is None else int(n)
        ld = n if ld is None else int(ld)
        ps = _PlantState()
        for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq", "foot_force", "mode"):
            setattr(ps, k, _ptr(state[k]))
        flags = (HOST_PTRS if host else DEVICE_PTRS) | (0 if (sync or host) else NO_SYNC)
        _check(self.lib.wbc_plant_dynamics_step(self.h, n, C.byref(ps), _ptr(tau), _ptr(push), ld, int(substeps), float(gamma), _ptr(diag), stream, flags),
               "wbc_plant_dynamics_step")

    def plant_contact_step(self, state, tau, push, ground_z=None, mu=None, n=None, ld=None, substeps=5, params=None, contact=None, diag=None,
                           status=None, stream=None, sync=True, terrain=None, plane_d=None):
        """Contact plant (wbc_plant_contact_step): unilateral, frictional foot contacts on per-foot ground planes.  `state` is a dict
        with base_pos, base_rot, base_rpy, base_vel, q, dq, foot_force (numpy arrays: host path, advanced in place; torch CUDA tensors:
        device path); its mode is not read.  ground_z [4, ld] (None: 0), mu [ld] (None: params.mu), params a ContactParams (None:
        the defaults); contact int32 [4, ld], diag [4, ld] and status int32 [ld] are filled when given.
        With terrain [40, ld] (the controller's per-foot frames n, t1, t2 and mu, as in `cycle`) and plane_d [4, ld] (None: 0), each
        foot stands on the plane n . p = d_k instead (wbc_plant_contact_step_terrain); ground_z and mu must then be None."""
        if terrain is None and plane_d is not None:
            raise ValueError("plant_contact_step: plane_d needs terrain")
        if terrain is not None and (ground_z is not None or mu is not None):
            raise ValueError("plant_contact_step: terrain replaces ground_z and mu; pass plane_d for the plane offsets")
        host = isinstance(state["q"], np.ndarray)
        n = int(state["q"].shape[1]) if n is None else int(n)
        ld = n if ld is None else int(ld)
        ps = _PlantState()
        for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q", "dq", "foot_force"):
            setattr(ps, k, _ptr(state[k]))
        ps.mode = _ptr(state.get("mode"))
        keep = []
        if host:
            for a in (state["base_pos"], state["base_rot"], state["base_rpy"], state["base_vel"], state["q"], state["dq"], state["foot_force"], diag):
                assert a is None or (a.flags.c_contiguous and a.dtype == np.float64)
            for a in (contact, status):
                assert a is None or (a.flags.c_contiguous and a.dtype == np.int32)
            tau, push = np.ascontiguousarray(tau, dtype=np.float64), np.ascontiguousarray(push, dtype=np.float64)
            ground_z = None if ground_z is None else np.ascontiguousarray(ground_z, dtype=np.float64)
            mu = None if mu is None else np.ascontiguousarray(mu, dtype=np.float64)
            terrain = None if terrain is None else np.ascontiguousarray(terrain, dtype=np.float64)
            plane_d = None if plane_d is None else np.ascontiguousarray(plane_d, dtype=np.float64)
            keep += [tau, push, ground_z, mu, terrain, plane_d]
        cp = params if params is not None else default_contact_params()
        flags = (HOST_PTRS if host else DEVICE_PTRS) | (0 if (sync or host) else NO_SYNC)
        if terrain is not None:
            _check(self.lib.wbc_plant_contact_step_terrain(self.h, n, C.byref(ps), _ptr(tau), _ptr(push), _ptr(terrain), _ptr(plane_d), ld,
                                                           int(substeps), C.byref(cp), _ptr(contact), _ptr(diag), _ptr(status), stream, flags),
                   "wbc_plant_contact_step_terrain")
            return
        _check(self.lib.wbc_plant_contact_step(self.h, n, C.byref(ps), _ptr(tau), _ptr(push), _ptr(ground_z), _ptr(mu), ld, int(substeps), C.byref(cp),
                                               _ptr(contact), _ptr(diag), _ptr(status), stream, flags), "wbc_plant_contact_step")

    @staticmethod
    def gait_state(n, device=None):
        """A zeroed gait state for n robots (wbc_gait_state): int32 phase, tick, landed [1, n] and float64 com_ref [4, n], v_ref [3, n],
        liftoff [6, n], target [6, n], offset [8, n]; numpy arrays, or torch tensors on `device` (e.g. "cuda:0")."""
        if device is None:
            st = {k: np.zeros((m, n), np.int32) for k, m in GAIT_INT_FIELDS}
            st.update({k: np.zeros((m, n)) for k, m in GAIT_FIELDS})
            return st
        import torch
        st = {k: torch.zeros(m, n, dtype=torch.int32, device=device) for k, m in GAIT_INT_FIELDS}
        st.update({k: torch.zeros(m, n, dtype=torch.float64, device=device) for k, m in GAIT_FIELDS})
        return st

    @staticmethod
    def _gait_structs(state, gs, others):
        """The plant-state and gait-state structs, and whether this is the host path (numpy state).  Every array -- state, gait state
        and the optional ones in `others` (name -> array or None) -- must live on the same side as state["q"]: numpy arrays on the host
        path, CUDA tensors (or raw device pointers) on the device path.  A pointer of the other side would reach the kernel as if it
        were of this one, so a mix is refused here."""
        host = isinstance(state["q"], np.ndarray)
        arrays = {k: state[k] for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q")}
        arrays.update({k: gs[k] for k, _ in GAIT_INT_FIELDS + GAIT_FIELDS})
        arrays.update({k: a for k, a in others.items() if a is not None})
        for k, a in arrays.items():
            on_host = isinstance(a, np.ndarray) or (hasattr(a, "is_cuda") and not a.is_cuda)
            if host != on_host:
                raise WbcError("gait: %r is %s memory but the state is %s memory: pass every array on the same side"
                               % (k, "host" if on_host else "device", "host" if host else "device"))
        ps = _PlantState()
        for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q"):
            setattr(ps, k, _ptr(state[k]))
        g = _GaitState()
        for k, _ in GAIT_INT_FIELDS + GAIT_FIELDS:
            setattr(g, k, _ptr(gs[k]))
        if host:
            for k in ("base_pos", "base_rot", "base_rpy", "base_vel", "q") + tuple(k for k, _ in GAIT_FIELDS):
                a = state[k] if k in state else gs[k]
                assert a.flags.c_contiguous and a.dtype == np.float64, k
            for k, _ in GAIT_INT_FIELDS:
                assert gs[k].flags.c_contiguous and gs[k].dtype == np.int32, k
        return ps, g, host

    @staticmethod
    def _host_in(a, dtype=np.float64):
        return None if a is None else (np.ascontiguousarray(a, dtype=dtype) if isinstance(a, np.ndarray) else a)

    def gait_init(self, state, gs, k0=None, terrain=None, plane_d=None, params=None, status=None, n=None, ld=None, stream=None, sync=True):
        """Capture the gait state `gs` (gait_state()) of the robots in `state` (a plant-state dict: base_pos, base_rot, base_rpy, base_vel,
        q) at start offsets k0 [n] (None: 0), on flat ground or on terrain [40, ld] / plane_d [4, ld] (wbc_gait_init).  numpy arrays: host
        path; torch CUDA tensors: device path."""
        ps, g, host = self._gait_structs(state, gs, {"k0": k0, "terrain": terrain, "plane_d": plane_d, "status": status})
        n = int(state["q"].shape[1]) if n is None else int(n)
        ld = n if ld is None else int(ld)
        k0, terrain, plane_d = self._host_in(k0, np.int32), self._host_in(terrain), self._host_in(plane_d)
        gp = params if params is not None else default_gait_params()
        flags = (HOST_PTRS if host else DEVICE_PTRS) | (0 if (sync or host) else NO_SYNC)
        _check(self.lib.wbc_gait_init(self.h, n, C.byref(gp), C.byref(ps), _ptr(k0), _ptr(terrain), _ptr(plane_d), C.byref(g), _ptr(status),
                                      ld, stream, flags), "wbc_gait_init")

    def gait_step(self, state, gs, cmd=None, contact=None, terrain=None, plane_d=None, out=None, params=None, status=None, n=None, ld=None,
                  stream=None, sync=True):
        """One gait step (wbc_gait_step): advances `gs` and writes the contact mode and the six desired arrays into `out`, a dict with
        "mode" [ld] (int32) and com_des_pos, com_des_vel, com_des_acc, sw_des_pos, sw_des_vel, sw_des_acc [6, ld] -- e.g. the input
        dict handed to cycle_device, so the controller reads them directly.  cmd [3, ld]
        (vx, vy in the heading frame, yaw rate; None: trot in place), contact [4, ld] int32 (the contact plant's flags of the previous
        step; None: no touchdown).  Every array must be on the same side as state["q"] (numpy: host path, CUDA tensors: device
        path).  out=None allocates the outputs there.  Returns `out`."""
        n = int(state["q"].shape[1]) if n is None else int(n)
        ld = n if ld is None else int(ld)
        if out is None:
            if isinstance(state["q"], np.ndarray):
                out = {"mode": np.zeros(ld, np.int32)}
                out.update({k: np.zeros((6, ld)) for k in TRAJ_FIELDS})
            else:
                import torch
                dev = state["q"].device
                out = {"mode": torch.zeros(ld, dtype=torch.int32, device=dev)}
                out.update({k: torch.zeros(6, ld, dtype=torch.float64, device=dev) for k in TRAJ_FIELDS})
        ps, g, host = self._gait_structs(state, gs, {"cmd": cmd, "contact": contact, "terrain": terrain, "plane_d": plane_d, "status": status,
                                                     "mode": out["mode"], **{k: out[k] for k in TRAJ_FIELDS}})
        cmd, terrain, plane_d, contact = self._host_in(cmd), self._host_in(terrain), self._host_in(plane_d), self._host_in(contact, np.int32)
        t = out[TRAJ_FIELDS[0]]
        out_ld = int(t.strides[0] // 8) if isinstance(t, np.ndarray) else (int(t.stride(0)) if hasattr(t, "stride") else ld)
        o = _TrajSamples(*[_ptr(out[k]) for k in TRAJ_FIELDS], out_ld)
        gp = params if params is not None else default_gait_params()
        flags = (HOST_PTRS if host else DEVICE_PTRS) | (0 if (sync or host) else NO_SYNC)
        _check(self.lib.wbc_gait_step(self.h, n, C.byref(gp), C.byref(g), C.byref(ps), _ptr(cmd), _ptr(contact), _ptr(terrain), _ptr(plane_d),
                                      _ptr(out["mode"]), C.byref(o), _ptr(status), ld, stream, flags), "wbc_gait_step")
        return out

    def last_timing(self):
        a, b = C.c_float(0), C.c_float(0)
        _check(self.lib.wbc_last_timing(self.h, C.byref(a), C.byref(b)), "wbc_last_timing")
        return a.value, b.value

    def last_solve_cycles(self, n):
        """Per-instance solve duration of the last cycle in SM clock cycles (numpy uint64 [n])."""
        out = np.zeros(n, dtype=np.uint64)
        _check(self.lib.wbc_last_solve_cycles(self.h, n, out.ctypes.data_as(C.POINTER(C.c_ulonglong))), "wbc_last_solve_cycles")
        return out

    def last_launches(self):
        return int(self.lib.wbc_last_launches(self.h))

    def solver_shape(self):
        """(resident solver CTAs per SM, shared-memory bytes per CTA, grid of the last cycle) of the persistent solver kernel the
        last cycle ran; its name is left in last_solver_kernel."""
        a, b, g, st = C.c_int(0), C.c_int(0), C.c_int(0), C.c_int(0)
        _check(self.lib.wbc_solver_shape(self.h, C.byref(a), C.byref(b), C.byref(g), C.byref(st)), "wbc_solver_shape")
        self.last_solver_kernel = SOLVER_KERNELS[st.value]
        return a.value, b.value, g.value

    def stage_profile(self):
        """Per-warp counters of the last staged solver launch (ctx created with WBC_STAGE_PROF=1): array [warps, 12]."""
        _, _, g = self.solver_shape()
        a = np.zeros((g, 12), dtype=np.uint64)
        rows = self.lib.wbc_stage_profile(self.h, a.ctypes.data_as(C.POINTER(C.c_ulonglong)), g)
        _check(min(rows, 0), "wbc_stage_profile")
        return a[:rows]

    def measure_dfma_peak(self):
        v = C.c_double(0)
        _check(self.lib.wbc_measure_dfma_peak(self.h, C.byref(v)), "wbc_measure_dfma_peak")
        return v.value


class OPT:
    """Mirror of the reference's OPT class (lopt.h:5-36): same method names and argument meaning, one QP per call.

    OPT(30, 86, 82) as constructed at main.cpp:266.  setQ / setc / setL_stance / setL_swing take dense arrays
    (the reference takes Eigen matrices by value); opt_stance / opt_swing return x (the reference fills a
    caller-allocated VectorXd and silently leaves it untouched on failure, lopt.cpp:114-116 -- here a failure
    raises WbcError instead).
    """

    def __init__(self, control_variables=30, stance_constraint=86, swing_constraint=82, batch=None, exact=False, warm_start=False):
        """exact=True: solve to the exact optimum (WBC_QP_EXACT) instead of DENSE-AUL at the reference's settings.
        warm_start=True (needs exact=True): opt_stance and opt_swing each start from the active set of their own previous solve
        (wbc_qp_solve_warm), which a control loop that solves almost the same QP every cycle gains from."""
        _warm_needs_exact(warm_start, exact)
        if control_variables != 30 or stance_constraint != 86 or swing_constraint != 82:
            raise WbcError("OPT is specialised to the controller's shapes OPT(30, 86, 82) (main.cpp:266)")
        self._own = batch is None
        self._b = batch or WbcBatch(1)
        self._Q = self._c = self._Ls = self._Lw = None
        self.exact = bool(exact)
        self.warm_start = bool(warm_start)
        self._active = {18: np.zeros((1, 3), np.uint32), 12: np.zeros((1, 3), np.uint32)}   # opt_stance's and opt_swing's sets

    def setQ(self, Q_):
        self._Q = np.array(Q_, dtype=np.float64).reshape(1, 30, 30)

    def setc(self, c_):
        self._c = np.array(c_, dtype=np.float64).reshape(1, 30)

    def setL_stance(self, L_stance):
        self._Ls = np.array(L_stance, dtype=np.float64).reshape(1, 86, 31)

    def setL_swing(self, L_swing):
        self._Lw = np.array(L_swing, dtype=np.float64).reshape(1, 82, 31)

    def _solve(self, L, neq):
        if self._Q is None or self._c is None or L is None:
            raise WbcError("OPT: setQ, setc and setL_* must be called before opt_*")
        if self.warm_start:
            x, status, _, _, self._active[neq] = self._b.qp_solve(self._Q, self._c, L, neq, exact=True, warm=True, active=self._active[neq])
        else:
            x, status, _, _ = self._b.qp_solve(self._Q, self._c, L, neq, exact=self.exact)
        if status[0] != 0:
            raise WbcError("OPT: QP solver failed with status %d" % status[0])
        return x[0]

    def opt_stance(self):
        return self._solve(self._Ls, 18)     # first 18 rows are equalities (lopt.cpp:40-47)

    def opt_swing(self):
        return self._solve(self._Lw, 12)     # first 12 rows are equalities (lopt.cpp:57-64)
