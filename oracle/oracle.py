"""ctypes wrapper of the CPU oracle ``oracle/_build/libba_oracle.so``.

TEST INFRASTRUCTURE ONLY. The POD structs are shared with the product's C ABI
(``camera_calibration_b200.cabi`` mirrors ``include/b200ba.h``) so that the same flattened
problem is handed to both sides.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from camera_calibration_b200 import cabi
from camera_calibration_b200.cabi import Camera, FlatProblem, FlatState, Options, Problem, Report, State

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_build", "libba_oracle.so")
_LIB = None
_D = C.POINTER(C.c_double)
_I32 = C.POINTER(C.c_int32)


def build(force: bool = False, native: bool = False) -> str:
    """Compile the oracle with the committed Makefile (g++, no dependencies) into oracle/_build/.
    ``native=True`` builds the -march=native variant used by the timing legs of bench.py into a
    fresh temporary directory instead: it must match the CPU it runs on, and the source tree may be
    read-only at that point. The directory is removed when the process exits."""
    if native:
        out = tempfile.mkdtemp(prefix="ba_oracle_native_")
        atexit.register(shutil.rmtree, out, True)
        subprocess.check_call(["make", "-C", _HERE, "-s", "native", f"BUILD={out}"], stdout=subprocess.DEVNULL)
        return os.path.join(out, "libba_oracle_native.so")
    target = os.path.join(_HERE, "_build", "libba_oracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("ba_oracle.cc", "ba_oracle.h", "ba_dense_fast.h")] + [
        os.path.join(_HERE, "..", "include", "b200ba.h")]
    if force or not os.path.exists(target) or os.path.getmtime(target) < max(os.path.getmtime(f) for f in srcs):
        cmd = ["make", "-C", _HERE, "-s"] + (["-B"] if force else [])
        subprocess.check_call(cmd, stdout=subprocess.DEVNULL)
    return target


def use_native(threads: int = 0) -> int:
    """Switch this process to a -march=native build made on this machine and set the host thread
    count of the full-size kernels (0 = all cores). Returns the thread count in effect."""
    global _LIB, LIB_PATH
    LIB_PATH = build(native=True)
    _LIB = None
    return set_threads(threads)


def set_threads(n: int) -> int:
    return int(lib().oracle_set_threads(int(n)))


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            build()
        l = C.CDLL(LIB_PATH)
        l.oracle_optimize.restype = C.c_int
        l.oracle_optimize.argtypes = [C.POINTER(Problem), C.POINTER(State), C.POINTER(Options), C.POINTER(Report)]
        l.oracle_evaluate.restype = C.c_int
        l.oracle_evaluate.argtypes = [C.POINTER(Problem), C.POINTER(State), C.POINTER(Options), C.c_int, _D, _D, _D,
                                      _D, _D, _D, _D, _I32, C.c_int32, _I32]
        l.oracle_build_system.restype = C.c_int
        l.oracle_build_system.argtypes = [C.POINTER(Problem), C.POINTER(State), C.POINTER(Options), C.c_int32, _D, _D, _D]
        l.oracle_degrees_of_freedom.restype = C.c_int32
        l.oracle_degrees_of_freedom.argtypes = [C.POINTER(Problem), C.POINTER(Options)]
        l.oracle_schur_solve.restype = C.c_int
        l.oracle_schur_solve.argtypes = [C.c_int32, C.c_int32, C.c_int32, _D, _D, _D, _D, _D, _D]
        l.oracle_solve_dense.restype = C.c_int
        l.oracle_solve_dense.argtypes = [C.c_int32, _D, _D, _D]
        l.oracle_apply_update.restype = C.c_int
        l.oracle_apply_update.argtypes = [C.POINTER(Problem), C.POINTER(State), C.POINTER(Options), _D]
        l.oracle_project.restype = C.c_int
        l.oracle_project.argtypes = [C.POINTER(Camera), _D, C.c_int64, _D, _D, _I32]
        l.oracle_unproject.restype = C.c_int
        l.oracle_unproject.argtypes = [C.POINTER(Camera), _D, C.c_int64, _D, _D, _D, _I32]
        l.oracle_unproject_jacobian.restype = C.c_int
        l.oracle_unproject_jacobian.argtypes = [C.POINTER(Camera), _D, C.c_int64, _D, _D, _D, _D, _I32]
        l.oracle_bspline_eval.restype = C.c_int
        l.oracle_bspline_eval.argtypes = [C.c_int32, C.c_int32, _D, C.c_double, C.c_double, C.c_int, _D]
        for n in ("oracle_huber_cost", "oracle_huber_weight", "oracle_huber_cost_sq", "oracle_huber_weight_sq"):
            getattr(l, n).restype = C.c_double
            getattr(l, n).argtypes = [C.c_double, C.c_double]
        l.oracle_time_jacobian.restype = C.c_double
        l.oracle_time_jacobian.argtypes = [C.POINTER(Problem), C.POINTER(State), C.POINTER(Options), C.c_int32,
                                           C.c_int32, C.c_int]
        l.oracle_time_contraction.restype = C.c_double
        l.oracle_time_contraction.argtypes = [C.c_int32, C.c_int32]
        l.oracle_time_ldlt.restype = C.c_double
        l.oracle_time_ldlt.argtypes = [C.c_int32]
        l.oracle_set_threads.restype = C.c_int
        l.oracle_set_threads.argtypes = [C.c_int]
        l.oracle_force_fast_dense.restype = None
        l.oracle_force_fast_dense.argtypes = [C.c_int]
        l.oracle_schur_solve_fast.restype = C.c_int
        l.oracle_schur_solve_fast.argtypes = [C.c_int32, C.c_int32, C.c_int32, _D, _D, _D, _D, _D, _D]
        _LIB = l
    return _LIB


def _p(a, t=C.c_double):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


def optimize(problem: FlatProblem, state: FlatState, opt: Options):
    """OptimizeJointly on the CPU. Returns (new_state, report); ``state`` is not modified."""
    st = state.copy()
    if st.last_projection is None:
        st.last_projection = np.zeros((problem.n_obs, 2))
    st.check(problem)
    rep = Report()
    cs = st.c_struct()
    rc = lib().oracle_optimize(C.byref(problem.c_struct()), C.byref(cs), C.byref(opt), C.byref(rep))
    if rc != 0:
        raise RuntimeError(f"oracle_optimize failed ({rc})")
    return st, rep


def evaluate(problem: FlatProblem, state: FlatState, opt: Options, compute_jacobians: bool, K: int = 0):
    """One pass of the cost function. Returns a dict; state.last_projection is updated in a copy."""
    st = state.copy()
    if st.last_projection is None:
        st.last_projection = np.zeros((problem.n_obs, 2))
    n = problem.n_obs
    out = {
        "residuals": np.zeros((n, 2)),
        "costs": np.zeros(n),
        "total_cost": C.c_double(0),
    }
    jp = jo = jr = ji = ii = hj = None
    if compute_jacobians:
        if K == 0:
            K = max(c.intrinsics_jacobian_size() for c in problem.cameras)
        jp = np.zeros((n, 2, 3))
        jo = np.zeros((n, 2, 6))
        jr = np.zeros((n, 2, 6))
        ji = np.zeros((n, 2, K))
        ii = np.full((n, K), -1, dtype=np.int32)
        hj = np.zeros(n, dtype=np.int32)
    cs = st.c_struct()
    rc = lib().oracle_evaluate(C.byref(problem.c_struct()), C.byref(cs), C.byref(opt), int(compute_jacobians),
                               _p(out["residuals"]), _p(out["costs"]), C.byref(out["total_cost"]), _p(jp), _p(jo),
                               _p(jr), _p(ji), _p(ii, C.c_int32), K, _p(hj, C.c_int32))
    if rc != 0:
        raise RuntimeError(f"oracle_evaluate failed ({rc})")
    out["total_cost"] = out["total_cost"].value
    out["last_projection"] = st.last_projection
    out.update(j_point=jp, j_pose=jo, j_rig=jr, j_intr=ji, intr_index=ii, has_jacobian=hj)
    return out


def degrees_of_freedom(problem: FlatProblem, opt: Options) -> int:
    return int(lib().oracle_degrees_of_freedom(C.byref(problem.c_struct()), C.byref(opt)))


def build_system(problem: FlatProblem, state: FlatState, opt: Options):
    st = state.copy()
    if st.last_projection is None:
        st.last_projection = np.zeros((problem.n_obs, 2))
    n = degrees_of_freedom(problem, opt)
    H = np.zeros((n, n))
    b = np.zeros(n)
    cost = C.c_double(0)
    cs = st.c_struct()
    rc = lib().oracle_build_system(C.byref(problem.c_struct()), C.byref(cs), C.byref(opt), n, _p(H), _p(b),
                                   C.byref(cost))
    if rc != 0:
        raise RuntimeError(f"oracle_build_system failed ({rc})")
    return H, b, cost.value


def schur_solve(block_size, D, B, Cm, b1, b2):
    D = np.ascontiguousarray(D, dtype=np.float64)
    B = np.ascontiguousarray(B, dtype=np.float64)
    Cm = np.ascontiguousarray(Cm, dtype=np.float64)
    b1 = np.ascontiguousarray(b1, dtype=np.float64)
    b2 = np.ascontiguousarray(b2, dtype=np.float64)
    nb = D.shape[0]
    nd = Cm.shape[0]
    x = np.zeros(nb * block_size + nd)
    lib().oracle_schur_solve(block_size, nb, nd, _p(D), _p(B), _p(Cm), _p(b1), _p(b2), _p(x))
    return x


def solve_dense(H, b):
    H = np.ascontiguousarray(H, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    x = np.zeros(len(b))
    lib().oracle_solve_dense(len(b), _p(H), _p(b), _p(x))
    return x


def apply_update(problem: FlatProblem, state: FlatState, opt: Options, delta):
    st = state.copy()
    delta = np.ascontiguousarray(delta, dtype=np.float64)
    cs = st.c_struct()
    rc = lib().oracle_apply_update(C.byref(problem.c_struct()), C.byref(cs), C.byref(opt), _p(delta))
    if rc != 0:
        raise RuntimeError("oracle_apply_update failed")
    return st


def project(cam: Camera, intrinsics, local_points, initial_pixels=None):
    lp = np.ascontiguousarray(local_points, dtype=np.float64).reshape(-1, 3)
    n = len(lp)
    if initial_pixels is None:
        cx = 0.5 * (cam.calibration_min_x + cam.calibration_max_x + 1)
        cy = 0.5 * (cam.calibration_min_y + cam.calibration_max_y + 1)
        px = np.tile(np.array([cx, cy]), (n, 1))
    else:
        px = np.array(initial_pixels, dtype=np.float64).reshape(-1, 2).copy()
    px = np.ascontiguousarray(px)
    ok = np.zeros(n, dtype=np.int32)
    intr = np.ascontiguousarray(intrinsics, dtype=np.float64).reshape(-1)
    lib().oracle_project(C.byref(cam), _p(intr), n, _p(lp), _p(px), _p(ok, C.c_int32))
    return px, ok.astype(bool)


def fit_directions(gw: int, gh: int, grid, grid_points, directions, max_iteration_count: int):
    """Returns (new grid [gh, gw, 3], FitReport)."""
    from camera_calibration_b200.cabi import FitReport
    g = np.ascontiguousarray(grid, dtype=np.float64).reshape(-1).copy()
    gp = np.ascontiguousarray(grid_points, dtype=np.float64).reshape(-1, 2)
    d = np.ascontiguousarray(directions, dtype=np.float64).reshape(-1, 3)
    rep = FitReport()
    f = lib().oracle_fit_directions
    f.restype = C.c_int
    f.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_double), C.c_int64, C.POINTER(C.c_double),
                  C.POINTER(C.c_double), C.c_int32, C.POINTER(FitReport)]
    rc = f(gw, gh, _p(g), len(gp), _p(gp), _p(d), max_iteration_count, C.byref(rep))
    if rc != 0:
        raise RuntimeError("oracle_fit_directions failed")
    return g.reshape(gh, gw, 3), rep


def unproject(cam: Camera, intrinsics, pixels, with_jacobian=False):
    px = np.ascontiguousarray(pixels, dtype=np.float64).reshape(-1, 2)
    n = len(px)
    d = np.zeros((n, 3))
    o = np.zeros((n, 3))
    ok = np.zeros(n, dtype=np.int32)
    intr = np.ascontiguousarray(intrinsics, dtype=np.float64).reshape(-1)
    if with_jacobian:
        rows = 3 if cam.model_type == cabi.MODEL_CENTRAL_GENERIC else 6
        J = np.zeros((n, rows, 2))
        lib().oracle_unproject_jacobian(C.byref(cam), _p(intr), n, _p(px), _p(d), _p(o), _p(J), _p(ok, C.c_int32))
        return d, o, J, ok.astype(bool)
    lib().oracle_unproject(C.byref(cam), _p(intr), n, _p(px), _p(d), _p(o), _p(ok, C.c_int32))
    return d, o, ok.astype(bool)


def bspline_eval(grid, x, y, slow=False):
    g = np.ascontiguousarray(grid, dtype=np.float64)
    gh, gw = g.shape[0], g.shape[1]
    out = np.zeros(3)
    lib().oracle_bspline_eval(gw, gh, _p(g), float(x), float(y), int(slow), _p(out))
    return out


def time_jacobian(problem, state, opt, first_imageset, count, compute_jacobians=True) -> float:
    st = state.copy()
    if st.last_projection is None:
        st.last_projection = np.zeros((problem.n_obs, 2))
    cs = st.c_struct()
    return float(lib().oracle_time_jacobian(C.byref(problem.c_struct()), C.byref(cs), C.byref(opt), first_imageset,
                                            count, int(compute_jacobians)))


def time_contraction(n_rows, n_cols) -> float:
    return float(lib().oracle_time_contraction(n_rows, n_cols))


def time_ldlt(n) -> float:
    return float(lib().oracle_time_ldlt(n))
