"""ORACLE — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

ctypes binding over oracle/liboracle.so (the CPU restatement of the
reference's dense ProxQP path, see oracle/proxqp_oracle.hpp).  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module.
"""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")
_lib = None

INFO_FIELDS = [
    "mu_eq", "mu_eq_inv", "mu_in", "mu_in_inv", "rho", "nu", "iter", "iter_ext",
    "mu_updates", "rho_updates", "status", "setup_time", "solve_time", "run_time",
    "objValue", "pri_res", "dua_res", "duality_gap", "iterative_residual",
    "minimal_H_eigenvalue_estimate",
]
COUNTER_FIELDS = [
    "n_factor", "factor_m2", "factor_m3", "n_solve", "solve_m2", "solve_m", "n_resid",
    "resid_nc", "rank_rt2", "rank_chunk_t2", "rank_rt", "n_insert", "insert_bytes",
    "n_delete", "delete_t2", "ls_evals", "n_cdx", "n_global_res", "n_newton",
]

# status.hpp:17-35, settings.hpp:26-45
PROXQP_SOLVED, PROXQP_MAX_ITER_REACHED, PROXQP_PRIMAL_INFEASIBLE = 0, 1, 2
PROXQP_SOLVED_CLOSEST_PRIMAL_FEASIBLE, PROXQP_DUAL_INFEASIBLE, PROXQP_NOT_RUN = 3, 4, 5
NO_INITIAL_GUESS, EQUALITY_CONSTRAINED_INITIAL_GUESS = 0, 1
WARM_START_WITH_PREVIOUS_RESULT, WARM_START, COLD_START_WITH_PREVIOUS_RESULT = 2, 3, 4
BACKEND_AUTOMATIC, BACKEND_PRIMAL_DUAL_LDLT, BACKEND_PRIMAL_LDLT = 0, 1, 2
HESSIAN_ZERO, HESSIAN_DENSE, HESSIAN_DIAGONAL = 0, 1, 2


def use_native() -> str:
    """bench.py only: rebuild the restatement with -march=native ON THE MACHINE THAT RUNS IT (the committed Makefile
    targets x86-64-v3 so that the prebuilt library of the tests runs on any box) into a temporary directory, removed at
    exit (the source tree may be read-only), and make this module load that library. Falls back to the portable build
    if the compiler is missing. Returns the flags used."""
    global _LIB_PATH, _lib
    out_dir = tempfile.mkdtemp(prefix="pqp_oracle_native_")
    atexit.register(shutil.rmtree, out_dir, True)
    out = os.path.join(out_dir, "liboracle.so")
    flags = "-O3 -march=native -std=c++17 -fopenmp -fPIC -DNDEBUG"
    try:
        subprocess.check_call(["/usr/bin/g++"] + flags.split() + ["-shared", "-o", out, os.path.join(_HERE, "oracle_capi.cpp")],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        C.CDLL(out)  # must load on this CPU
    except Exception:
        build()
        return "-march=x86-64-v3 (portable build; native rebuild failed)"
    _LIB_PATH = out
    _lib = None
    return flags


def build(force: bool = False) -> str:
    """Compile liboracle.so with the committed Makefile (g++, no Eigen)."""
    srcs = ["oracle_capi.cpp", "proxqp_oracle.hpp", "proxqp_solver.hpp", "ldlt.hpp",
            os.path.join("..", "proxsuite_b200", "csrc", "random_qp.hpp")]
    stale = force or not os.path.exists(_LIB_PATH)
    if not stale:
        t = os.path.getmtime(_LIB_PATH)
        stale = any(os.path.getmtime(os.path.join(_HERE, s)) > t for s in srcs)
    if stale:
        subprocess.check_call(["make", "-C", _HERE, "-B", "liboracle.so"],
                              stdout=subprocess.DEVNULL)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        dp = C.POINTER(C.c_double)
        L.orc_last_error.restype = C.c_char_p
        L.orc_qp_create.restype = C.c_void_p
        L.orc_qp_create.argtypes = [C.c_longlong] * 3 + [C.c_int] * 3
        L.orc_qp_destroy.argtypes = [C.c_void_p]
        L.orc_qp_set.argtypes = [C.c_void_p, C.c_char_p, C.c_double]
        L.orc_qp_get.argtypes = [C.c_void_p, C.c_char_p]
        L.orc_qp_get.restype = C.c_double
        L.orc_qp_init.argtypes = [C.c_void_p] + [C.c_void_p] * 9 + [C.c_int] + [C.c_void_p] * 4
        L.orc_qp_update.argtypes = [C.c_void_p] + [C.c_void_p] * 9 + [C.c_int] + [C.c_void_p] * 4
        L.orc_qp_solve.argtypes = [C.c_void_p] + [C.c_void_p] * 3
        L.orc_qp_cleanup.argtypes = [C.c_void_p]
        L.orc_qp_results.argtypes = [C.c_void_p] + [C.c_void_p] * 6
        L.orc_qp_scaled.argtypes = [C.c_void_p] + [C.c_void_p] * 9
        L.orc_qp_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.orc_qp_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double] + [C.c_void_p] * 7
        L.orc_batch_create.restype = C.c_void_p
        L.orc_batch_create.argtypes = [C.c_longlong] * 4 + [C.c_int] * 3
        L.orc_batch_destroy.argtypes = [C.c_void_p]
        L.orc_batch_qp.restype = C.c_void_p
        L.orc_batch_qp.argtypes = [C.c_void_p, C.c_longlong]
        L.orc_batch_size.restype = C.c_longlong
        L.orc_batch_size.argtypes = [C.c_void_p]
        L.orc_batch_solve.restype = C.c_double
        L.orc_batch_solve.argtypes = [C.c_void_p, C.c_longlong]
        L.orc_batch_solve_serial.restype = C.c_double
        L.orc_batch_solve_serial.argtypes = [C.c_void_p]
        L.orc_batch_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.orc_ldlt_create.restype = C.c_void_p
        L.orc_ldlt_create.argtypes = [C.c_void_p, C.c_longlong, C.c_longlong]
        L.orc_ldlt_destroy.argtypes = [C.c_void_p]
        L.orc_ldlt_dim.restype = C.c_longlong
        L.orc_ldlt_dim.argtypes = [C.c_void_p]
        L.orc_ldlt_solve.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_ldlt_reconstruct.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_ldlt_delete_at.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong]
        L.orc_ldlt_insert_block_at.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong]
        L.orc_ldlt_diagonal_update.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]
        L.orc_ldlt_rank_r_update.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]
        L.orc_lehmer_stream.argtypes = [C.c_ulonglong, C.c_longlong, C.c_void_p]
        L.orc_gen_qp.argtypes = [C.c_int, C.c_ulonglong, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double] + [C.c_void_p] * 9
        del dp
        _lib = L
    return _lib


def _p(a):
    """numpy array (or None) -> void pointer; keeps C-contiguous float64."""
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


def _arr(a, shape=None):
    if a is None:
        return None
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    if shape is not None and a.size != int(np.prod(shape)):
        raise ValueError(f"wrong argument size: expected {shape}, got {a.shape}")
    return a


def _opt_scalar(v):
    if v is None:
        return None, None
    c = C.c_double(float(v))
    return c, C.cast(C.pointer(c), C.c_void_p)


class Info:
    pass


class OracleQP:
    """Mirror of proxsuite.proxqp.dense.QP backed by the CPU restatement."""

    def __init__(self, n, n_eq, n_in, box_constraints=False, hessian_type=HESSIAN_DENSE,
                 dense_backend=BACKEND_PRIMAL_DUAL_LDLT, _handle=None, _owner=None):
        self.n, self.n_eq, self.n_in, self.box = int(n), int(n_eq), int(n_in), bool(box_constraints)
        self.n_cons = self.n_in + (self.n if self.box else 0)
        self._owner = _owner
        if _handle is None:
            self._h = lib().orc_qp_create(self.n, self.n_eq, self.n_in, int(self.box), int(hessian_type), int(dense_backend))
            if not self._h:
                raise ValueError(lib().orc_last_error().decode())
            self._own = True
        else:
            self._h = _handle
            self._own = False

    def __del__(self):
        if getattr(self, "_own", False) and self._h:
            lib().orc_qp_destroy(self._h)
            self._h = None

    def set(self, **kw):
        for k, v in kw.items():
            if lib().orc_qp_set(self._h, k.encode(), float(v)) != 0:
                raise KeyError(k)
        return self

    def get(self, name):
        return lib().orc_qp_get(self._h, name.encode())

    def _data(self, H, g, A, b, C_, l, u, l_box, u_box):
        n, ne, ni = self.n, self.n_eq, self.n_in
        arrs = [_arr(H, (n, n)), _arr(g, (n,)), _arr(A, (ne, n)), _arr(b, (ne,)), _arr(C_, (ni, n)),
                _arr(l, (ni,)), _arr(u, (ni,)), _arr(l_box, (n,)), _arr(u_box, (n,))]
        # empty arrays mean "absent" (wrapper.hpp:380-451 resets size-0 inputs)
        arrs = [a if (a is not None and a.size > 0) else None for a in arrs]
        return arrs

    def init(self, H=None, g=None, A=None, b=None, C=None, l=None, u=None, l_box=None, u_box=None,
             compute_preconditioner=True, rho=None, mu_eq=None, mu_in=None, manual_minimal_H_eigenvalue=None):
        arrs = self._data(H, g, A, b, C, l, u, l_box, u_box)
        keep = [_opt_scalar(v) for v in (rho, mu_eq, mu_in, manual_minimal_H_eigenvalue)]
        rc = lib().orc_qp_init(self._h, *[_p(a) for a in arrs], int(compute_preconditioner), *[k[1] for k in keep])
        if rc != 0:
            raise ValueError(lib().orc_last_error().decode())

    def update(self, H=None, g=None, A=None, b=None, C=None, l=None, u=None, l_box=None, u_box=None,
               update_preconditioner=False, rho=None, mu_eq=None, mu_in=None, manual_minimal_H_eigenvalue=None):
        arrs = self._data(H, g, A, b, C, l, u, l_box, u_box)
        keep = [_opt_scalar(v) for v in (rho, mu_eq, mu_in, manual_minimal_H_eigenvalue)]
        rc = lib().orc_qp_update(self._h, *[_p(a) for a in arrs], int(update_preconditioner), *[k[1] for k in keep])
        if rc != 0:
            raise ValueError(lib().orc_last_error().decode())

    def solve(self, x=None, y=None, z=None):
        xs = [_arr(x, (self.n,)), _arr(y, (self.n_eq,)), _arr(z, (self.n_cons,))]
        rc = lib().orc_qp_solve(self._h, *[_p(a) for a in xs])
        if rc != 0:
            raise ValueError(lib().orc_last_error().decode())
        return self.results()

    def cleanup(self):
        lib().orc_qp_cleanup(self._h)

    def results(self):
        x = np.zeros(self.n)
        y = np.zeros(self.n_eq)
        z = np.zeros(self.n_cons)
        se = np.zeros(self.n_eq)
        si = np.zeros(self.n_cons)
        info = np.zeros(20)
        lib().orc_qp_results(self._h, _p(x), _p(y), _p(z), _p(se), _p(si), _p(info))
        inf = Info()
        for k, v in zip(INFO_FIELDS, info):
            setattr(inf, k, int(v) if k in ("iter", "iter_ext", "mu_updates", "rho_updates", "status") else float(v))
        r = Info()
        r.x, r.y, r.z, r.se, r.si, r.info = x, y, z, se, si, inf
        return r

    def scaled(self):
        n, ne, ni = self.n, self.n_eq, self.n_in
        H = np.zeros((n, n)); g = np.zeros(n); A = np.zeros((ne, n)); b = np.zeros(ne)
        Cm = np.zeros((ni, n)); u = np.zeros(ni); l = np.zeros(ni)
        delta = np.zeros(n + ne + self.n_cons)
        c = C.c_double(0)
        lib().orc_qp_scaled(self._h, _p(H), _p(g), _p(A), _p(b), _p(Cm), _p(u), _p(l), _p(delta), C.cast(C.pointer(c), C.c_void_p))
        return dict(H=H, g=g, A=A, b=b, C=Cm, u=u, l=l, delta=delta, c=c.value)

    def counters(self, reset=False):
        out = np.zeros(19)
        lib().orc_qp_counters(self._h, _p(out), int(reset))
        return dict(zip(COUNTER_FIELDS, out))

    def backward(self, loss_derivative, eps=1e-4, rho_new=1e-6, mu_new=1e-6):
        """dense::compute_backward (dense/compute_ECJ.hpp:29-125) on the solved QP: returns the
        BackwardData jacobians dL_dH, dL_dg, dL_dA, dL_db, dL_dC, dL_du, dL_dl."""
        n, ne, ni = self.n, self.n_eq, self.n_in
        ld = np.ascontiguousarray(np.asarray(loss_derivative, dtype=np.float64))
        if ld.size != n + ne + ni:
            raise ValueError("loss_derivative must have dim + n_eq + n_in entries")
        out = dict(dL_dH=np.zeros((n, n)), dL_dg=np.zeros(n), dL_dA=np.zeros((ne, n)), dL_db=np.zeros(ne),
                   dL_dC=np.zeros((ni, n)), dL_du=np.zeros(ni), dL_dl=np.zeros(ni))
        rc = lib().orc_qp_backward(self._h, _p(ld), float(eps), float(rho_new), float(mu_new), *[_p(out[k]) for k in
                                   ("dL_dH", "dL_dg", "dL_dA", "dL_db", "dL_dC", "dL_du", "dL_dl")])
        if rc != 0:
            raise ValueError(lib().orc_last_error().decode())
        return out


class OracleBatch:
    """std::vector<QP> / BatchQP + solve_in_parallel of the restatement."""

    def __init__(self, batch, n, n_eq, n_in, box_constraints=False, hessian_type=HESSIAN_DENSE,
                 dense_backend=BACKEND_PRIMAL_DUAL_LDLT):
        self._h = lib().orc_batch_create(batch, n, n_eq, n_in, int(box_constraints), int(hessian_type), int(dense_backend))
        if not self._h:
            raise ValueError(lib().orc_last_error().decode())
        self.dims = (n, n_eq, n_in, box_constraints, hessian_type, dense_backend)
        self.size = batch

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_batch_destroy(self._h)
            self._h = None

    def __len__(self):
        return self.size

    def __getitem__(self, i):
        n, ne, ni, box, ht, be = self.dims
        return OracleQP(n, ne, ni, box, ht, be, _handle=lib().orc_batch_qp(self._h, i), _owner=self)

    def solve(self, num_threads=0):
        return lib().orc_batch_solve(self._h, int(num_threads))

    def solve_serial(self):
        return lib().orc_batch_solve_serial(self._h)

    def counters(self, reset=False):
        out = np.zeros(19)
        lib().orc_batch_counters(self._h, _p(out), int(reset))
        return dict(zip(COUNTER_FIELDS, out))


def omp_max_threads():
    return lib().orc_omp_max_threads()


def lehmer_uniforms(seed, count):
    out = np.zeros(count)
    lib().orc_lehmer_stream(int(seed), int(count), _p(out))
    return out


GEN_KINDS = {"strongly_convex": 0, "not_strongly_convex": 1, "degenerate": 2, "box_constrained": 3,
             "box_benchmark": 4, "diagonal_benchmark": 5}


def generate_qp(kind, seed, n, n_eq, n_in, sparsity=0.15, strong_convexity=1e-2):
    """Reference-specified synthetic QP (utils/random_qp_problems.hpp), row-major."""
    k = GEN_KINDS[kind]
    rows_in = 2 * n_in if k == 2 else n_in
    H = np.zeros((n, n)); g = np.zeros(n); A = np.zeros((n_eq, n)); b = np.zeros(n_eq)
    Cm = np.zeros((rows_in, n)); u = np.zeros(rows_in); l = np.zeros(rows_in)
    ub = np.zeros(n); lb = np.zeros(n)
    rc = lib().orc_gen_qp(k, int(seed), n, n_eq, n_in, float(sparsity), float(strong_convexity),
                          _p(H), _p(g), _p(A), _p(b), _p(Cm), _p(u), _p(l), _p(ub), _p(lb))
    assert rc == 0
    out = dict(H=H, g=g, A=A, b=b, C=Cm, u=u, l=l)
    if k >= 4:
        out.update(u_box=ub, l_box=lb)
    return out


class OracleLdlt:
    def __init__(self, mat, cap=None):
        mat = _arr(mat)
        m = mat.shape[0]
        self._h = lib().orc_ldlt_create(_p(mat), m, cap or m)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().orc_ldlt_destroy(self._h)
            self._h = None

    def dim(self):
        return lib().orc_ldlt_dim(self._h)

    def solve(self, rhs):
        r = _arr(rhs).copy()
        lib().orc_ldlt_solve(self._h, _p(r))
        return r

    def reconstruct(self):
        m = self.dim()
        out = np.zeros((m, m))
        lib().orc_ldlt_reconstruct(self._h, _p(out))
        return out

    def delete_at(self, idx):
        idx = np.ascontiguousarray(np.asarray(idx, dtype=np.int64))
        lib().orc_ldlt_delete_at(self._h, idx.ctypes.data_as(C.c_void_p), len(idx))

    def insert_block_at(self, i, a):
        a = np.asfortranarray(np.asarray(a, dtype=np.float64))
        lib().orc_ldlt_insert_block_at(self._h, int(i), a.ctypes.data_as(C.c_void_p), a.shape[1])

    def diagonal_update(self, idx, alpha):
        idx = np.ascontiguousarray(np.asarray(idx, dtype=np.int64))
        alpha = _arr(alpha)
        lib().orc_ldlt_diagonal_update(self._h, idx.ctypes.data_as(C.c_void_p), len(idx), _p(alpha))

    def rank_r_update(self, w, alpha):
        w = np.asfortranarray(np.asarray(w, dtype=np.float64))
        alpha = _arr(alpha)
        lib().orc_ldlt_rank_r_update(self._h, w.ctypes.data_as(C.c_void_p), w.shape[1], _p(alpha))
