"""ORACLE -- TEST INFRASTRUCTURE ONLY (ctypes view of oracle/liboracle.so).

CPU restatement of the reference's hot path.  May be imported only by tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None
i64p = C.POINTER(C.c_int64)
f64p = C.POINTER(C.c_double)
i8p = C.POINTER(C.c_int8)


_build = "-O3 -march=x86-64-v3 (oracle/liboracle.so, portable build of the Makefile)"


def build_flags():
    """How the loaded library was compiled (the CPU-baseline legs of bench.py report it)."""
    lib()
    return _build


def _native_lib():
    """ORACLE_NATIVE=1 (set by bench.py's CPU legs): compile the port for THIS host, `gcc -O3 -march=native`
    (BASELINE.md section 3), into a new private directory (mkdtemp: owned by this user, mode 0700, unpredictable
    name), load it and delete the directory again.  Nothing is written into the source tree, which may be read-only,
    nothing is left behind, and no library that another user could have placed is ever loaded.  The portable library
    stays the fallback: a library built with -march=native on one machine may not run on another, so it is never
    shipped."""
    import glob
    import shutil
    import subprocess
    import tempfile
    if os.environ.get("ORACLE_NATIVE", "0") != "1":
        return None
    srcs = sorted(glob.glob(os.path.join(_HERE, "*.c")))
    tmp = tempfile.mkdtemp(prefix="clarabel_b200_oracle_")
    try:
        out = os.path.join(tmp, "liboracle_native.so")
        subprocess.check_call(["gcc", "-O3", "-march=native", "-fPIC", "-shared", "-o", out] + srcs + ["-lm"],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=300)
        return C.CDLL(out)          # the mapping outlives the file
    except Exception:
        return None
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def lib():
    global _lib, _build
    if _lib is None:
        path = os.path.join(_HERE, "liboracle.so")
        L = _native_lib()
        if L is not None:
            _build = "-O3 -march=native, compiled on this host"
        elif not os.path.exists(path):
            raise RuntimeError("oracle/liboracle.so missing: run `make` (or __graft_entry__.build())")
        else:
            L = C.CDLL(path)
        vp = C.c_void_p
        L.oq_new.argtypes = [C.POINTER(vp), C.c_int64, C.c_int64, i64p, i64p, f64p, i64p, i8p,
                             C.c_int, C.c_int, C.c_double, C.c_double]
        L.oq_free.argtypes = [vp]
        L.oq_free.restype = None
        L.oq_refactor.argtypes = [vp]
        L.oq_solve.argtypes = [vp, f64p]
        L.oq_update_values.argtypes = [vp, i64p, f64p, C.c_int64]
        L.oq_update_values.restype = None
        L.oq_scale_values.argtypes = [vp, i64p, C.c_int64, C.c_double]
        L.oq_scale_values.restype = None
        L.oq_offset_values.argtypes = [vp, i64p, C.c_int64, C.c_double, i8p]
        L.oq_offset_values.restype = None
        L.oq_dinv_is_finite.argtypes = [vp]
        for nm in ["oq_n", "oq_nnzA", "oq_nnzL", "oq_regularize_count", "oq_positive_inertia"]:
            getattr(L, nm).argtypes = [vp]
            getattr(L, nm).restype = C.c_int64
        for nm in ["oq_Lp", "oq_Li", "oq_etree_ptr", "oq_Lnz", "oq_permA_colptr", "oq_permA_rowval",
                   "oq_AtoPAPt"]:
            getattr(L, nm).argtypes = [vp]
            getattr(L, nm).restype = i64p
        for nm in ["oq_Lx", "oq_D", "oq_Dinv", "oq_permA_nzval"]:
            getattr(L, nm).argtypes = [vp]
            getattr(L, nm).restype = f64p
        L.oq_invperm.argtypes = [C.c_int64, i64p, i64p]
        L.oq_permute.argtypes = [C.c_int64, f64p, f64p, i64p]
        L.oq_permute.restype = None
        L.oq_ipermute.argtypes = [C.c_int64, f64p, f64p, i64p]
        L.oq_ipermute.restype = None
        L.oq_permute_symmetric.argtypes = [C.c_int64, i64p, i64p, f64p, i64p, i64p, i64p, f64p, i64p]
        L.oq_permute_symmetric.restype = None
        L.oq_etree.argtypes = [C.c_int64, i64p, i64p, i64p, i64p, i64p]
        L.oq_etree.restype = None
        for nm in ["oq_lsolve", "oq_ltsolve"]:
            getattr(L, nm).argtypes = [C.c_int64, i64p, i64p, f64p, f64p]
            getattr(L, nm).restype = None
        L.oq_dltsolve.argtypes = [C.c_int64, i64p, i64p, f64p, f64p, f64p]
        L.oq_dltsolve.restype = None
        L.oq_solve_factors.argtypes = [C.c_int64, i64p, i64p, f64p, f64p, f64p]
        L.oq_solve_factors.restype = None
        _lib = L
    return _lib


def I(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def F(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def P(a):
    if a.dtype == np.int64:
        return a.ctypes.data_as(i64p)
    if a.dtype == np.float64:
        return a.ctypes.data_as(f64p)
    if a.dtype == np.int8:
        return a.ctypes.data_as(i8p)
    raise TypeError(a.dtype)


class QDLDLError(Exception):
    def __init__(self, code):
        names = {-1: "IncompatibleDimension", -2: "EmptyColumn", -3: "NotUpperTriangular",
                 -4: "ZeroPivot", -5: "InvalidPermutation"}
        super().__init__(names.get(code, str(code)))
        self.code = code


class QDLDL:
    """Oracle factorisation object (mirrors QDLDLFactorisation, qdldl.rs:72-211)."""

    def __init__(self, shape, colptr, rowval, nzval, perm, dsigns=None, logical=False,
                 regularize_enable=True, regularize_eps=1e-12, regularize_delta=1e-7):
        L = lib()
        self._L = L
        m, n = shape
        cp, rv, nz, pm = I(colptr), I(rowval), F(nzval), I(perm)
        ds = np.ascontiguousarray(dsigns, dtype=np.int8) if dsigns is not None else None
        h = C.c_void_p()
        rc = L.oq_new(C.byref(h), m, n, P(cp), P(rv), P(nz), P(pm), P(ds) if ds is not None else None,
                      1 if logical else 0, 1 if regularize_enable else 0, regularize_eps, regularize_delta)
        if rc:
            raise QDLDLError(rc)
        self._h = h
        self.n = n

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.oq_free(self._h)
            self._h = None

    def refactor(self):
        rc = self._L.oq_refactor(self._h)
        if rc:
            raise QDLDLError(rc)

    def refactor_ok(self):
        """Adapter-level bool (ldlsolvers/qdldl.rs:99-106)."""
        self.refactor()
        return bool(self._L.oq_dinv_is_finite(self._h))

    def solve(self, b):
        x = F(b).copy()
        if self._L.oq_solve(self._h, P(x)) != 0:
            raise AssertionError("solve on a logical factorisation (qdldl.rs:118)")
        return x

    def update_values(self, index, values):
        idx, v = I(index), F(values)
        self._L.oq_update_values(self._h, P(idx), P(v), idx.size)

    def scale_values(self, index, scale):
        idx = I(index)
        self._L.oq_scale_values(self._h, P(idx), idx.size, float(scale))

    def offset_values(self, index, offset, signs):
        idx = I(index)
        sg = np.ascontiguousarray(signs, dtype=np.int8)
        assert idx.size == sg.size
        self._L.oq_offset_values(self._h, P(idx), idx.size, float(offset), P(sg))

    def _arr(self, fn, n, dt):
        p = getattr(self._L, fn)(self._h)
        return np.ctypeslib.as_array(p, shape=(max(int(n), 1),))[:int(n)].astype(dt, copy=True)

    @property
    def nnzL(self):
        return int(self._L.oq_nnzL(self._h))

    @property
    def nnzA(self):
        return int(self._L.oq_nnzA(self._h))

    @property
    def regularize_count(self):
        return int(self._L.oq_regularize_count(self._h))

    @property
    def positive_inertia(self):
        return int(self._L.oq_positive_inertia(self._h))

    @property
    def D(self):
        return self._arr("oq_D", self.n, np.float64)

    @property
    def Dinv(self):
        return self._arr("oq_Dinv", self.n, np.float64)

    @property
    def Lp(self):
        return self._arr("oq_Lp", self.n + 1, np.int64)

    @property
    def Li(self):
        return self._arr("oq_Li", self.nnzL, np.int64)

    @property
    def Lx(self):
        return self._arr("oq_Lx", self.nnzL, np.float64)

    @property
    def etree(self):
        return self._arr("oq_etree_ptr", self.n, np.int64)

    @property
    def permA(self):
        cp = self._arr("oq_permA_colptr", self.n + 1, np.int64)
        return (cp, self._arr("oq_permA_rowval", self.nnzA, np.int64),
                self._arr("oq_permA_nzval", self.nnzA, np.float64))

    @property
    def AtoPAPt(self):
        return self._arr("oq_AtoPAPt", self.nnzA, np.int64)


# ---------------------------------------------------------------------------
# IPM oracle (oracle/ipm_oracle.c)
# ---------------------------------------------------------------------------
CONE_CODES = {"zero": 0, "nonneg": 1, "soc": 2, "psd": 3, "exp": 4, "pow": 5, "genpow": 6}
STATUS_NAMES = ["Unsolved", "Solved", "PrimalInfeasible", "DualInfeasible", "AlmostSolved",
                "AlmostPrimalInfeasible", "AlmostDualInfeasible", "MaxIterations", "MaxTime",
                "NumericalError", "InsufficientProgress"]


class Settings(C.Structure):
    _fields_ = [
        ("max_iter", C.c_int32), ("time_limit", C.c_double), ("max_step_fraction", C.c_double),
        ("tol_gap_abs", C.c_double), ("tol_gap_rel", C.c_double), ("tol_feas", C.c_double),
        ("tol_infeas_abs", C.c_double), ("tol_infeas_rel", C.c_double), ("tol_ktratio", C.c_double),
        ("reduced_tol_gap_abs", C.c_double), ("reduced_tol_gap_rel", C.c_double),
        ("reduced_tol_feas", C.c_double), ("reduced_tol_infeas_abs", C.c_double),
        ("reduced_tol_infeas_rel", C.c_double), ("reduced_tol_ktratio", C.c_double),
        ("equilibrate_enable", C.c_int32), ("equilibrate_max_iter", C.c_int32),
        ("equilibrate_min_scaling", C.c_double), ("equilibrate_max_scaling", C.c_double),
        ("min_terminate_step_length", C.c_double),
        ("static_regularization_enable", C.c_int32),
        ("static_regularization_constant", C.c_double),
        ("static_regularization_proportional", C.c_double),
        ("dynamic_regularization_enable", C.c_int32),
        ("dynamic_regularization_eps", C.c_double), ("dynamic_regularization_delta", C.c_double),
        ("iterative_refinement_enable", C.c_int32),
        ("iterative_refinement_reltol", C.c_double), ("iterative_refinement_abstol", C.c_double),
        ("iterative_refinement_max_iter", C.c_int32),
        ("iterative_refinement_stop_ratio", C.c_double),
        ("linesearch_backtrack_step", C.c_double), ("min_switch_step_length", C.c_double),
        ("presolve_enable", C.c_int32),
    ]


class Info(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("iterations", C.c_int32),
        ("cost_primal", C.c_double), ("cost_dual", C.c_double), ("res_primal", C.c_double),
        ("res_dual", C.c_double), ("res_primal_inf", C.c_double), ("res_dual_inf", C.c_double),
        ("gap_abs", C.c_double), ("gap_rel", C.c_double), ("ktratio", C.c_double), ("mu", C.c_double),
        ("step_length", C.c_double), ("sigma", C.c_double),
        ("solve_time", C.c_double), ("t_kkt_update", C.c_double), ("t_kkt_solve", C.c_double),
        ("t_scale_cones", C.c_double),
        ("n_refactor", C.c_int64), ("n_ldl_solve", C.c_int64), ("nnzL", C.c_int64), ("nnzK", C.c_int64),
    ]

    @property
    def status_name(self):
        return STATUS_NAMES[self.status]


_ipm_ready = False


def _ipm_lib():
    global _ipm_ready
    L = lib()
    if not _ipm_ready:
        vp = C.c_void_p
        i32p = C.POINTER(C.c_int32)
        L.oipm_default_settings.argtypes = [C.POINTER(Settings)]
        L.oipm_default_settings.restype = None
        L.oipm_new.argtypes = [C.POINTER(vp), C.c_int64, C.c_int64, i64p, i64p, f64p, f64p, i64p, i64p,
                               f64p, f64p, C.c_int64, i32p, i64p, C.POINTER(Settings)]
        L.oipm_new_ex.argtypes = [C.POINTER(vp), C.c_int64, C.c_int64, i64p, i64p, f64p, f64p, i64p, i64p,
                                  f64p, f64p, C.c_int64, i32p, i64p, f64p, C.POINTER(Settings)]
        L.oipm_new_gp.argtypes = [C.POINTER(vp), C.c_int64, C.c_int64, i64p, i64p, f64p, f64p, i64p, i64p,
                                  f64p, f64p, C.c_int64, i32p, i64p, f64p, i64p, f64p, C.POINTER(Settings)]
        L.oipm_free.argtypes = [vp]
        L.oipm_free.restype = None
        L.oipm_test_update_scaling_ex.argtypes = [vp, f64p, f64p, C.c_double, C.c_int]
        L.oipm_test_compute_barrier.argtypes = [vp, f64p, f64p, f64p, f64p, C.c_double]
        L.oipm_test_compute_barrier.restype = C.c_double
        L.oipm_test_unit_initialization.argtypes = [vp, f64p, f64p]
        L.oipm_test_unit_initialization.restype = None
        L.oipm_test_wright_omega.argtypes = [C.c_double]
        L.oipm_test_wright_omega.restype = C.c_double
        L.oipm_test_ns3_state.argtypes = [vp, C.c_int64, f64p]
        L.oipm_test_ns3_state.restype = None
        L.oipm_test_affine_ds_ex.argtypes = [vp, f64p, f64p]
        L.oipm_test_affine_ds_ex.restype = None
        L.oipm_kkt_dim.argtypes = [vp]
        L.oipm_kkt_dim.restype = C.c_int64
        L.oipm_m_reduced.argtypes = [vp]
        L.oipm_m_reduced.restype = C.c_int64
        L.oipm_kkt_nnz.argtypes = [vp]
        L.oipm_kkt_nnz.restype = C.c_int64
        for nm in ["oipm_kkt_colptr", "oipm_kkt_rowval"]:
            getattr(L, nm).argtypes = [vp]
            getattr(L, nm).restype = i64p
        L.oipm_kkt_nzval.argtypes = [vp]
        L.oipm_kkt_nzval.restype = f64p
        L.oipm_kkt_dsigns.argtypes = [vp]
        L.oipm_kkt_dsigns.restype = i8p
        L.oipm_map.argtypes = [vp, C.c_int, i64p]
        L.oipm_map.restype = i64p
        L.oipm_sparse_map.argtypes = [vp, C.c_int64, C.c_int, i64p]
        L.oipm_sparse_map.restype = i64p
        L.oipm_genpow_map.argtypes = [vp, C.c_int64, C.c_int, i64p]
        L.oipm_genpow_map.restype = i64p
        L.oipm_test_kkt_update.argtypes = [vp]
        L.oipm_equil.argtypes = [vp, C.c_int]
        L.oipm_equil.restype = f64p
        L.oipm_scaled_data.argtypes = [vp, C.c_int]
        L.oipm_scaled_data.restype = f64p
        L.oipm_set_perm.argtypes = [vp, i64p]
        L.oipm_solve.argtypes = [vp, f64p, C.c_int32]
        L.oipm_get_solution.argtypes = [vp, f64p, f64p, f64p, f64p, f64p]
        L.oipm_get_solution.restype = None
        L.oipm_get_info.argtypes = [vp, C.POINTER(Info)]
        L.oipm_get_info.restype = None
        L.oipm_nHs.argtypes = [vp]
        L.oipm_nHs.restype = C.c_int64
        L.oipm_test_update_scaling.argtypes = [vp, f64p, f64p]
        L.oipm_test_get_Hs.argtypes = [vp, f64p]
        L.oipm_test_get_Hs.restype = None
        L.oipm_test_mul_Hs.argtypes = [vp, f64p, f64p]
        L.oipm_test_mul_Hs.restype = None
        L.oipm_test_affine_ds.argtypes = [vp, f64p]
        L.oipm_test_affine_ds.restype = None
        L.oipm_test_combined_ds_shift.argtypes = [vp, f64p, f64p, f64p, C.c_double]
        L.oipm_test_combined_ds_shift.restype = None
        L.oipm_test_ds_from_dz_offset.argtypes = [vp, f64p, f64p, f64p]
        L.oipm_test_ds_from_dz_offset.restype = None
        L.oipm_test_step_length.argtypes = [vp, f64p, f64p, f64p, f64p, C.c_double]
        L.oipm_test_step_length.restype = C.c_double
        _ipm_ready = True
    return L


def default_settings(**kw):
    s = Settings()
    _ipm_lib().oipm_default_settings(C.byref(s))
    for k, v in kw.items():
        setattr(s, k, v)
    return s


def get_infinity():
    L = _ipm_lib(); L.oipm_get_infinity.restype = C.c_double
    return float(L.oipm_get_infinity())


def set_infinity(v):
    L = _ipm_lib(); L.oipm_set_infinity.argtypes = [C.c_double]; L.oipm_set_infinity.restype = None
    L.oipm_set_infinity(float(v))


def default_infinity():
    L = _ipm_lib(); L.oipm_default_infinity.restype = None
    L.oipm_default_infinity()


def check_dimensions(P, q, A, b, cones):
    """check_dimensions (src/solver/implementations/default/solver.rs:129-159), the order of the tests included;
    SupportedConeT::nvars as in supportedcone.rs:54-71"""
    def nvars(kind, d):
        if kind in ("exp", "pow"):
            return 3
        if kind == "psd":
            return int(d) * (int(d) + 1) // 2
        if kind == "genpow":
            return len(d[0]) + int(d[1])
        return int(d)
    m, n = len(b), len(q)
    if m != A.shape[0]:
        raise ValueError("A and b incompatible dimensions")
    if sum(nvars(k, d) for k, d in cones) != m:
        raise ValueError("Constraint dimensions inconsistent with size of cones")
    if n != A.shape[1]:
        raise ValueError("A and q incompatible dimensions")
    if n != P.shape[1]:
        raise ValueError("P and q incompatible dimensions")
    if P.shape[0] != P.shape[1]:
        raise ValueError("P not square")


class IPM:
    """Oracle interior-point solver (mirrors DefaultSolver::new / solve()).

    P is any scipy sparse symmetric or upper-triangular matrix (converted to
    triu like problemdata.rs:79-81), A scipy sparse, cones a list of
    (kind, dim) with kind in {"zero","nonneg","soc","psd"}, ("exp", 3) for an
    ExponentialConeT(), ("pow", alpha) for a PowerConeT(alpha) or
    ("genpow", (alphas, dim2)) for a GenPowerConeT(alphas, dim2).
    """

    def __init__(self, P, q, A, b, cones, settings=None):
        import scipy.sparse as sp
        L = _ipm_lib()
        self._L = L
        P, A = sp.csc_matrix(P), sp.csc_matrix(A)
        check_dimensions(P, q, A, b, cones)
        P = sp.triu(P, format="csc")
        P.sort_indices()
        A.sort_indices()
        n, m = P.shape[0], A.shape[0]
        self.n, self.m = n, m
        ct = np.ascontiguousarray([CONE_CODES[k] for k, _ in cones], dtype=np.int32)
        cd = I([3 if k in ("exp", "pow") else (len(d[0]) if k == "genpow" else d) for k, d in cones])
        cpar = F([float(d) if k == "pow" else 0.0 for k, d in cones])
        gdim2 = I([int(d[1]) if k == "genpow" else 0 for k, d in cones])
        galpha = F([a for k, d in cones if k == "genpow" for a in d[0]] or [0.0])
        self.settings = settings if settings is not None else default_settings()
        h = C.c_void_p()
        Pp, Pi, Px = I(P.indptr), I(P.indices), F(P.data)
        Ap, Ai, Ax = I(A.indptr), I(A.indices), F(A.data)
        rc = L.oipm_new_gp(C.byref(h), n, m, P_(Pp), P_(Pi), P_(Px), P_(F(q)), P_(Ap), P_(Ai), P_(Ax), P_(F(b)),
                           len(cones), ct.ctypes.data_as(C.POINTER(C.c_int32)), P_(cd), P_(cpar), P_(gdim2), P_(galpha),
                           C.byref(self.settings))
        if rc:
            raise ValueError(f"oipm_new failed: {rc}")
        self._h = h
        self.N = int(L.oipm_kkt_dim(h))
        self.m_reduced = int(L.oipm_m_reduced(h))     # rows left after the inf-bound presolve (== m without it)

    def __del__(self):
        if getattr(self, "_h", None):
            self._L.oipm_free(self._h)
            self._h = None

    def kkt(self):
        L, h = self._L, self._h
        N, nnz = self.N, int(L.oipm_kkt_nnz(h))
        cp = np.ctypeslib.as_array(L.oipm_kkt_colptr(h), shape=(N + 1,)).copy()
        rv = np.ctypeslib.as_array(L.oipm_kkt_rowval(h), shape=(max(nnz, 1),))[:nnz].copy()
        nz = np.ctypeslib.as_array(L.oipm_kkt_nzval(h), shape=(max(nnz, 1),))[:nnz].copy()
        ds = np.ctypeslib.as_array(L.oipm_kkt_dsigns(h), shape=(N,)).copy()
        return N, cp, rv, nz, ds

    def map(self, which):
        ln = C.c_int64()
        p = self._L.oipm_map(self._h, {"P": 0, "A": 1, "Hsblocks": 2, "diagP": 3, "diag_full": 4}[which], C.byref(ln))
        return np.ctypeslib.as_array(p, shape=(max(ln.value, 1),))[:ln.value].copy()

    def sparse_map(self, k, which):
        ln = C.c_int64()
        p = self._L.oipm_sparse_map(self._h, k, {"u": 0, "v": 1, "D": 2}[which], C.byref(ln))
        return np.ctypeslib.as_array(p, shape=(max(ln.value, 1),))[:ln.value].copy()

    def genpow_map(self, k, which):
        ln = C.c_int64()
        p = self._L.oipm_genpow_map(self._h, k, {"q": 0, "r": 1, "p": 2, "D": 3}[which], C.byref(ln))
        return np.ctypeslib.as_array(p, shape=(max(ln.value, 1),))[:ln.value].copy()

    def kkt_update(self):
        """KKTSolver::update with the current cone scalings (set_perm first)"""
        return bool(self._L.oipm_test_kkt_update(self._h))

    def equilibration(self):
        L, h = self._L, self._h
        d = np.ctypeslib.as_array(L.oipm_equil(h, 0), shape=(max(self.n, 1),))[:self.n].copy()
        e = np.ctypeslib.as_array(L.oipm_equil(h, 1), shape=(max(self.m, 1),))[:self.m_reduced].copy()
        c = float(L.oipm_equil(h, 2)[0])
        return d, e, c

    def set_perm(self, perm):
        rc = self._L.oipm_set_perm(self._h, P_(I(perm)))
        if rc:
            raise QDLDLError(rc)

    def regularize_count(self):
        """dynamically regularised pivots of the last refactorisation"""
        self._L.oipm_regularize_count.restype = C.c_int64
        self._L.oipm_regularize_count.argtypes = [C.c_void_p]
        return int(self._L.oipm_regularize_count(self._h))

    def solve(self, trace_cap=256):
        tr = np.zeros((trace_cap, 6))
        rc = self._L.oipm_solve(self._h, P_(tr.reshape(-1)), trace_cap)
        if rc:
            raise RuntimeError("oipm_solve: set_perm() first")
        info = Info()
        self._L.oipm_get_info(self._h, C.byref(info))
        x, z, s = np.zeros(max(self.n, 1)), np.zeros(max(self.m, 1)), np.zeros(max(self.m, 1))
        obj, objd = C.c_double(), C.c_double()
        self._L.oipm_get_solution(self._h, P_(x), P_(z), P_(s), C.byref(obj), C.byref(objd))
        self.info = info
        self.trace = tr[:min(info.iterations + 1, trace_cap)]
        return dict(status=info.status_name, iterations=info.iterations, x=x[:self.n], z=z[:self.m], s=s[:self.m],
                    obj_val=obj.value, obj_val_dual=objd.value, info=info)

    # cone-level entry points for unit parity tests of the CUDA cone kernels
    def update_scaling(self, s, z):
        return bool(self._L.oipm_test_update_scaling(self._h, P_(F(s)), P_(F(z))))

    def update_scaling_ex(self, s, z, mu, strategy):
        """strategy: 0 primal-dual, 1 dual (ScalingStrategy, cones/mod.rs)"""
        return bool(self._L.oipm_test_update_scaling_ex(self._h, P_(F(s)), P_(F(z)), float(mu), int(strategy)))

    def ns3_state(self, k):
        out = np.zeros(18)
        self._L.oipm_test_ns3_state(self._h, int(k), P_(out))
        return dict(H_dual=out[:6].copy(), Hs=out[6:12].copy(), grad=out[12:15].copy(), z=out[15:18].copy())

    def compute_barrier(self, z, s, dz, ds, alpha):
        return float(self._L.oipm_test_compute_barrier(self._h, P_(F(z)), P_(F(s)), P_(F(dz)), P_(F(ds)), float(alpha)))

    def unit_initialization(self):
        z, s = np.zeros(max(self.m, 1)), np.zeros(max(self.m, 1))
        self._L.oipm_test_unit_initialization(self._h, P_(z), P_(s))
        return z[:self.m], s[:self.m]

    def affine_ds_ex(self, s):
        y = np.zeros(max(self.m, 1))
        self._L.oipm_test_affine_ds_ex(self._h, P_(y), P_(F(s)))
        return y[:self.m]

    def get_Hs(self):
        out = np.zeros(max(int(self._L.oipm_nHs(self._h)), 1))
        self._L.oipm_test_get_Hs(self._h, P_(out))
        return out[:int(self._L.oipm_nHs(self._h))]

    def mul_Hs(self, x):
        y = np.zeros(max(self.m, 1))
        self._L.oipm_test_mul_Hs(self._h, P_(y), P_(F(x)))
        return y[:self.m]

    def affine_ds(self):
        y = np.zeros(max(self.m, 1))
        self._L.oipm_test_affine_ds(self._h, P_(y))
        return y[:self.m]

    def combined_ds_shift(self, step_z, step_s, sigmamu):
        sh, sz, ss = np.zeros(max(self.m, 1)), F(step_z).copy(), F(step_s).copy()
        self._L.oipm_test_combined_ds_shift(self._h, P_(sh), P_(sz), P_(ss), float(sigmamu))
        return sh[:self.m]

    def ds_from_dz_offset(self, ds, z):
        out = np.zeros(max(self.m, 1))
        self._L.oipm_test_ds_from_dz_offset(self._h, P_(out), P_(F(ds)), P_(F(z)))
        return out[:self.m]

    def step_length(self, dz, ds, z, s, amax=1.0):
        return float(self._L.oipm_test_step_length(self._h, P_(F(dz)), P_(F(ds)), P_(F(z)), P_(F(s)), amax))


P_ = P
