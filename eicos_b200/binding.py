"""ctypes binding of the C ABI declared in include/eicos_b200.h.

`Library(path)` wraps one shared object; `load()` returns the product library
(eicos_b200/libeicos_b200.so, hand-written CUDA for sm_100a) and raises if it is missing -
there is no CPU fallback.  Host-side classes mirror the reference's interface:
`Solver` ~ EiCOS::Solver (pointer ctor, include/eicos.hpp:151-163 of the reference) and
`BatchSolver` is the batched overload over stacked instance data.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PRODUCT_LIB = os.path.join(HERE, "libeicos_b200.so")

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class Info(C.Structure):
    _fields_ = [(k, C.c_double) for k in
                ("pcost", "dcost", "pres", "dres", "pinfres", "dinfres", "gap", "relgap",
                 "sigma", "mu", "step", "step_aff", "kapovert")] + \
               [(k, C.c_int) for k in
                ("pinf", "dinf", "has_pinfres", "has_dinfres", "has_relgap",
                 "iter", "iter_max", "nitref1", "nitref2", "nitref3")]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class Settings(C.Structure):
    """eicos_settings: the solver settings a handle applies to every later solve (include/eicos_b200.h)."""
    _fields_ = [(k, C.c_double) for k in
                ("feastol", "abstol", "reltol", "feastol_inacc", "abstol_inacc", "reltol_inacc",
                 "linsysacc", "irerrfact", "gamma", "stepmin", "stepmax", "sigmamin", "sigmamax", "safeguard")] + \
               [(k, C.c_int) for k in ("nitref", "iter_max")]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class _HasSettings:
    """settings() / set_settings(**fields) over the handle's get / set functions (_GET, _SET)."""

    def settings(self):
        """The handle's solver settings as a dict (the keys of eicos_settings)."""
        st = Settings()
        self.lib.check(getattr(self.lib.L, self._GET)(self.h, C.byref(st)))
        return st.asdict()

    def set_settings(self, **fields):
        """Merge `fields` into the current settings; every later solve uses them.  An unknown key raises
        ValueError; a value out of range raises RuntimeError naming the field and changes nothing."""
        cur = self.settings()
        unknown = sorted(set(fields) - set(cur))
        if unknown:
            raise ValueError(f"unknown solver settings: {', '.join(unknown)} (known: {', '.join(cur)})")
        cur.update(fields)
        self.lib.check(getattr(self.lib.L, self._SET)(self.h, C.byref(Settings(**cur))))


def default_settings(lib=None):
    """The reference's default settings (eicos_default_settings) as a dict."""
    st = Settings()
    (lib or load()).L.eicos_default_settings(C.byref(st))
    return st.asdict()


class BatchStats(C.Structure):
    _fields_ = [("chunks", C.c_int), ("ipm_iterations", C.c_int), ("launches", C.c_longlong),
                ("ir_rounds", C.c_ulonglong), ("ms_total", C.c_double), ("ms_factor", C.c_double),
                ("ms_solve", C.c_double), ("ms_other", C.c_double),
                ("factor_launch_tiles", C.c_longlong), ("solve_launch_tiles", C.c_longlong),
                ("factor_launches", C.c_int), ("solve_launches", C.c_int), ("compactions", C.c_int),
                ("kkt_phase_cycles", C.c_ulonglong * 5),
                ("ms_resid", C.c_double), ("ms_vector", C.c_double),
                ("resid_launch_tiles", C.c_longlong), ("vector_launch_tiles", C.c_longlong),
                ("resid_launches", C.c_int), ("vector_launches", C.c_int), ("lane_rounds", C.c_ulonglong)]

    def asdict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_}
        d["kkt_phase_cycles"] = list(d["kkt_phase_cycles"])
        return d


class BatchDims(C.Structure):
    _fields_ = [(k, C.c_int) for k in
                ("n", "m", "p", "l", "ncones", "dim_K", "nnzK", "nnzL", "nnzV", "nnzG", "nnzA",
                 "etree_height", "max_col", "tile_width", "workers")] + \
               [(k, C.c_longlong) for k in ("ldl_fma", "capacity", "workspace_bytes", "rows_per_instance")]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ProgramStats(C.Structure):
    _fields_ = [("sw_slots", C.c_int), ("fa_slots", C.c_int), ("fa_fast", C.c_int),
                ("sw_far", C.c_longlong), ("sw_direct", C.c_longlong), ("fa_home", C.c_longlong),
                ("fw_loads", C.c_int), ("bw_loads", C.c_int), ("fa_loads", C.c_int), ("mv_loads", C.c_int)]

    def asdict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


EXPORTS = [
    "eicos_setup", "eicos_update_data", "eicos_update_data_full", "eicos_solve", "eicos_solution",
    "eicos_get_duals", "eicos_get_info", "eicos_cleanup",
    "eicos_default_settings", "eicos_set_settings", "eicos_get_settings",
    "eicos_batch_set_settings", "eicos_batch_get_settings", "eicos_multi_set_settings", "eicos_multi_get_settings",
    "eicos_batch_setup", "eicos_batch_setup_ex", "eicos_batch_update_matrices", "eicos_batch_solve",
    "eicos_batch_solve_matrices", "eicos_batch_solve_device", "eicos_batch_solve_matrices_device",
    "eicos_batch_adjoint", "eicos_batch_adjoint_device", "eicos_batch_tangent", "eicos_batch_tangent_device",
    "eicos_batch_set_timing", "eicos_batch_set_compaction", "eicos_batch_get_stats", "eicos_batch_get_dims", "eicos_batch_get_program_stats", "eicos_batch_get_symbolic",
    "eicos_batch_debug_init", "eicos_batch_debug_line_search", "eicos_batch_debug_set_iter_max", "eicos_batch_stream", "eicos_batch_cleanup",
    "eicos_multi_setup", "eicos_multi_solve", "eicos_multi_ngpu", "eicos_multi_slice", "eicos_multi_cleanup",
    "eicos_last_error", "eicos_device_count",
]


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _i(a):
    return None if a is None else a.ctypes.data_as(_ip)


def _arr(v, dt):
    if v is None:
        return None
    a = np.ascontiguousarray(v, dtype=dt)
    return a if a.size else None


class Library:
    def __init__(self, path):
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). eicos_b200 has no CPU fallback.")
        self.path = path
        L = self.L = C.CDLL(path)
        setup_args = [C.c_int] * 5 + [_ip, _dp, _ip, _ip, _dp, _ip, _ip, _dp, _dp, _dp]
        L.eicos_setup.restype = C.c_void_p
        L.eicos_setup.argtypes = setup_args + [C.c_int]
        for f in (L.eicos_update_data, L.eicos_update_data_full):
            f.restype = C.c_int
            f.argtypes = [C.c_void_p] + [_dp] * 5
        L.eicos_solve.restype = C.c_int
        L.eicos_solve.argtypes = [C.c_void_p]
        L.eicos_solution.restype = _dp
        L.eicos_solution.argtypes = [C.c_void_p]
        L.eicos_get_duals.restype = C.c_int
        L.eicos_get_duals.argtypes = [C.c_void_p, _dp, _dp, _dp]
        L.eicos_get_info.restype = C.c_int
        L.eicos_get_info.argtypes = [C.c_void_p, C.POINTER(Info)]
        L.eicos_cleanup.restype = None
        L.eicos_cleanup.argtypes = [C.c_void_p]
        L.eicos_batch_setup.restype = C.c_void_p
        L.eicos_batch_setup.argtypes = setup_args + [C.c_int, C.c_longlong, C.c_int]
        L.eicos_batch_setup_ex.restype = C.c_void_p
        L.eicos_batch_setup_ex.argtypes = setup_args + [C.c_int, C.c_longlong, C.c_int, C.c_int]
        L.eicos_batch_solve_matrices.restype = C.c_int
        L.eicos_batch_solve_matrices.argtypes = [C.c_void_p, C.c_int] + [_dp] * 9 + [_ip, C.POINTER(Info)]
        L.eicos_batch_update_matrices.restype = C.c_int
        L.eicos_batch_update_matrices.argtypes = [C.c_void_p, _dp, _dp]
        L.eicos_batch_solve.restype = C.c_int
        L.eicos_batch_solve.argtypes = [C.c_void_p, C.c_int] + [_dp] * 7 + [_ip, C.POINTER(Info)]
        L.eicos_batch_solve_device.restype = C.c_int
        L.eicos_batch_solve_device.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 9
        L.eicos_batch_solve_matrices_device.restype = C.c_int
        L.eicos_batch_solve_matrices_device.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 11
        L.eicos_batch_adjoint.restype = C.c_int
        L.eicos_batch_adjoint.argtypes = [C.c_void_p, C.c_int] + [_dp] * 6 + [_ip] + [_dp] * 8 + [_ip]
        L.eicos_batch_adjoint_device.restype = C.c_int
        L.eicos_batch_adjoint_device.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 16
        L.eicos_batch_tangent.restype = C.c_int
        L.eicos_batch_tangent.argtypes = [C.c_void_p, C.c_int] + [_dp] * 6 + [_ip] + [_dp] * 9 + [_ip]
        L.eicos_batch_tangent_device.restype = C.c_int
        L.eicos_batch_tangent_device.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 17
        L.eicos_batch_set_timing.restype = C.c_int
        L.eicos_batch_set_timing.argtypes = [C.c_void_p, C.c_int]
        L.eicos_batch_set_compaction.restype = C.c_int
        L.eicos_batch_set_compaction.argtypes = [C.c_void_p, C.c_int]
        L.eicos_batch_get_stats.restype = C.c_int
        L.eicos_batch_get_stats.argtypes = [C.c_void_p, C.POINTER(BatchStats)]
        L.eicos_batch_get_program_stats.restype = C.c_int
        L.eicos_batch_get_program_stats.argtypes = [C.c_void_p, C.POINTER(ProgramStats)]
        L.eicos_batch_get_dims.restype = C.c_int
        L.eicos_batch_get_dims.argtypes = [C.c_void_p, C.POINTER(BatchDims)]
        L.eicos_batch_get_symbolic.restype = C.c_int
        L.eicos_batch_get_symbolic.argtypes = [C.c_void_p] + [_ip] * 6
        L.eicos_batch_debug_init.restype = C.c_int
        L.eicos_batch_debug_init.argtypes = [C.c_void_p, C.c_int] + [_dp] * 7 + [_ip]
        L.eicos_batch_debug_set_iter_max.restype = C.c_int
        L.eicos_batch_debug_set_iter_max.argtypes = [C.c_void_p, C.c_int]
        L.eicos_batch_debug_line_search.restype = C.c_int
        L.eicos_batch_debug_line_search.argtypes = [C.c_void_p, C.c_int] + [_dp] * 5
        L.eicos_multi_setup.restype = C.c_void_p
        L.eicos_multi_setup.argtypes = setup_args + [C.c_int, _ip, C.c_longlong, C.c_int, C.c_int]
        L.eicos_multi_solve.restype = C.c_int
        L.eicos_multi_solve.argtypes = [C.c_void_p, C.c_int] + [_dp] * 9 + [_ip, C.POINTER(Info)]
        L.eicos_multi_ngpu.restype = C.c_int
        L.eicos_multi_ngpu.argtypes = [C.c_void_p]
        L.eicos_multi_slice.restype = C.c_int
        L.eicos_multi_slice.argtypes = [C.c_void_p, C.c_int, C.c_int, _ip, _ip]
        L.eicos_multi_cleanup.restype = None
        L.eicos_multi_cleanup.argtypes = [C.c_void_p]
        L.eicos_batch_stream.restype = C.c_void_p
        L.eicos_batch_stream.argtypes = [C.c_void_p]
        L.eicos_batch_cleanup.restype = None
        L.eicos_batch_cleanup.argtypes = [C.c_void_p]
        L.eicos_last_error.restype = C.c_char_p
        L.eicos_last_error.argtypes = []
        L.eicos_device_count.restype = C.c_int
        L.eicos_device_count.argtypes = []
        L.eicos_default_settings.restype = None
        L.eicos_default_settings.argtypes = [C.POINTER(Settings)]
        for kind in ("", "batch_", "multi_"):
            getattr(L, f"eicos_{kind}set_settings").restype = C.c_int
            getattr(L, f"eicos_{kind}set_settings").argtypes = [C.c_void_p, C.POINTER(Settings)]
            getattr(L, f"eicos_{kind}get_settings").restype = C.c_int
            getattr(L, f"eicos_{kind}get_settings").argtypes = [C.c_void_p, C.POINTER(Settings)]

    def last_error(self):
        return (self.L.eicos_last_error() or b"").decode()

    def check(self, rc):
        if rc != 0:
            raise RuntimeError(f"eicos_b200 error {rc}: {self.last_error()}")


_product = None


def load():
    """The product library (CUDA). Raises if it has not been built - no fallback."""
    global _product
    if _product is None:
        _product = Library(PRODUCT_LIB)
    return _product


def _problem_args(P):
    q = _arr(P.get("q"), np.int32)
    Gpr, Gjc, Gir = _arr(P.get("Gpr"), np.float64), _arr(P.get("Gjc"), np.int32), _arr(P.get("Gir"), np.int32)
    Apr, Ajc, Air = _arr(P.get("Apr"), np.float64), _arr(P.get("Ajc"), np.int32), _arr(P.get("Air"), np.int32)
    c, h, b = _arr(P.get("c"), np.float64), _arr(P.get("h"), np.float64), _arr(P.get("b"), np.float64)
    if Gpr is None:
        Gjc = Gir = None
    if Apr is None:
        Ajc = Air = None
    keep = [q, Gpr, Gjc, Gir, Apr, Ajc, Air, c, h, b]
    n, m, p = int(P["n"]), int(P["m"]), int(P["p"])
    args = [n, m, p, int(P.get("l", 0)), 0 if q is None else int(q.size),
            _i(q), _d(Gpr), _i(Gjc), _i(Gir), _d(Apr), _i(Ajc), _i(Air), _d(c), _d(h), _d(b)]
    return keep, args, (n, m if Gpr is not None else 0, p if Apr is not None else 0)


class Solver(_HasSettings):
    """Single-instance solver; same call sequence as EiCOS::Solver / the ECOS shim
    (reference test/ecos.h:11-34): Solver(problem) -> solve() -> update_data(...) -> solve()."""

    _GET, _SET = "eicos_get_settings", "eicos_set_settings"

    def __init__(self, problem, device=0, lib=None):
        self.lib = lib or load()
        self._keep, args, (self.n, self.m, self.p) = _problem_args(problem)
        self.h = self.lib.L.eicos_setup(*args, int(device))
        if not self.h:
            raise RuntimeError("eicos_setup failed: " + self.lib.last_error())

    def close(self):
        if getattr(self, "h", None):
            self.lib.L.eicos_cleanup(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def solve(self):
        return int(self.lib.L.eicos_solve(self.h))

    def update_data(self, Gpr=None, Apr=None, c=None, h=None, b=None, full=False):
        a = [_arr(v, np.float64) for v in (Gpr, Apr, c, h, b)]
        fn = self.lib.L.eicos_update_data_full if full else self.lib.L.eicos_update_data
        self.lib.check(fn(self.h, *[_d(v) for v in a]))

    def solution(self):
        ptr = self.lib.L.eicos_solution(self.h)
        return np.ctypeslib.as_array(ptr, shape=(self.n,)).copy() if self.n else np.zeros(0)

    def duals(self):
        y, z, s = np.zeros(self.p), np.zeros(self.m), np.zeros(self.m)
        self.lib.check(self.lib.L.eicos_get_duals(self.h, _d(y), _d(z), _d(s)))
        return y, z, s

    def info(self):
        i = Info()
        self.lib.check(self.lib.L.eicos_get_info(self.h, C.byref(i)))
        return i.asdict()


class BatchSolver(_HasSettings):
    """Batched overload: one pattern + shared G/A values, stacked per-instance c/h/b.
    instance_matrices=True: instances may also bring their own G/A values (solve(..., Gs=, As=))."""

    _GET, _SET = "eicos_batch_get_settings", "eicos_batch_set_settings"

    INSTANCE_MATRICES = 1

    def __init__(self, problem, device=0, capacity=0, workers=0, lib=None, instance_matrices=False):
        self.lib = lib or load()
        self.instance_matrices = bool(instance_matrices)
        self._keep, args, (self.n, self.m, self.p) = _problem_args(problem)
        self.h = self.lib.L.eicos_batch_setup_ex(*args, int(device), int(capacity), int(workers),
                                                 self.INSTANCE_MATRICES if instance_matrices else 0)
        if not self.h:
            raise RuntimeError("eicos_batch_setup failed: " + self.lib.last_error())
        d = self.dims()  # problems without G or A have no "Gpr" / "Apr" entry (or None): the handle knows
        self.nnzG, self.nnzA = d["nnzG"], d["nnzA"]

    def close(self):
        if getattr(self, "h", None):
            self.lib.L.eicos_batch_cleanup(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def dims(self):
        d = BatchDims()
        self.lib.check(self.lib.L.eicos_batch_get_dims(self.h, C.byref(d)))
        return d.asdict()

    def program_stats(self):
        p = ProgramStats()
        self.lib.check(self.lib.L.eicos_batch_get_program_stats(self.h, C.byref(p)))
        return p.asdict()

    def symbolic(self):
        d = self.dims()
        N, nnzK, nnzL = d["dim_K"], d["nnzK"], d["nnzL"]
        pinv, parent = np.zeros(N, np.int32), np.zeros(N, np.int32)
        Lp, Li = np.zeros(N + 1, np.int32), np.zeros(nnzL, np.int32)
        Kp, Ki = np.zeros(N + 1, np.int32), np.zeros(nnzK, np.int32)
        self.lib.check(self.lib.L.eicos_batch_get_symbolic(self.h, _i(pinv), _i(parent), _i(Lp), _i(Li), _i(Kp), _i(Ki)))
        return dict(pinv=pinv, parent=parent, Lp=Lp, Li=Li, Kp=Kp, Ki=Ki)

    def update_matrices(self, Gpr=None, Apr=None):
        a = [_arr(v, np.float64) for v in (Gpr, Apr)]
        self.lib.check(self.lib.L.eicos_batch_update_matrices(self.h, _d(a[0]), _d(a[1])))

    def set_timing(self, on=True):
        self.lib.check(self.lib.L.eicos_batch_set_timing(self.h, int(on)))

    def debug_set_iter_max(self, iter_max):
        """Test hook: cap the interior-point iterations at min(iter_max, 100) (0 = the reference's 100); the cap is
        settings()["iter_max"]."""
        self.lib.check(self.lib.L.eicos_batch_debug_set_iter_max(self.h, int(iter_max)))

    def set_compaction(self, on=True):
        self.lib.check(self.lib.L.eicos_batch_set_compaction(self.h, int(on)))

    def stats(self):
        s = BatchStats()
        self.lib.check(self.lib.L.eicos_batch_get_stats(self.h, C.byref(s)))
        return s.asdict()

    def stream(self):
        return self.lib.L.eicos_batch_stream(self.h)

    def solve(self, batch, cs=None, hs=None, bs=None, want=("x", "y", "z", "s"), want_info=True, Gs=None, As=None):
        """Host buffers in, host buffers out (copies included)."""
        cs, hs, bs, Gs, As = (_arr(v, np.float64) for v in (cs, hs, bs, Gs, As))
        for a, k in ((cs, self.n), (hs, self.m), (bs, self.p), (Gs, self.nnzG), (As, self.nnzA)):
            if a is not None and a.size != batch * k:
                raise ValueError("stacked vector has the wrong size")
        out = {}
        out["x"] = np.zeros((batch, self.n)) if "x" in want else None
        out["y"] = np.zeros((batch, self.p)) if "y" in want else None
        out["z"] = np.zeros((batch, self.m)) if "z" in want else None
        out["s"] = np.zeros((batch, self.m)) if "s" in want else None
        ex = np.zeros(batch, np.int32)
        info = (Info * batch)() if want_info else None
        self.lib.check(self.lib.L.eicos_batch_solve_matrices(
            self.h, int(batch), _d(Gs), _d(As), _d(cs), _d(hs), _d(bs),
            _d(out["x"]), _d(out["y"]), _d(out["z"]), _d(out["s"]), _i(ex), info))
        out["exit"] = ex
        if want_info:
            out["info"] = [info[k].asdict() for k in range(batch)]
            out["iter"] = np.array([i["iter"] for i in out["info"]], np.int32)
        return out

    def solve_device(self, batch, d_cs=0, d_hs=0, d_bs=0, d_x=0, d_y=0, d_z=0, d_s=0, d_exit=0, d_iter=0, d_Gs=0, d_As=0):
        """Raw device pointers (ints); results stay in HBM."""
        self.lib.check(self.lib.L.eicos_batch_solve_matrices_device(
            self.h, int(batch), *[C.c_void_p(int(v) or None) for v in (d_Gs, d_As, d_cs, d_hs, d_bs, d_x, d_y, d_z, d_s, d_exit, d_iter)]))

    ADJOINT_OUTPUTS = ("c", "h", "b", "G", "A")

    def adjoint(self, out, gx=None, gy=None, gz=None, Gs=None, As=None, want=ADJOINT_OUTPUTS):
        """Gradients of L(x, y, z) with respect to the problem data of the instances `out` = solve(...) returned
        (eicos_batch_adjoint): gx [batch x n], gy [batch x p], gz [batch x m] are dL/dx, dL/dy, dL/dz (None = zero);
        Gs / As: the forward's per-instance matrices (instance-matrices handles only; None = the setup values).
        Returns {"c": [batch x n], "h": [batch x m], "b": [batch x p], "G": [batch x nnzG], "A": [batch x nnzA]}
        for the names in `want`, and "status" [batch] (0 differentiated, 1 not optimal, 2 not interior, 3 not
        finite; instances with status != 0 get zeros)."""
        unknown = sorted(set(want) - set(self.ADJOINT_OUTPUTS))
        if unknown:
            raise ValueError(f"unknown adjoint outputs: {', '.join(unknown)}")
        batch = int(np.asarray(out["exit"]).size)
        sizes = {"x": self.n, "y": self.p, "z": self.m, "s": self.m}
        it = {k: np.ascontiguousarray(out[k], np.float64) for k in sizes}
        ex = np.ascontiguousarray(out["exit"], np.int32)
        g = {k: _arr(v, np.float64) for k, v in (("x", gx), ("y", gy), ("z", gz))}
        Gs, As = _arr(Gs, np.float64), _arr(As, np.float64)
        for k, a in it.items():
            if a.size != batch * sizes[k]:
                raise ValueError(f"out[{k!r}] has the wrong size")
        for k, a in g.items():
            if a is not None and a.size != batch * sizes[k]:
                raise ValueError(f"g{k} has the wrong size")
        for a, k in ((Gs, self.nnzG), (As, self.nnzA)):
            if a is not None and a.size != batch * k:
                raise ValueError("stacked matrix values have the wrong size")
        dims = {"c": self.n, "h": self.m, "b": self.p, "G": self.nnzG, "A": self.nnzA}
        res = {k: np.zeros((batch, dims[k])) if k in want else None for k in self.ADJOINT_OUTPUTS}
        status = np.zeros(batch, np.int32)
        self.lib.check(self.lib.L.eicos_batch_adjoint(
            self.h, batch, _d(Gs), _d(As), *[_d(it[k]) for k in "xyzs"], _i(ex), _d(g["x"]), _d(g["y"]), _d(g["z"]),
            *[_d(res[k]) for k in self.ADJOINT_OUTPUTS], _i(status)))
        res = {k: v for k, v in res.items() if v is not None}
        res["status"] = status
        return res

    def adjoint_device(self, batch, d_x=0, d_y=0, d_z=0, d_s=0, d_exit=0, d_gx=0, d_gy=0, d_gz=0,
                       d_dc=0, d_dh=0, d_db=0, d_dG=0, d_dA=0, d_status=0, d_Gs=0, d_As=0):
        """eicos_batch_adjoint_device on raw device pointers (ints, 0 = NULL); results stay in HBM."""
        self.lib.check(self.lib.L.eicos_batch_adjoint_device(
            self.h, int(batch), *[C.c_void_p(int(v) or None) for v in
                                  (d_Gs, d_As, d_x, d_y, d_z, d_s, d_exit, d_gx, d_gy, d_gz,
                                   d_dc, d_dh, d_db, d_dG, d_dA, d_status)]))

    TANGENT_OUTPUTS = ("x", "y", "z", "s")

    def tangent(self, out, dc=None, dh=None, db=None, dG=None, dA=None, Gs=None, As=None, want=TANGENT_OUTPUTS):
        """Derivatives of the solutions `out` = solve(...) returned along a direction in the problem data
        (eicos_batch_tangent): dc [batch x n], dh [batch x m], db [batch x p], dG [batch x nnzG], dA [batch x nnzA]
        (CSC order; both kinds of handle); None = zero.  Gs / As: the forward's per-instance matrices
        (instance-matrices handles only; None = the setup values).
        Returns {"x": [batch x n], "y": [batch x p], "z": [batch x m], "s": [batch x m]} for the names in `want`, and
        "status" [batch] (0 differentiated, 1 not optimal, 2 not interior, 3 not finite; instances with status != 0
        get zeros)."""
        unknown = sorted(set(want) - set(self.TANGENT_OUTPUTS))
        if unknown:
            raise ValueError(f"unknown tangent outputs: {', '.join(unknown)}")
        batch = int(np.asarray(out["exit"]).size)
        sizes = {"x": self.n, "y": self.p, "z": self.m, "s": self.m}
        it = {k: np.ascontiguousarray(out[k], np.float64) for k in sizes}
        ex = np.ascontiguousarray(out["exit"], np.int32)
        dims = {"c": self.n, "h": self.m, "b": self.p, "G": self.nnzG, "A": self.nnzA}
        v = {k: _arr(a, np.float64) for k, a in (("c", dc), ("h", dh), ("b", db), ("G", dG), ("A", dA))}
        Gs, As = _arr(Gs, np.float64), _arr(As, np.float64)
        for k, a in it.items():
            if a.size != batch * sizes[k]:
                raise ValueError(f"out[{k!r}] has the wrong size")
        for k, a in v.items():
            if a is not None and a.size != batch * dims[k]:
                raise ValueError(f"d{k} has the wrong size")
        for a, k in ((Gs, self.nnzG), (As, self.nnzA)):
            if a is not None and a.size != batch * k:
                raise ValueError("stacked matrix values have the wrong size")
        res = {k: np.zeros((batch, sizes[k])) if k in want else None for k in self.TANGENT_OUTPUTS}
        status = np.zeros(batch, np.int32)
        self.lib.check(self.lib.L.eicos_batch_tangent(
            self.h, batch, _d(Gs), _d(As), *[_d(it[k]) for k in "xyzs"], _i(ex),
            *[_d(v[k]) for k in ("c", "h", "b", "G", "A")], *[_d(res[k]) for k in self.TANGENT_OUTPUTS], _i(status)))
        res = {k: a for k, a in res.items() if a is not None}
        res["status"] = status
        return res

    def tangent_device(self, batch, d_x=0, d_y=0, d_z=0, d_s=0, d_exit=0, d_dc=0, d_dh=0, d_db=0, d_dG=0, d_dA=0,
                       d_ox=0, d_oy=0, d_oz=0, d_os=0, d_status=0, d_Gs=0, d_As=0):
        """eicos_batch_tangent_device on raw device pointers (ints, 0 = NULL); results (d_ox .. d_os = dx, dy, dz,
        ds) stay in HBM."""
        self.lib.check(self.lib.L.eicos_batch_tangent_device(
            self.h, int(batch), *[C.c_void_p(int(v) or None) for v in
                                  (d_Gs, d_As, d_x, d_y, d_z, d_s, d_exit, d_dc, d_dh, d_db, d_dG, d_dA,
                                   d_ox, d_oy, d_oz, d_os, d_status)]))

    def debug_line_search(self, lam, ds, dz, scalars):
        """lineSearch on caller data: lam, ds, dz [batch x m] in z order, scalars [batch x 4] = tau, dtau, kap, dkap."""
        lam, ds, dz, scalars = (np.ascontiguousarray(v, np.float64) for v in (lam, ds, dz, scalars))
        alpha = np.zeros(lam.shape[0])
        self.lib.check(self.lib.L.eicos_batch_debug_line_search(self.h, int(lam.shape[0]), _d(lam), _d(ds), _d(dz), _d(scalars), _d(alpha)))
        return alpha

    def debug_init(self, batch, cs=None, hs=None, bs=None):
        d = self.dims()
        cs, hs, bs = (_arr(v, np.float64) for v in (cs, hs, bs))
        Lx, D = np.zeros((batch, d["nnzL"])), np.zeros((batch, d["dim_K"]))
        s1, s2 = np.zeros((batch, d["dim_K"])), np.zeros((batch, d["dim_K"]))
        nit = np.zeros((batch, 2), np.int32)
        self.lib.check(self.lib.L.eicos_batch_debug_init(self.h, int(batch), _d(cs), _d(hs), _d(bs),
                                                         _d(Lx), _d(D), _d(s1), _d(s2), _i(nit)))
        return dict(Lx=Lx, D=D, sol1=s1, sol2=s2, nitref=nit)


class MultiBatchSolver(_HasSettings):
    """The batched overload over several GPUs of one node (eicos_multi_*): contiguous slices of the batch, one
    device and one host thread each, results gathered into the caller's arrays; no collective."""

    _GET, _SET = "eicos_multi_get_settings", "eicos_multi_set_settings"

    def __init__(self, problem, devices=(0,), capacity=0, workers=0, lib=None, instance_matrices=False):
        self.lib = lib or load()
        self._keep, args, (self.n, self.m, self.p) = _problem_args(problem)
        dev = np.ascontiguousarray(list(devices), dtype=np.int32)
        self.h = self.lib.L.eicos_multi_setup(*args, int(dev.size), _i(dev), int(capacity), int(workers),
                                              BatchSolver.INSTANCE_MATRICES if instance_matrices else 0)
        if not self.h:
            raise RuntimeError("eicos_multi_setup failed: " + self.lib.last_error())

    def close(self):
        if getattr(self, "h", None):
            self.lib.L.eicos_multi_cleanup(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def ngpu(self):
        return int(self.lib.L.eicos_multi_ngpu(self.h))

    def slice(self, batch, k):
        first, count = C.c_int(), C.c_int()
        self.lib.check(self.lib.L.eicos_multi_slice(self.h, int(batch), int(k), C.byref(first), C.byref(count)))
        return first.value, count.value

    def solve(self, batch, cs=None, hs=None, bs=None, Gs=None, As=None):
        a = [_arr(v, np.float64) for v in (Gs, As, cs, hs, bs)]
        x, y = np.zeros((batch, self.n)), np.zeros((batch, self.p))
        z, s = np.zeros((batch, self.m)), np.zeros((batch, self.m))
        ex = np.zeros(batch, np.int32)
        info = (Info * batch)()
        self.lib.check(self.lib.L.eicos_multi_solve(self.h, int(batch), *[_d(v) for v in a], _d(x), _d(y), _d(z), _d(s), _i(ex), info))
        return dict(x=x, y=y, z=z, s=s, exit=ex, iter=np.array([i.iter for i in info], np.int32), info=info)
