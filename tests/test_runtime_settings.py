"""Solver settings per handle (eicos_settings; Solver / BatchSolver / MultiBatchSolver .settings() and
.set_settings()): tolerances, iteration limit, refinement and step control are values every kernel reads at run
time instead of compile-time constants.

The CPU tier runs the kernel sources on the emulator (tests/emu); the gpu tier runs the CUDA library.  Results
under non-default settings are compared with the CPU oracle under the same settings.  The oracle source
(oracle/eicos_oracle.cpp) holds the reference's settings as constants and stays exactly as every other parity test
uses it, so `settings_oracle` compiles a private copy of it in which only those constants are assignable and
checks that the copy at the default values reproduces the stock oracle bit for bit."""
import ctypes as C
import importlib.util
import os
import re
import subprocess
import struct

import numpy as np
import pytest

from conftest import ROOT, relerr

TOL = 1e-7
DEFAULTS = dict(feastol=1e-8, abstol=1e-8, reltol=1e-8, feastol_inacc=1e-4, abstol_inacc=5e-5, reltol_inacc=5e-5,
                linsysacc=1e-14, irerrfact=6.0, gamma=0.99, stepmin=1e-6, stepmax=0.999, sigmamin=1e-4, sigmamax=1.0,
                safeguard=500.0, nitref=9, iter_max=100)
CASES = {
    "a_loose": dict(feastol=1e-6, abstol=1e-6, reltol=1e-6, feastol_inacc=1e-3, abstol_inacc=1e-3, reltol_inacc=1e-3),
    "b_iter7": dict(iter_max=7),
    "c_refine": dict(nitref=1, linsysacc=1e-10, irerrfact=3.0),
    "d_step": dict(gamma=0.95, stepmin=1e-5, stepmax=0.98, sigmamin=1e-3, sigmamax=0.9),
    "e_safeguard": dict(safeguard=50.0),
}
KEYS = ("x", "y", "z", "s", "exit", "iter", "nitref1", "nitref2", "nitref3")


# ------------------------------------------------------------------ oracle under settings
ORACLE_CONSTANTS = [
    "static const double GAMMA = 0.99, DELTASTAT = 7e-8;",
    "static const double FEASTOL = 1e-8, ABSTOL = 1e-8, RELTOL = 1e-8;",
    "static const double FEASTOL_INACC = 1e-4, ABSTOL_INACC = 5e-5, RELTOL_INACC = 5e-5;",
    "static const int NITREF = 9, EQUIL_ITERS = 3, ITER_MAX = 100;",
    "static const double LINSYSACC = 1e-14, IRERRFACT = 6, STEPMIN = 1e-6, STEPMAX = 0.999;",
    "static const double SIGMAMIN = 1e-4, SIGMAMAX = 1.0, SAFEGUARD = 500;",
]
ORACLE_SETTER = """
extern "C" void ora_test_set_settings(const double *d, const int *i)
{
    ora::FEASTOL = d[0], ora::ABSTOL = d[1], ora::RELTOL = d[2];
    ora::FEASTOL_INACC = d[3], ora::ABSTOL_INACC = d[4], ora::RELTOL_INACC = d[5];
    ora::LINSYSACC = d[6], ora::IRERRFACT = d[7], ora::GAMMA = d[8], ora::STEPMIN = d[9], ora::STEPMAX = d[10];
    ora::SIGMAMIN = d[11], ora::SIGMAMAX = d[12], ora::SAFEGUARD = d[13];
    ora::NITREF = i[0], ora::ITER_MAX = i[1];
}
"""
DOUBLES = ("feastol", "abstol", "reltol", "feastol_inacc", "abstol_inacc", "reltol_inacc", "linsysacc", "irerrfact",
           "gamma", "stepmin", "stepmax", "sigmamin", "sigmamax", "safeguard")


class SettingsOracle:
    """The oracle with assignable settings; solve() runs each instance as a fresh OracleSolver."""

    def __init__(self, mod):
        self.mod = mod

    def set(self, **fields):
        s = dict(DEFAULTS, **fields)
        d = (C.c_double * 14)(*[s[k] for k in DOUBLES])
        i = (C.c_int * 2)(s["nitref"], s["iter_max"])
        self.mod.lib().ora_test_set_settings(d, i)

    def solve(self, P, W, **fields):
        self.set(**fields)
        Gs, As, hs, bs = (W.get(k) for k in ("Gs", "As", "hs", "bs"))
        batch = next(len(v) for v in (Gs, As, hs, bs) if v is not None)
        rows = []
        for k in range(batch):
            Pk = dict(P)
            for key, st in (("Gpr", Gs), ("Apr", As), ("h", hs), ("b", bs)):
                if st is not None:
                    Pk[key] = st[k]
            O = self.mod.OracleSolver(Pk)
            code = O.solve()
            x, y, z, s = O.solution()
            rows.append((x, y, z, s, code, O.info()))
            O.close()
        self.set()
        out = {k: np.array([r[i] for r in rows]) for i, k in enumerate("xyzs")}
        out["exit"] = np.array([r[4] for r in rows], np.int32)
        for k in ("iter", "nitref1", "nitref2", "nitref3"):
            out[k] = np.array([r[5][k] for r in rows], np.int32)
        return out


@pytest.fixture(scope="session")
def settings_oracle(oracle_mod, tmp_path_factory):
    src = open(os.path.join(ROOT, "oracle", "eicos_oracle.cpp")).read()
    for line in ORACLE_CONSTANTS:
        assert src.count(line) == 1, f"oracle settings block changed: {line}"
        src = src.replace(line, line.replace("static const", "static"))
    d = tmp_path_factory.mktemp("settings_oracle")
    cpp, so = d / "eicos_oracle_settings.cpp", d / "libeicos_oracle_settings.so"
    cpp.write_text(src + ORACLE_SETTER)
    flags = re.search(r"CXXFLAGS \?= (.*)", open(os.path.join(ROOT, "oracle", "Makefile")).read()).group(1).split()
    subprocess.check_call(["g++"] + flags + ["-I", os.path.join(ROOT, "oracle"), "-shared", "-o", str(so), str(cpp)])
    spec = importlib.util.spec_from_file_location("oracle_with_settings", os.path.join(ROOT, "oracle", "oracle.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.LIB, mod._lib = str(so), None
    mod.lib().ora_test_set_settings.restype = None
    return SettingsOracle(mod)


# ------------------------------------------------------------------ problems
def _problem(name):
    import oracle
    from eicos_b200.workloads import perturbed, perturbed_matrices, soc_mpc, soc_mpc_batch
    if name == "MPC02":
        P = oracle.load_fixture("MPC02")
        return P, perturbed(P, 12, rel={"h": 0.002, "b": 0.02}, seed=5), False
    if name == "MPC02_5pc":  # +-5 %: some instances are primal infeasible, so the certificate tests run
        P = oracle.load_fixture("MPC02")
        return P, perturbed(P, 12, rel=0.05, seed=5), False
    if name == "socmpc":
        P = soc_mpc(T=6)
        return P, soc_mpc_batch(P, 12), False
    if name == "lp_afiro":
        P = oracle.load_fixture("lp_afiro")
        return P, perturbed(P, 8, rel=0.02, seed=5), False
    if name == "pim":
        P = oracle.load_fixture("update_data_1")
        return P, perturbed_matrices(P, 8, rel=0.02, seed=3), True
    raise KeyError(name)


def _engine(lib, P, W, pim=False, settings=None, capacity=None, **kw):
    from eicos_b200.binding import BatchSolver
    batch = next(len(v) for v in (W.get("Gs"), W.get("As"), W.get("hs"), W.get("bs")) if v is not None)
    B = BatchSolver(P, lib=lib, capacity=capacity or batch, instance_matrices=pim, **kw)
    if settings:
        B.set_settings(**settings)
    out = B.solve(batch, hs=W.get("hs"), bs=W.get("bs"), Gs=W.get("Gs"), As=W.get("As"))
    for k in ("nitref1", "nitref2", "nitref3", "iter_max"):
        out[k] = np.array([i[k] for i in out["info"]], np.int32)
    B.close()
    return out


def _assert_parity(out, ref, duals=True):
    """test_batched_perturbed_parity's acceptance, plus refinement counts (nitref3 may differ by one round on a
    near-tie of the stopping rule)."""
    assert np.array_equal(out["exit"], ref["exit"]), (out["exit"], ref["exit"])
    assert np.array_equal(out["iter"], ref["iter"]), (out["iter"], ref["iter"])
    assert np.array_equal(out["nitref1"], ref["nitref1"]) and np.array_equal(out["nitref2"], ref["nitref2"])
    assert np.max(np.abs(out["nitref3"] - ref["nitref3"])) <= 1
    ok = np.isin(ref["exit"], (0, 10, -1))  # certificates of infeasibility are not solutions
    for k in ("xyzs" if duals else "xs"):
        if ok.any():
            assert relerr(out[k][ok], ref[k][ok]) <= TOL, k


def _assert_bits(a, b):
    for k in KEYS:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k


# ------------------------------------------------------------------ CPU tier (emulator)
def test_defaults(emu_lib):
    from eicos_b200.binding import BatchSolver, Solver, default_settings
    import oracle
    assert default_settings(emu_lib) == DEFAULTS
    P = oracle.load_fixture("lp_afiro")
    B = BatchSolver(P, lib=emu_lib, capacity=4)
    assert B.settings() == DEFAULTS
    new = dict(CASES["a_loose"], **CASES["c_refine"], **CASES["d_step"], safeguard=50.0, iter_max=300)
    B.set_settings(**new)
    assert B.settings() == dict(DEFAULTS, **new)
    S = Solver(P, lib=emu_lib)
    assert S.settings() == DEFAULTS
    S.set_settings(iter_max=12)
    assert S.settings() == dict(DEFAULTS, iter_max=12)


def test_settings_oracle_at_defaults_is_the_oracle(oracle_mod, settings_oracle):
    P, W, _ = _problem("MPC02_5pc")
    ref = oracle_mod.batch_run(P, 12, hs=W["hs"], bs=W["bs"])
    mine = settings_oracle.solve(P, W)
    for k in ("x", "y", "z", "s", "exit", "iter"):
        assert np.array_equal(mine[k], ref[k]), k


@pytest.mark.parametrize("name", ["MPC02", "socmpc", "lp_afiro"])
def test_explicit_defaults_change_nothing(emu_lib, name):
    import oracle
    from eicos_b200.workloads import perturbed, soc_mpc, soc_mpc_batch
    # the workloads of test_vector_passes.py
    if name == "MPC02":
        P = oracle.load_fixture("MPC02")
        W = perturbed(P, 64, rel={"h": 0.002, "b": 0.02}, seed=5)
    elif name == "socmpc":
        P = soc_mpc(T=12)
        W = soc_mpc_batch(P, 32)
    else:
        P = oracle.load_fixture("lp_afiro")
        W = perturbed(P, 16, rel=0.02, seed=5)
    _assert_bits(_engine(emu_lib, P, W, settings=DEFAULTS, workers=3), _engine(emu_lib, P, W, workers=3))


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("name", ["MPC02", "MPC02_5pc", "socmpc", "lp_afiro", "pim"])
def test_parity_under_settings(emu_lib, settings_oracle, name, case):
    P, W, pim = _problem(name)
    out = _engine(emu_lib, P, W, pim=pim, settings=CASES[case])
    ref = settings_oracle.solve(P, W, **CASES[case])
    _assert_parity(out, ref, duals=name != "socmpc")


def test_settings_take_effect(emu_lib):
    import oracle
    from eicos_b200.workloads import perturbed
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 24, rel={"h": 0.002, "b": 0.02}, seed=9)
    base = _engine(emu_lib, P, W)
    loose = _engine(emu_lib, P, W, settings=CASES["a_loose"])
    assert loose["iter"].mean() < base["iter"].mean()
    assert np.isin(loose["exit"], (0, 10)).all()
    capped = _engine(emu_lib, P, W, settings=dict(iter_max=7))
    long_ = base["iter"] > 7
    assert long_.any()
    assert (capped["exit"][long_] == -1).all() and (capped["iter"][long_] == 7).all()
    assert (capped["iter_max"] == 7).all() and (base["iter_max"] == 100).all()
    nr = _engine(emu_lib, P, W, settings=dict(nitref=0))
    for k in ("nitref1", "nitref2", "nitref3"):
        assert (nr[k] == 0).all(), k
    assert (base["nitref1"] > 0).any()


BAD = [("feastol", 0.0), ("abstol", -1e-8), ("reltol", float("nan")), ("feastol_inacc", float("inf")),
       ("abstol_inacc", 0.0), ("reltol_inacc", -1.0), ("linsysacc", 0.0), ("irerrfact", -6.0),
       ("gamma", 0.0), ("gamma", 1.01), ("stepmin", 0.0), ("stepmin", 0.9995), ("stepmax", 1.5),
       ("sigmamin", -1e-4), ("sigmamin", 0.5, dict(sigmamax=0.4)), ("sigmamax", 1.01), ("safeguard", 0.5),
       ("nitref", -1), ("nitref", 33), ("iter_max", 0), ("iter_max", 1001)]


def test_bad_input_is_rejected(emu_lib):
    import oracle
    from eicos_b200.binding import BatchSolver, MultiBatchSolver, Solver
    P = oracle.load_fixture("lp_afiro")
    handles = [BatchSolver(P, lib=emu_lib, capacity=2), Solver(P, lib=emu_lib), MultiBatchSolver(P, lib=emu_lib, capacity=2)]
    good = dict(iter_max=50, gamma=0.9)
    for H in handles:
        H.set_settings(**good)
        for bad in BAD:
            field, value = bad[0], bad[1]
            extra = bad[2] if len(bad) > 2 else {}
            with pytest.raises(RuntimeError, match=rf"eicos_settings\.{field}\b"):
                H.set_settings(**{field: value}, **extra)
            assert H.settings() == dict(DEFAULTS, **good), bad
        with pytest.raises(ValueError, match="maxit"):
            H.set_settings(maxit=5)
        H.set_settings(stepmin=0.5, stepmax=0.5, sigmamin=0.0, sigmamax=0.0, gamma=1.0, safeguard=1.0, nitref=32, iter_max=1000)


def test_settings_persist(emu_lib):
    """Over repeated solves, update_matrices and chunking: 160 instances at capacity 64 equal capacity 160."""
    import oracle
    from eicos_b200.binding import BatchSolver
    from eicos_b200.workloads import perturbed
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 160, rel={"h": 0.002, "b": 0.02}, seed=13)
    st = dict(CASES["a_loose"], **CASES["c_refine"])
    whole = _engine(emu_lib, P, W, settings=st, capacity=160)
    B = BatchSolver(P, lib=emu_lib, capacity=64)
    B.set_settings(**st)
    for _ in range(2):
        out = B.solve(160, hs=W["hs"], bs=W["bs"])
        for k in ("nitref1", "nitref2", "nitref3"):
            out[k] = np.array([i[k] for i in out["info"]], np.int32)
        _assert_bits(out, whole)
    B.update_matrices(P["Gpr"], P["Apr"])
    assert B.settings() == dict(DEFAULTS, **st)
    out = B.solve(160, hs=W["hs"], bs=W["bs"])
    for k in "xyzs":
        assert np.array_equal(out[k], whole[k]), k


def test_every_form_reads_the_settings(emu_lib, monkeypatch):
    """Shallow or deep ring, one- or two-job solves, one-warp or wide kernels: a form that still read a
    compile-time constant would part from the others here."""
    import oracle
    from eicos_b200.workloads import perturbed
    P = oracle.load_fixture("update_data_1")
    W = perturbed(P, 5, rel=0.05, seed=11)
    st = dict(CASES["a_loose"], **CASES["c_refine"])
    outs = []
    for ring, pair, wide in (("0", "0", "0"), ("1", "0", "0"), ("0", "1", "0"), ("0", "0", "1")):
        monkeypatch.setenv("EICOS_RING_VARIANT", ring)
        monkeypatch.setenv("EICOS_PAIR_SOLVES", pair)
        monkeypatch.setenv("EICOS_WIDE", wide)
        outs.append(_engine(emu_lib, P, W, settings=st))
    for o in outs[1:]:
        _assert_bits(o, outs[0])
    monkeypatch.delenv("EICOS_RING_VARIANT")
    monkeypatch.delenv("EICOS_PAIR_SOLVES")
    monkeypatch.delenv("EICOS_WIDE")
    base = _engine(emu_lib, P, W)
    assert any(not np.array_equal(outs[0][k], base[k]) for k in KEYS)  # the settings do change the results


def _multi_equals_single(lib, devices):
    import oracle
    from eicos_b200.binding import MultiBatchSolver
    from eicos_b200.workloads import perturbed
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 20, rel=0.05, seed=17)
    st = dict(CASES["a_loose"], **CASES["d_step"])
    M = MultiBatchSolver(P, devices=devices, lib=lib, capacity=16)
    M.set_settings(**st)
    assert M.settings() == dict(DEFAULTS, **st)
    multi = M.solve(20, hs=W["hs"], bs=W["bs"])
    single = _engine(lib, P, W, settings=st)
    for k in ("x", "y", "z", "s", "exit", "iter"):
        assert np.array_equal(multi[k], single[k]), k


def test_multi_equals_single(emu_lib):
    _multi_equals_single(emu_lib, (0, 0))


def _single_instance(lib, settings_oracle):
    import oracle
    from eicos_b200.binding import Solver
    P1, P2 = oracle.load_fixture("update_data_1"), oracle.load_fixture("update_data_2")
    st = dict(CASES["a_loose"], **CASES["c_refine"], **CASES["d_step"])
    S = Solver(P1, lib=lib)
    S.set_settings(**st)
    for P in (P1, P2):
        if P is P2:
            S.update_data(P["Gpr"], P["Apr"], P["c"], P["h"], P["b"], full=True)
            assert S.settings() == dict(DEFAULTS, **st)
        code = S.solve()
        ref = settings_oracle.solve(P, {"hs": P["h"][None, :]}, **st)
        info = S.info()
        assert code == ref["exit"][0] and info["iter"] == ref["iter"][0] and info["iter_max"] == 100
        assert info["nitref1"] == ref["nitref1"][0] and info["nitref2"] == ref["nitref2"][0]
        assert relerr(S.solution(), ref["x"][0]) <= TOL


def test_single_instance(emu_lib, settings_oracle):
    _single_instance(emu_lib, settings_oracle)


def test_iter_max_hook(emu_lib):
    import oracle
    from eicos_b200.binding import BatchSolver
    B = BatchSolver(oracle.load_fixture("lp_afiro"), lib=emu_lib, capacity=2)
    B.debug_set_iter_max(9)
    assert B.settings()["iter_max"] == 9
    B.debug_set_iter_max(500)  # the hook caps at the reference's 100
    assert B.settings()["iter_max"] == 100
    B.set_settings(iter_max=400)
    B.debug_set_iter_max(0)
    assert B.settings()["iter_max"] == 100


# ------------------------------------------------------------------ C++ facade
def _facade(binary, tmp_path, settings):
    import oracle
    from eicos_b200.workloads import perturbed
    P = oracle.load_fixture("MPC02")
    W = perturbed(P, 6, rel=0.05, seed=21)
    s = dict(DEFAULTS, **settings)
    n, m, p = int(P["n"]), int(P["m"]), int(P["p"])
    f64 = lambda a: np.ascontiguousarray(a, np.float64).tobytes()
    i32 = lambda a: np.ascontiguousarray(a, np.int32).tobytes()
    q = np.asarray(P["q"], np.int32) if P.get("q") is not None else np.zeros(0, np.int32)
    script = tmp_path / "settings.bin"
    with open(script, "wb") as f:
        f.write(struct.pack("<7i", n, m, p, int(P.get("l", 0)), q.size, np.size(P["Gpr"]), np.size(P["Apr"])))
        f.write(i32(q) + i32(P["Gjc"]) + i32(P["Gir"]) + i32(P["Ajc"]) + i32(P["Air"]))
        f.write(f64(P["Gpr"]) + f64(P["Apr"]) + f64(P["c"]) + f64(P["h"]) + f64(P["b"]))
        f.write(f64([s[k] for k in DOUBLES]) + i32([s["nitref"], s["iter_max"]]))
        f.write(struct.pack("<i", 6) + f64(W["hs"]) + f64(W["bs"]))
    run = subprocess.run([binary, str(script)], capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stderr
    lines = [l.split() for l in run.stdout.splitlines()]
    bits = lambda t: np.array([int(v, 16) for v in t[1:]], np.uint64).view(np.float64)
    single = dict(exit=int(lines[0][1]), iter=int(lines[0][2]), iter_max=int(lines[0][3]), x=bits(lines[1]))
    batch = [(list(map(int, lines[2 + 3 * k][1:])), bits(lines[3 + 3 * k]), bits(lines[4 + 3 * k])) for k in range(6)]
    assert lines[-1] == ["rejected", "gamma"]
    return P, W, single, batch


def _build_driver(lib, tmp_path):
    """tests/cpp/settings_driver.cpp linked against `lib` (the emulator or the CUDA library), built in tmp_path."""
    libdir, name = os.path.split(lib.path)
    out = str(tmp_path / "settings_driver")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-Wextra", "-I", os.path.join(ROOT, "include"),
                           "-o", out, os.path.join(ROOT, "tests", "cpp", "settings_driver.cpp"),
                           "-L", libdir, "-l" + name[3:-3], "-Wl,-rpath," + libdir])
    return out


def _facade_matches_python(lib, binary, tmp_path):
    from eicos_b200.binding import Solver
    st = dict(CASES["a_loose"], **CASES["c_refine"], iter_max=40)
    P, W, single, batch = _facade(binary, tmp_path, st)
    S = Solver(P, lib=lib)
    S.set_settings(**st)
    assert single["exit"] == S.solve() and single["iter"] == S.info()["iter"] and single["iter_max"] == 40
    assert np.array_equal(single["x"], S.solution())
    out = _engine(lib, P, W, settings=st)
    for k, (ints, x, z) in enumerate(batch):
        assert ints == [out["exit"][k], out["iter"][k], 40, out["nitref1"][k], out["nitref2"][k], out["nitref3"][k]]
        assert np.array_equal(x, out["x"][k]) and np.array_equal(z, out["z"][k])


def test_cpp_facade_settings(emu_lib, tmp_path):
    _facade_matches_python(emu_lib, _build_driver(emu_lib, tmp_path), tmp_path)


# ------------------------------------------------------------------ gpu tier (CUDA library)
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["MPC02", "socmpc"])
def test_gpu_explicit_defaults_change_nothing(gpu_lib, name):
    P, W, _ = _problem(name)
    _assert_bits(_engine(gpu_lib, P, W, settings=DEFAULTS), _engine(gpu_lib, P, W))


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("name", ["MPC02", "MPC02_5pc", "socmpc"])
def test_gpu_parity_under_settings(gpu_lib, settings_oracle, name, case):
    P, W, pim = _problem(name)
    _assert_parity(_engine(gpu_lib, P, W, pim=pim, settings=CASES[case]), settings_oracle.solve(P, W, **CASES[case]),
                   duals=name != "socmpc")


@pytest.mark.gpu
def test_gpu_settings_take_effect(gpu_lib):
    test_settings_take_effect(gpu_lib)


@pytest.mark.gpu
def test_gpu_every_form_reads_the_settings(gpu_lib, monkeypatch):
    test_every_form_reads_the_settings(gpu_lib, monkeypatch)


@pytest.mark.gpu
def test_gpu_multi_same_device_twice(gpu_lib):
    _multi_equals_single(gpu_lib, (0, 0))


@pytest.mark.gpu
def test_gpu_single_instance(gpu_lib, settings_oracle):
    _single_instance(gpu_lib, settings_oracle)


@pytest.mark.gpu
def test_gpu_cpp_facade_settings(gpu_lib, tmp_path):
    _facade_matches_python(gpu_lib, _build_driver(gpu_lib, tmp_path), tmp_path)
