"""The 18 tests of the reference's tester (test/ecostester.cpp of EmbersArc/EiCOS, minus MPC01, whose data the
reference does not contain), run on the engine.  Each sets one fixture up through the ECOS C names, solves it and
asserts the exit flag the reference asserts.  The fixture data and those exit flags were taken from the reference's
test headers (tests/golden/make_fixtures.py) and are stored under tests/golden/fixtures; here they are written back
as headers in the reference's format (eicos_b200/ecos_format.py) under the reference's file names, compiled with
oracle/ref_tester_main.cpp against the ECOS-name shim (tests/cpp/shim) and run on the kernel emulator and on the
CUDA library."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import EMU_LIB, ROOT

TESTS = ["MPC02", "update_data", "unboundedLP1", "unboundedMaxSqrt", "feas", "infeasible1", "lp_25fv47",
         "lp_adlittle", "lp_afiro", "lp_agg", "lp_agg2", "lp_agg3", "lp_bandm", "lp_beaconfd", "lp_blend",
         "lp_bnl1", "emptyProblem", "issue98"]
# The ONE expectation of the reference's tester that is not reproduced (DESIGN.md section 6): unboundedMaxSqrt
# expects DINF; the double-precision runs (oracle, emulator, GPU alike) miss `dinfres < feastol` by 15 % (closest
# approach 1.15e-8) and end in the pres safeguard with NUMERICS, while the same algorithm in extended precision
# reaches DINF (tests/test_oracle.py::test_unbounded_maxsqrt_is_a_rounding_knife_edge prints the margins).
CHAOTIC = {"unboundedMaxSqrt"}
FLAG = {0: "ECOS_OPTIMAL", 1: "ECOS_PINF", 2: "ECOS_DINF", 10: "ECOS_OPTIMAL + ECOS_INACC_OFFSET"}
_BINARIES = {}


def _accepts(codes):
    """The exit flags a reference test accepts, as the right-hand side of write_header's `exitflag == ...`."""
    return " || exitflag == ".join(FLAG[c] for c in codes)


def _update_data_header(oracle_mod):
    """test/updateData/update_data.h: set up with the first data set, solve, updateData with all of the second
    (G, A, c, h, b), solve again; both solves must end optimal."""
    from eicos_b200 import ecos_format as ef
    P1, P2 = oracle_mod.load_fixture("update_data_1"), oracle_mod.load_fixture("update_data_2")
    ok = _accepts(P1["expect"])
    arg = lambda pre, P, k: f"{pre}_{k}" if np.asarray(P[k]).size else "NULL"
    setup = ", ".join(arg("udd1", P1, k) for k in ("Gpr", "Gjc", "Gir", "Apr", "Ajc", "Air", "c", "h", "b"))
    update = ", ".join(arg("udd2", P2, k) for k in ("Gpr", "Apr", "c", "h", "b"))
    return "\n".join([ef.write_header(P1, "udd1"), ef.write_header(P2, "udd2"), f"""
static char *test_update_data()
{{
    idxint exitflag = ECOS_FATAL;
    pwork *mywork = ECOS_setup({P1['n']}, {P1['m']}, {P1['p']}, {P1['l']}, {P1['ncones']}, {arg("udd1", P1, "q")}, 0, {setup});
    mu_assert("update_data: setup failed", mywork != NULL);
    exitflag = ECOS_solve(mywork);
    mu_assert("update_data: unexpected exit flag of the first solve", exitflag == {ok});
    ECOS_updateData(mywork, {update});
    exitflag = ECOS_solve(mywork);
    mu_assert("update_data: unexpected exit flag after updateData", exitflag == {ok});
    ECOS_cleanup(mywork, 0);
    return 0;
}}
"""])


def _binary(kind, oracle_mod, tmp_path_factory):
    """oracle/ref_tester_main.cpp with the fixture headers, linked with the emulator ("emu") or the CUDA library."""
    if kind in _BINARIES:
        return _BINARIES[kind]
    from eicos_b200 import ecos_format as ef
    from eicos_b200.binding import PRODUCT_LIB
    work = tmp_path_factory.mktemp("ref_tester")
    with open(os.path.join(ROOT, "tests", "golden", "fixtures", "manifest.json")) as f:
        manifest = json.load(f)
    for name in TESTS:
        if name == "update_data":
            rel, text = "updateData/update_data.h", _update_data_header(oracle_mod)
        else:
            P = oracle_mod.load_fixture(name)
            rel = manifest[name]["source"].split(":")[0][len("test/"):]
            text = ef.write_header(P, name, _accepts(P["expect"]))
        (work / rel).parent.mkdir(parents=True, exist_ok=True)
        (work / rel).write_text(text)
    libdir, lib = ((os.path.dirname(EMU_LIB), "eicos_emu") if kind == "emu" else
                   (os.path.dirname(PRODUCT_LIB), "eicos_b200"))
    exe = str(work / f"ecostester_{kind}")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-w", "-I", os.path.join(ROOT, "include"),
                           "-I", str(work), "-I", os.path.join(ROOT, "tests", "cpp", "shim"),
                           "-o", exe, os.path.join(ROOT, "oracle", "ref_tester_main.cpp"),
                           "-L", libdir, "-l" + lib, f"-Wl,-rpath,{libdir}"])
    _BINARIES[kind] = exe
    return exe


def _run(binary, name):
    out = subprocess.run([binary, name], capture_output=True, text=True, timeout=900)
    ok = out.returncode == 0 and out.stdout.strip().endswith("PASS " + name)
    if name in CHAOTIC and not ok:
        pytest.xfail("DINF expected; double precision misses dinfres < feastol by 15 % (closest 1.15e-8) and ends with NUMERICS, extended precision "
                     "reaches DINF - tests/test_oracle.py::test_unbounded_maxsqrt_is_a_rounding_knife_edge: " + out.stdout.strip()[-120:])
    assert ok, (out.returncode, out.stdout[-500:], out.stderr[-500:])


def test_binary_lists_the_reference_tests(emu_lib, oracle_mod, tmp_path_factory):
    out = subprocess.run([_binary("emu", oracle_mod, tmp_path_factory)], capture_output=True, text=True, timeout=60)
    assert out.stdout.split() == TESTS


@pytest.mark.parametrize("name", TESTS)
def test_reference_fixture_emulated(emu_lib, oracle_mod, tmp_path_factory, name):
    _run(_binary("emu", oracle_mod, tmp_path_factory), name)


@pytest.mark.gpu
@pytest.mark.parametrize("name", TESTS)
def test_reference_fixture_gpu(gpu_lib, oracle_mod, tmp_path_factory, name):
    _run(_binary("gpu", oracle_mod, tmp_path_factory), name)
