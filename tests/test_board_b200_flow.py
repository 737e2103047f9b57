"""The BOARD=b200 make flow (include/makefiles/Makefile.common): the reference's UNCHANGED test directories
build against libcoast_rt.so -- `make -C <coast>/tests/<t> LEVEL=<repo>/include BOARD=b200 exe`.

CPU part (needs the reference checkout): the flow builds, the coast pass redirected the protected-region calls,
the binary links the runtime.  GPU part: the binaries built here travel with the snapshot (oracle/_ref/b200/, where
every output of compiling reference sources goes) and must print what the reference harness greps for."""
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from build_reference_tests import CASES, OUT, REF, exe_path, make_cmd, run_env  # noqa: E402  (the list build() uses too)


@pytest.mark.skipif(not os.path.isdir(REF), reason="reference checkout absent (GPU box)")
@pytest.mark.parametrize("tdir,target,extra,entry,_re,_rc", CASES)
def test_unchanged_reference_tests_build_against_the_runtime(built_lib, tdir, target, extra, entry, _re, _rc):
    res = subprocess.run(make_cmd(tdir, extra, rebuild=True), capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    exe = exe_path(target, extra)
    assert os.path.exists(exe)
    odir = os.path.dirname(exe)
    asm = "".join(open(os.path.join(odir, f)).read() for f in os.listdir(odir) if f.endswith(".xmr.s"))
    assert re.search(r"call\s+" + entry + r"@PLT", asm), "the pass did not redirect the protected-region call"
    needed = subprocess.run(["readelf", "-d", exe], capture_output=True, text=True).stdout
    assert "libcoast_rt.so" in needed
    glue = open(os.path.join(odir, "coast_glue.c")).read()
    assert "coast_set_opt_passes" in glue


def test_coast_h_has_the_full_macro_surface():
    """every macro of the reference's tests/COAST.h:11-67 exists, and the header is gcc-clean in all positions the tests use"""
    src = r'''
    #include <stddef.h>
    #include "COAST.h"
    __DEFAULT_NO_xMR
    unsigned __xMR g1[4]; unsigned __NO_xMR g2[4]; int __COAST_VOLATILE keep;
    int checkGolden() __NO_xMR { int __xMR n = 0; return n; }
    void __xMR f1(void) {}  __attribute__((noinline)) int __xMR f2(int a) { return a; }
    void isr(void) __ISR_FUNC; int rv(void) __xMR_RET_VAL; int pl(void) __xMR_PROT_LIB; int ac(int*) __xMR_ALL_AFTER_CALL;
    int __xMR_AFTER_CALL(scanf, 1_2)(const char*, ...);
    MALLOC_WRAPPER_REGISTER(my_malloc); PRINTF_WRAPPER_REGISTER(my_printf); void* GENERIC_COAST_WRAPPER(thing)(void);
    void ig(void) __COAST_IGNORE_GLOBAL(g1); void na(int a, int b) __NO_xMR_ARG(1); void ni(void) __COAST_NO_INLINE;
    void fc(void) __xMR_FN_CALL; void sk(void) __SKIP_FN_CALL;
    int main(void) { void* p = MALLOC_WRAPPER_CALL(my_malloc, 4); (void)p; return __xMR_DEFAULT_BEHAVIOR__; }
    '''
    res = subprocess.run(["gcc", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"), "-x", "c", "-"],
                         input=src, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("tdir,target,extra,entry,regex,rc", CASES)
def test_unchanged_reference_tests_run_on_the_gpu(tdir, target, extra, entry, regex, rc):
    exe = exe_path(target, extra)
    if not os.path.exists(exe):
        pytest.skip("binary was not built on the CPU box (needs the reference checkout)")
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=run_env())
    assert res.returncode == rc, res.stdout + res.stderr          # unittest.py:76-78: non-zero exit = fail
    assert re.search(regex, res.stdout), res.stdout + res.stderr   # unittest.py:80-86 regex on stdout


# unittest/cfg/full.yml:17-36 -- the OPT_PASSES sweep unittest.py runs over every benchmark (by rebuilding with
# `make exe OPT_PASSES=...`, unittest.py:61).  The sources are not on the GPU box, so the built binaries are re-protected
# through COAST_OPT_PASSES_OVERRIDE (coast_glue.c) instead.
FULL_YML_SWEEP = [
    "", "-DWC", "-TMR", "-TMR -countErrors",
    "-DWC -noMemReplication", "-TMR -noMemReplication",
    "-DWC -noLoadSync", "-TMR -noLoadSync",
    "-DWC -noStoreDataSync", "-TMR -noStoreDataSync",
    "-DWC -noStoreAddrSync", "-TMR -noStoreAddrSync",
    "-DWC -noMemReplication -noLoadSync", "-TMR -noMemReplication -noLoadSync",
    "-DWC -noMemReplication -noStoreDataSync", "-TMR -noMemReplication -noStoreDataSync",
    "-DWC -noMemReplication -noStoreAddrSync", "-TMR -noMemReplication -noStoreAddrSync",
]


def test_sweep_list_is_the_reference_one():
    """the OPT_PASSES of the reference's unittest/cfg/full.yml, stored by tests/golden/make_golden.py"""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_programs.json")) as f:
        assert json.load(f)["full_yml_opt_passes"] == FULL_YML_SWEEP


def test_every_sweep_entry_parses_without_an_ignored_token(built_lib):
    import ctypes as C
    lib = C.CDLL(built_lib)
    for passes in FULL_YML_SWEEP:
        nc, fl = C.c_uint32(), C.c_uint32()
        code = ("import ctypes as C,sys; l=C.CDLL(sys.argv[1]); n=C.c_uint32(); f=C.c_uint32(); "
                "sys.exit(l.coast_parse_opt_passes(sys.argv[2].encode(), C.byref(n), C.byref(f)) * 0 + n.value)")
        res = subprocess.run([sys.executable, "-c", code, built_lib, passes], capture_output=True, text=True)
        assert "ignored" not in res.stderr and "not emulated" not in res.stderr, (passes, res.stderr)
        assert res.returncode == (3 if "-TMR" in passes else 2 if "-DWC" in passes else 1), passes
        assert lib.coast_parse_opt_passes(passes.encode(), C.byref(nc), C.byref(fl)) == 0


def _store_votes(passes):
    return ("-noMemReplication" in passes or "-storeDataSync" in passes) and "-noStoreDataSync" not in passes


@pytest.mark.gpu
@pytest.mark.parametrize("target,regex", [("matrixMultiply", r"Number of errors: 0"), ("crc16", r"result: 5ba3"),
                                          ("aes", r"Number of errors: 0")])
def test_unittest_full_yml_sweep_on_the_gpu(target, regex):
    """unittest.py:61-86 over cfg/full.yml: every benchmark x every OPT_PASSES must exit 0 and match its regex -- and the
    variants must DIFFER where the reference's do (VERDICT r01): -noMemReplication turns every assignment into a sync point
    (synchronization.cpp:205-215), which shows in __SYNC_COUNT (crc16: 3 per byte + 1 for the 13-byte message = 40 instead of 1;
    matrixMultiply 9x9: 81 x (9 + 1) per matrix_multiply call instead of 81) and in the kernel the runtime picks; a kernel that
    cannot honour the flag (aes) says so on stderr instead of silently running the default."""
    exe = os.path.join(OUT, target, target + ".out")
    if not os.path.exists(exe):
        pytest.skip("binary was not built on the CPU box (needs the reference checkout)")
    seen = {}
    for passes in FULL_YML_SWEEP:
        count = " -countErrors -countSyncs" if "-TMR" in passes else ""
        env = run_env(COAST_OPT_PASSES_OVERRIDE=passes + count + " -verbose", COAST_REPORT_COUNTERS="1")
        res = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=env)
        assert res.returncode == 0, (passes, res.stdout + res.stderr)
        assert re.search(regex, res.stdout), (passes, res.stdout + res.stderr)
        want = "_nc3_" if "-TMR" in passes else "_nc2_" if "-DWC" in passes else "_nc1_"
        assert want in res.stderr, (passes, res.stderr)      # -verbose names the kernel actually launched
        m = re.search(r"TMR_ERROR_CNT=(\d+) __SYNC_COUNT=(\d+)", res.stderr)
        assert m and int(m.group(1)) == 0, (passes, res.stderr)
        seen[passes] = int(m.group(2))
        warned = "NOT honoured" in res.stderr
        assert warned == (target == "aes" and _store_votes(passes)), (passes, res.stderr)
    if target == "crc16":
        assert seen["-TMR -countErrors"] == seen["-TMR"] == 1 and seen["-TMR -noMemReplication"] == 3 * 13 + 1
        assert seen["-TMR -noMemReplication -noStoreDataSync"] == 1 and seen["-TMR -noMemReplication -noLoadSync"] == 40
        assert seen["-DWC -noMemReplication"] == 0            # __SYNC_COUNT only exists under TMR -countErrors (:1415-1425)
    if target == "matrixMultiply":
        calls = seen["-TMR"] // 81                            # generateGolden + test: matrix_multiply is called twice (matrixMultiply.c:131-139)
        assert calls >= 1 and seen["-TMR"] == 81 * calls and seen["-TMR -noMemReplication"] == 81 * (9 + 1) * calls
    if target == "aes":
        assert len(set(seen[p] for p in FULL_YML_SWEEP if "-TMR" in p)) == 1     # and says so: see `warned`


@pytest.mark.gpu
def test_strict_flags_turn_an_unhonoured_flag_into_an_error():
    exe = os.path.join(OUT, "aes", "aes.out")
    if not os.path.exists(exe):
        pytest.skip("binary was not built on the CPU box (needs the reference checkout)")
    env = run_env(COAST_OPT_PASSES_OVERRIDE="-TMR -noMemReplication", COAST_STRICT_FLAGS="1")
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=env)
    assert res.returncode != 0 and "has no in-loop store votes" in res.stderr
