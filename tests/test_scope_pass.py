"""The BOARD=b200 pass gives the COAST.h directives their meaning (VERDICT r01 item 6; reference:
projects/dataflowProtection/interface.cpp:364-532 processAnnotations): the sphere of replication is read from the program's
own directives, calls are redirected only for functions that are IN it and have a kernel, __NO_xMR keeps a kernel-capable
function on the CPU, and an explicit __xMR that cannot be honoured fails the build naming the function.
The programs below are this repo's own (written for the test), built in a temp directory with the same Makefile contract
as the reference's test directories.  No GPU: the cases that run a binary are the ones whose protected region stays on the CPU."""
import json
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVEL = os.path.join(ROOT, "include")

CRC = r'''
unsigned short %(anno)s crc16(const unsigned char* data_p, unsigned char length) {
    unsigned char x; unsigned short crc = 0xFFFF;
    while (length--) { x = crc >> 8 ^ *data_p++; x ^= x >> 4; crc = (crc << 8) ^ ((unsigned short)(x << 12)) ^ ((unsigned short)(x << 5)) ^ ((unsigned short)x); }
    return crc;
}
'''
MAIN = r'''
#include <stdio.h>
#include "COAST.h"
%(default)s
%(crc)s
%(extra)s
int main(void) { const unsigned char m[] = "Automated TMR"; %(call)s; return 0; }
'''


def build(tmp_path, built_lib, src, passes="-TMR -countErrors", host_ok=None, name="prog"):
    d = tmp_path / name
    d.mkdir()
    (d / f"{name}.c").write_text(src)
    (d / "Makefile").write_text(f"LEVEL = {LEVEL}\nTARGET = {name}\nOPT_PASSES = {passes}\ninclude $(LEVEL)/makefiles/Makefile.common\n")
    cmd = ["make", "-C", str(d), f"OUT_DIR={d}/out", "BOARD=b200", "exe"] + ([f"COAST_HOST_OK={host_ok}"] if host_ok is not None else [])
    res = subprocess.run(cmd, capture_output=True, text=True)
    return res, d / "out"


def prog(anno="", default="", extra="", call='printf("result: %hx\\n", crc16(m, 13))'):
    return MAIN % dict(default=default, crc=CRC % dict(anno=anno), extra=extra, call=call)


def redirected(out, fn="crc16"):
    asm = "".join(p.read_text() for p in out.glob("*.xmr.s"))
    return bool(re.search(r"call\s+coast_xmr_" + fn + r"@PLT", asm))


def test_default_scope_offloads_a_function_that_has_a_kernel(tmp_path, built_lib):
    res, out = build(tmp_path, built_lib, prog())
    assert res.returncode == 0, res.stdout + res.stderr
    assert "offload   crc16 -> coast_xmr_crc16   (default scope)" in res.stdout and redirected(out)


def test_no_xmr_keeps_the_call_on_the_cpu_and_the_binary_runs_without_a_gpu(tmp_path, built_lib):
    res, out = build(tmp_path, built_lib, prog(anno="__NO_xMR"))
    assert res.returncode == 0, res.stdout + res.stderr
    assert "cpu-only  crc16 stays on the CPU, unprotected (__NO_xMR)" in res.stdout and not redirected(out)
    assert "nothing in this program is offloaded" in res.stdout
    run = subprocess.run([str(out / "prog.out")], capture_output=True, text=True)      # its own crc16, on this CPU-only box
    assert run.returncode == 0 and "result: 5ba3" in run.stdout


def test_default_no_xmr_leaves_an_unmarked_function_out_and_an_explicit_one_in(tmp_path, built_lib):
    res, out = build(tmp_path, built_lib, prog(default="__DEFAULT_NO_xMR"), name="a")
    assert res.returncode == 0 and "scope: default no_xMR" in res.stdout and not redirected(out)
    res, out = build(tmp_path, built_lib, prog(default="__DEFAULT_NO_xMR", anno="__xMR"), name="b")
    assert res.returncode == 0 and "offload   crc16 -> coast_xmr_crc16   (__xMR)" in res.stdout and redirected(out)


def test_an_xmr_function_without_a_kernel_fails_the_build_naming_it(tmp_path, built_lib):
    res, out = build(tmp_path, built_lib, prog(extra="int __xMR foo(int a) { return 2 * a; }", call="return foo(3) == 6 ? 0 : crc16(m, 13)"))
    assert res.returncode != 0
    assert "function 'foo' is marked __xMR but libcoast_rt has no protected kernel for it" in res.stderr
    assert "kernel entries: crc16 sha256_hash aes_enc_dec matrix_multiply" in res.stderr and not (out / "prog.out").exists()
    # the escape hatch is explicit and loud
    res, out = build(tmp_path, built_lib, prog(extra="int __xMR foo(int a) { return 2 * a; }", call="return foo(3) == 6 ? 0 : crc16(m, 13)"),
                     host_ok="foo", name="ok")
    assert res.returncode == 0 and "WARNING   foo is marked __xMR but has no kernel: it runs UNPROTECTED" in res.stdout


def test_an_xmr_wrapper_around_a_kernel_entry_is_accepted_and_reported(tmp_path, built_lib):
    extra = "unsigned short __xMR run_test(const unsigned char* p) { return crc16(p, 13); }\nint checkGolden(unsigned short v) __NO_xMR { return v != 0x5ba3; }"
    res, out = build(tmp_path, built_lib, prog(default="__DEFAULT_NO_xMR", anno="__xMR", extra=extra, call="return checkGolden(run_test(m))"))
    assert res.returncode == 0, res.stdout + res.stderr
    assert "wrapper   run_test runs on the host; its protected work is the kernel entry it calls (__xMR)" in res.stdout and redirected(out)


def scope_tool(tmp_path):
    tool = str(tmp_path / "coast_scope")
    subprocess.run(["gcc", "-O1", "-o", tool, os.path.join(LEVEL, "makefiles", "coast_scope.c")], check=True)
    return tool


def scan(tmp_path, src):
    tool = scope_tool(tmp_path)
    pre = subprocess.run(["gcc", "-E", "-w", "-DCOAST_SCOPE_SCAN", "-include", os.path.join(LEVEL, "coast_shim.h"), "-I", LEVEL, "-x", "c", "-"],
                         input=src, capture_output=True, text=True, check=True).stdout
    return subprocess.run([tool, "scan"], input=pre, capture_output=True, text=True, check=True).stdout.splitlines()


def test_scanner_reads_directives_in_every_position_the_reference_tests_use(tmp_path):
    facts = scan(tmp_path, r'''
    __DEFAULT_NO_xMR
    unsigned __xMR results[9][9] = { {1, 2}, {3} };  unsigned __NO_xMR golden[9][9];
    struct S { int a; } __xMR sv;
    typedef int (*fp_t)(int);
    int checkGolden() __NO_xMR { int __xMR n = 0; return n; }
    __attribute__((noinline)) void __xMR sha256_hash(unsigned char d[], unsigned len) { (void)d; (void)len; }
    static char* __xMR name_of(int k) { return k ? "a(" : "b{"; }
    void isr(void) __ISR_FUNC;  int rv(void) __xMR_RET_VAL;  void lib(void) __xMR_PROT_LIB;
    void plain(int x) { if (x) sha256_hash(0, 1); while (x--) isr(); }
    ''')
    assert "default no_xMR" in facts
    for want in ("var results xMR", "var golden no_xMR", "var sv xMR", "fn checkGolden no_xMR", "def checkGolden", "local checkGolden xMR",
                 "fn sha256_hash xMR", "def sha256_hash", "fn name_of xMR", "def name_of", "fn isr isr_function", "fn rv repl_return_val",
                 "fn lib protected_lib", "def plain", "call plain sha256_hash", "call plain isr"):
        assert want in facts, (want, facts)
    assert not [f for f in facts if f.startswith("call") and f.split()[2] in ("if", "while", "return", "sizeof")]
    assert not [f for f in facts if "fp_t" in f]


def test_the_reference_tests_get_the_scope_their_directives_ask_for(tmp_path):
    """matrixMultiply.c: `int checkGolden() __NO_xMR` stays on the CPU, matrix_multiply (default scope) is offloaded, the explicitly
    __xMR `initialize()` is reported as unprotected; sha256_tmr.c: __DEFAULT_NO_xMR + `void __xMR sha256_hash`.
    The scope facts the scanner reads out of those two programs are stored in tests/golden/reference_programs.json
    (tests/golden/make_golden.py); the pass decides from them as the make flow would, with each program's own -verbose."""
    with open(os.path.join(ROOT, "tests", "golden", "reference_programs.json")) as f:
        facts = json.load(f)["scope_facts"]
    tool = scope_tool(tmp_path)
    for target, verbose, wants in (
        ("matrixMultiply", "0", ["offload   matrix_multiply -> coast_xmr_matrix_multiply   (default scope)", "WARNING   initialize is marked __xMR"]),
        ("sha256_tmr", "1",
         ["scope: default no_xMR", "offload   sha256_hash -> coast_xmr_sha256_hash   (__xMR)", "inside    sha256_transform", "wrapper   sha_run_test",
          "WARNING   checkGolden is marked __xMR", "cpu-only  main"]),
    ):
        scope = tmp_path / f"{target}.scope"
        scope.write_text(facts[target])
        res = subprocess.run([tool, "plan", os.path.join(LEVEL, "makefiles", "coast_entries.tab"), str(tmp_path / f"{target}.sed"),
                              "checkGolden initialize", verbose, str(scope)], capture_output=True, text=True)
        assert res.returncode == 0, res.stdout + res.stderr
        for w in wants:
            assert w in res.stdout, (w, res.stdout)
        assert "coast_xmr_" in (tmp_path / f"{target}.sed").read_text()
