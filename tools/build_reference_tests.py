#!/usr/bin/env python3
"""Build the reference's UNCHANGED test directories against libcoast_rt.so with the BOARD=b200 make flow
(include/makefiles/Makefile.common).  Needs the reference checkout; outputs go to oracle/_ref/b200/<TARGET>/ (git-ignored,
they are compiled reference code) and travel to the GPU box with the snapshot, where tests/test_board_b200_flow.py runs
them.  Called by __graft_entry__.build() and by the CPU tests."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference/tests"
OUT = os.path.join(ROOT, "oracle", "_ref", "b200")

# test dir, TARGET, extra make vars, runtime entry the pass must have wired in, expected stdout regex, expected exit code
CASES = [
    ("crc16", "crc16", [], "coast_xmr_crc16", r"result: 5ba3", 0),                                  # crc16.c:42
    ("aes", "aes", [], "coast_xmr_aes_enc_dec", r"Number of errors: 0", 0),                         # aes.c:114 (568 NIST KATs)
    ("matrixMultiply", "matrixMultiply", [], "coast_xmr_matrix_multiply", r"Number of errors: 0", 0),   # unittest/cfg/full.yml:2-3
    ("sha256_common", "sha256_tmr", ["SRCFILES={ref}/sha256_common/sha256_tmr.c"], "coast_xmr_sha256_hash",
     r"C:0 E:0 F:0 T:0us", 0),                                                                      # sha256_tmr.c:30
    ("mm_common", "mm_tmr", ["SRCFILES={ref}/mm_common/mm_tmr.c", "TARGET=mm_tmr", "OPT_PASSES=-TMR -countErrors"],
     "coast_xmr_matrix_multiply", r"Error\?: 0", 0),                                                # mm_tmr.c:38
    ("chstone/sha", "sha_driver", [], "coast_xmr_sha_stream", r"RESULT: PASS", 0),                  # unittest/cfg/full.yml:5-6
    ("chstone/aes", "aes", ["OUT_DIR={out}/chstone_aes"], "coast_xmr_chaes_encrypt",
     r"encrypted message \t3925841d02dc09fbdc118597196a0b32\ndecrypto message\t3243f6a8885a308d313198a2e0370734RESULT: PASS", 0),   # aes.c:137-139
]


def run_env(**extra) -> dict:
    """Environment that runs a built program against THIS tree's coast_b200/libcoast_rt.so.  The programs' rpath is relative
    to $ORIGIN, which the loader takes from the executable's resolved path: when oracle/_ref reaches the tree through a
    link (or a copy made elsewhere), that path lies outside the tree.  LD_LIBRARY_PATH is searched before the rpath."""
    env = dict(os.environ, **extra)
    env["LD_LIBRARY_PATH"] = os.pathsep.join(p for p in (os.path.join(ROOT, "coast_b200"), os.environ.get("LD_LIBRARY_PATH")) if p)
    return env


def available() -> bool:
    return os.path.isdir(REF)


def make_cmd(tdir, extra, rebuild=False):
    return ["make", "-s", "-C", os.path.join(REF, tdir), f"LEVEL={ROOT}/include", "BOARD=b200"] + (["-B"] if rebuild else []) + \
           [e.format(ref=REF, out=OUT) for e in extra] + ["exe"]


def exe_path(target, extra):
    """TARGET `aes` exists twice (tests/aes and tests/chstone/aes): a case may move its OUT_DIR"""
    for e in extra:
        if e.startswith("OUT_DIR="):
            return os.path.join(e[len("OUT_DIR="):].format(ref=REF, out=OUT), target + ".out")
    return os.path.join(OUT, target, target + ".out")


def build_all(rebuild: bool = False) -> None:
    """No-op where the reference checkout is absent (the GPU box uses the prebuilt binaries)."""
    if not available():
        return
    for tdir, target, extra, *_ in CASES:
        res = subprocess.run(make_cmd(tdir, extra, rebuild), capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"BOARD=b200 flow failed for {tdir}:\n{res.stdout}{res.stderr}")
        assert os.path.exists(exe_path(target, extra))


if __name__ == "__main__":
    build_all(rebuild="-B" in sys.argv)
    print("built:", ", ".join(c[1] for c in CASES) if available() else "reference checkout absent")
