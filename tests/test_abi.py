"""CPU: the C-ABI library builds, loads without a GPU, exports every symbol include/coast_rt.h declares,
parses OPT_PASSES like the reference's Makefiles write them, and fails LOUDLY (no CPU fallback)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "coast_rt.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    fns = re.findall(r"^\s*(?:int|void|unsigned short|uint32_t|const char\*)\s+(\w+)\s*\(", src, flags=re.M)
    vars_ = re.findall(r"^\s*extern\s+\w+\s+(\w+);", src, flags=re.M)
    return sorted(set(fns)), sorted(set(vars_))


def test_library_exports_everything_the_header_declares(built_lib):
    fns, vars_ = declared_symbols()
    assert "coast_launch" in fns and "FAULT_DETECTED_DWC" in fns and len(fns) >= 30
    assert vars_ == ["TMR_ERROR_CNT", "__SYNC_COUNT"]
    L = C.CDLL(built_lib)
    for name in fns + vars_:
        assert hasattr(L, name), f"libcoast_rt.so does not export {name}"
    import coast_b200.runtime as r
    assert set(fns + vars_) == set(r.EXPORTS)
    assert C.c_uint32.in_dll(L, "TMR_ERROR_CNT").value == 0       # zero-initialised (synchronization.cpp:278-290)
    assert C.c_uint64.in_dll(L, "__SYNC_COUNT").value == 0


def test_sm100a_cubin_is_embedded(built_lib):
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", os.path.join(ROOT, "coast_b200", "csrc", "coast_kernels.cubin")],
                         capture_output=True, text=True).stdout
    assert "sm_100a" in out
    blob = open(built_lib, "rb").read()
    cubin = open(os.path.join(ROOT, "coast_b200", "csrc", "coast_kernels.cubin"), "rb").read()
    assert cubin[:4] == b"\x7fELF" and cubin in blob


def test_cubin_kernels_are_exactly_those_the_host_code_can_name(built_lib):
    """coast_rt.c builds kernel names with snprintf; a typo would only show up as a launch failure on a GPU box.  Conversely, every
    kernel in the cubin is one the host code can launch: nothing is built that no path reaches."""
    import itertools
    import re
    import subprocess
    src = open(os.path.join(ROOT, "coast_b200", "csrc", "coast_rt.c")).read()
    fmts = set(re.findall(r'"(xmr_[A-Za-z0-9_%]+)"', src))
    stems = {"xmr_aes128_enc", "xmr_aes128_dec", "xmr_aes128_enck", "xmr_aes128_deck",
             "xmr_chaes_enc", "xmr_chaes_dec"}               # stems of a "%s_nc%u_inj%d"
    assert stems <= fmts
    fmts = (fmts - stems) | {s + "_nc%u_inj%d" for s in stems}
    names = set()
    for f in fmts:
        ncs = ["1", "2"] if f.startswith("xmr_gemm_tf32p_") else ["1", "2", "3"]     # CTA pairs for nc < 3 only
        opts = [["tc", "tct"] if tok == "%s" else ncs if tok == "%u" else ["0", "1"] for tok in re.findall(r"%[sud]", f)]
        for combo in itertools.product(*opts):
            it = iter(combo)
            names.add(re.sub(r"%[sud]", lambda m: next(it), f))
    sass = subprocess.run(["cuobjdump", "-elf", os.path.join(ROOT, "coast_b200", "csrc", "coast_kernels.cubin")],
                          capture_output=True, text=True).stdout
    have = set(re.findall(r"\.text\.(xmr_\w+)", sass))
    assert len(names) > 80 and not (names - have), sorted(names - have)
    assert not (have - names), sorted(have - names)


@pytest.mark.parametrize("s,nc,fl", [
    ("-TMR -reportErrors", 3, 0x40),                       # tests/crc16/Makefile:3
    ("-TMR -verbose -countErrors", 3, 0x21),               # tests/sha256_common/Makefile:3
    ("-DWC #-DebugStatements", 2, 0),                      # tests/matrixMultiply/Makefile:3
    ("", 1, 0),                                            # tests/aes/Makefile:3
    ("-TMR -countErrors -countSyncs -noMemReplication -i", 3, 0x1 | 0x2 | 0x4 | 0x8),
    ("-DWC -noLoadSync -noStoreDataSync -noStoreAddrSync -s", 2, 0x10 | 0x400 | 0x800 | 0x1000),   # unittest/cfg/full.yml sweep
    ("-TMR -noMemReplication -storeDataSync -countErrors -countSyncs", 3, 0x4 | 0x200 | 0x3),
    ("-TMR -CFCSS -someUnknownPass", 3, 0),                # unknown tokens: warn and ignore
])
def test_parse_opt_passes(built_lib, s, nc, fl):
    import coast_b200 as cb
    assert cb.parse_opt_passes(s) == (nc, fl)


def test_tmr_and_dwc_are_exclusive(built_lib):
    import coast_b200 as cb
    with pytest.raises(cb.CoastError):
        cb.parse_opt_passes("-TMR -DWC")


def test_geometry_matches_oracle_spec(built_lib, oracle):
    import coast_b200 as cb
    L = cb.load_library()
    for k in range(5):
        assert L.coast_out_bytes_per_unit(k) == oracle.out_bytes_per_unit(k)
        assert L.coast_votes_per_unit(k) == oracle.votes_per_unit(k)
        for ub in (0, 1, 10, 13, 55, 56, 64, 119, 120, 255, 4000):
            for K in (0, 9, 4096):
                n = L.coast_fault_sites(k, ub, K)
                assert n == oracle.fault_sites(k, ub, K)
                for site in {0, n // 2, max(n, 1) - 1}:
                    assert L.coast_fault_site_bits(k, ub, K, site) == oracle.fault_site_bits(k, ub, K, site)


def _has_gpu():
    return os.path.exists("/dev/nvidiactl")


@pytest.mark.skipif(_has_gpu(), reason="this test documents the no-GPU behaviour")
def test_no_gpu_fails_loudly_never_falls_back(built_lib):
    import coast_b200 as cb
    L = cb.load_library()
    d = cb.LaunchDesc()
    d.kernel, d.num_clones, d.n_units = cb.K_SHA256, 3, 1
    assert L.coast_launch(C.byref(d), None) == cb.runtime.ERR_NOT_INIT
    assert b"coast_init" in L.coast_last_error()
    assert L.coast_init(0) == cb.runtime.ERR_NO_DRIVER
    assert b"no CPU fallback" in L.coast_last_error()
    with pytest.raises(cb.CoastError) as e:
        cb.Runtime(0)
    assert e.value.code == cb.runtime.ERR_NO_DRIVER


def test_product_never_touches_the_oracle():
    """oracle/ is test infrastructure: nothing under coast_b200/ or include/ may import, include or load it
    (comments that say the fault-site spec is shared with oracle/ are fine)."""
    pat = re.compile(r"pyoracle|liboracle|coast_oracle|(?:import|from)\s+oracle|#\s*include\s+\"[^\"]*oracle|_ref/libref")
    bad = []
    for base in ("coast_b200", "include"):
        for dp, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".c", ".cu", ".cuh", ".h", ".S")) or f == "Makefile":
                    if pat.search(open(os.path.join(dp, f), errors="ignore").read()):
                        bad.append(os.path.join(dp, f))
    assert not bad, bad


def _build_c_demo(built_lib, out_dir):
    import subprocess
    exe = os.path.join(out_dir, "abi_demo")
    cmd = ["gcc", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "c", "abi_demo.c"),
           "-L", os.path.join(ROOT, "coast_b200"), "-lcoast_rt", f"-Wl,-rpath,{os.path.join(ROOT, 'coast_b200')}", "-o", exe]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def test_plain_c_caller_compiles_and_links(built_lib, tmp_path):
    """include/coast_rt.h is usable from plain C (no CUDA headers) and a user FAULT_DETECTED_DWC overrides the weak default"""
    import subprocess
    exe = _build_c_demo(built_lib, str(tmp_path))
    syms = subprocess.run(["nm", "-D", "--defined-only", exe], capture_output=True, text=True).stdout
    assert "FAULT_DETECTED_DWC" in syms
    if not _has_gpu():
        res = subprocess.run([exe], capture_output=True, text=True)
        assert res.returncode == 2 and "no CPU fallback" in res.stderr      # fails loudly without a driver


@pytest.mark.gpu
def test_plain_c_caller_runs_on_the_gpu(built_lib, tmp_path):
    import subprocess
    exe = _build_c_demo(built_lib, str(tmp_path))
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "result: 5ba3" in res.stdout and "C:0 E:0 F:" in res.stdout and "handler_calls=1" in res.stdout and "abi_demo ok" in res.stdout


def test_flags_honoured_says_what_each_kernel_really_does(built_lib):
    """coast_flags_honoured(): counting flags everywhere; in-loop store votes for CRC16 / MM_U32 / SHA256 only; -i is every kernel's native
    replica placement (adjacent lanes / back-to-back MMAs), -s (separate warps) exists for SHA-256 TMR only"""
    import coast_b200.runtime as r
    L = r.load_library()
    F_CE, F_CS, F_NOMEM, F_I, F_S, F_SDS = 0x1, 0x2, 0x4, 0x8, 0x10, 0x200
    K_CRC, K_SHA, K_AES, K_MM, K_GEMM, K_QS = 0, 1, 2, 3, 4, 5
    for k in (K_CRC, K_SHA, K_AES, K_MM, K_GEMM, K_QS):
        for nc in (2, 3):
            h = L.coast_flags_honoured(k, nc, F_CE | F_CS | F_I | F_S | F_NOMEM | F_SDS)
            assert h & F_CE and h & F_CS and h & F_I, (k, nc, hex(h))
            assert bool(h & F_S) == (k == K_SHA and nc == 3), (k, nc, hex(h))
            assert bool(h & F_NOMEM) == bool(h & F_SDS) == (k in (K_CRC, K_SHA, K_MM)), (k, nc, hex(h))


def _sass(fun):
    import subprocess
    cubin = os.path.join(ROOT, "coast_b200", "csrc", "coast_kernels.cubin")
    return subprocess.run(["cuobjdump", "-sass", "-fun", fun, cubin], capture_output=True, text=True, timeout=300).stdout


def test_sass_carries_the_blackwell_instructions_the_design_claims(built_lib):
    """cuobjdump of the embedded sm_100a cubin: tcgen05 MMAs (UTCHMMA / UTCIMMA), TMA loads (UTMALDG), TMEM loads (LDTM); the
    replicated TF32 MMAs keep A in the collector (A_KEEP / A_REUSE); the CTA-pair kernels issue .2CTA MMAs, .2CTA TMA loads and multicast
    commits; the headline SHA-256 kernel has no local-memory traffic"""
    tmr = _sass("xmr_gemm_tf32_nc3_inj0")
    assert tmr.count("UTCHMMA") >= 12 and "UTMALDG" in tmr and "LDTM" in tmr
    assert "A_KEEP" in tmr and "A_REUSE" in tmr and ".2CTA" not in tmr
    pair = _sass("xmr_gemm_tf32p_nc2_inj0")
    assert "UTCHMMA.2CTA" in pair and "UTMALDG.2D.2CTA" in pair and "UTMALDG.3D.2CTA" in pair and "UTCBAR.2CTA.MULTICAST" in pair
    assert "UCGABAR_ARV" in pair and "UCGABAR_WAIT" in pair                     # the cluster barrier around TMEM allocation / teardown
    limb = _sass("xmr_mm_u32_tc_nc3_inj0")
    assert limb.count("UTCIMMA") >= 120 and "A_KEEP" in limb
    sha = _sass("xmr_sha256_b64_seg_nc3_inj1")
    assert "UTMALDG" in sha and "STL" not in sha and "LDL" not in sha
    aes = _sass("xmr_aes128_enc_nc2_inj1")
    assert "UTMALDG" in aes and "SYNCS" in aes and "PRMT" in aes                # TMA ring on mbarriers, byte-permute table addressing
