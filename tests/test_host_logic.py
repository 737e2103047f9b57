"""Host logic of libcoast_rt.so (coast_b200/csrc/coast_rt.c) on a GPU-less box, against a MOCK driver
(tests/mock_cuda/mock_cuda.c, test infrastructure: it runs no workload, it records and bounds-checks driver calls):
launch geometry and shared memory within sm_100 limits, tensor maps inside the caller's buffers, the argument block every
kernel receives, the chunk schedule of coast_run_host() (every byte copied exactly once, per-chunk unit_base), scratch and
staging memory released, loud failures for bad arguments and for a non-sm_100 device."""
import ctypes as C
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K_CRC16, K_SHA256, K_AES128, K_MM_U32, K_GEMM_TF32, K_QSORT, K_CHSTONE_SHA = range(7)


class XmrArgs(C.Structure):                     # coast_b200/csrc/xmr_args.h
    _fields_ = [("inp", C.c_uint64), ("out", C.c_uint64), ("aux", C.c_uint64), ("n_units", C.c_uint64), ("unit_base", C.c_uint64),
                ("counters", C.c_uint64), ("plan_table", C.c_uint64), ("status", C.c_uint64),
                ("unit_bytes", C.c_uint32), ("flags", C.c_uint32), ("mode", C.c_uint32), ("M", C.c_uint32), ("N", C.c_uint32),
                ("K", C.c_uint32), ("plan_mode", C.c_uint32), ("seed_lo", C.c_uint32), ("seed_hi", C.c_uint32),
                ("threshold", C.c_uint32), ("n_sites", C.c_uint32), ("n_tiles", C.c_uint32), ("key", C.c_uint8 * 16)]


@pytest.fixture(scope="session")
def mock_dir(tmp_path_factory, built_lib):
    d = tmp_path_factory.mktemp("mockcuda")
    subprocess.run(["gcc", "-O1", "-shared", "-fPIC", "-Wall", "-I/usr/local/cuda/include", "-o", str(d / "libcuda.so.1"),
                    os.path.join(ROOT, "tests", "mock_cuda", "mock_cuda.c")], check=True)
    return d


def run_child(mock_dir, tmp_path, ops, env_extra=None):
    log = tmp_path / "mock.log"
    if log.exists():
        log.unlink()                                        # one log per child run
    env = dict(os.environ, LD_LIBRARY_PATH=f"{mock_dir}:" + os.environ.get("LD_LIBRARY_PATH", ""), MOCK_CUDA_LOG=str(log))
    env.update(env_extra or {})
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "mock_cuda", "child.py"), json.dumps({"ops": ops})],
                         capture_output=True, text=True, env=env, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    events = [json.loads(ln) for ln in open(log)] if log.exists() else []
    return json.loads(res.stdout.strip().splitlines()[-1]), events


def args_of(ev):
    assert sizeof_args() == 128
    return XmrArgs.from_buffer_copy(bytes.fromhex(ev["arg0"]))


def sizeof_args():
    return C.sizeof(XmrArgs)


def test_argument_block_mirror_matches_the_header():
    src = open(os.path.join(ROOT, "coast_b200", "csrc", "xmr_args.h")).read()
    assert sizeof_args() == 128 and "unsigned char key[16];" in src and src.index("n_tiles") < src.index("key[16]")


@pytest.mark.parametrize("kernel,nc,n,ub,in_b,out_b,want", [
    (K_SHA256, 3, 100000, 64, 6400000, 3200000, ("xmr_sha256_b64_seg_nc3_inj0", 384, 128)),
    (K_SHA256, 2, 100000, 64, 6400000, 3200000, ("xmr_sha256_b64_nc2_inj0", 256, 128)),
    (K_SHA256, 3, 1000, 100, 100000, 32000, ("xmr_sha256_gen_nc3_inj0", 256, None)),
    (K_CRC16, 3, 100000, 64, 6400000, 200000, ("xmr_crc16_b64_nc3_inj0", 1024, 320)),
    (K_CRC16, 1, 100000, 64, 6400000, 200000, ("xmr_crc16_b64_nc1_inj0", 768, 768)),
    (K_CRC16, 3, 5, 13, 65, 10, ("xmr_crc16_gen_nc3_inj0", 256, None)),
    (K_AES128, 2, 1 << 20, 0, 16 << 20, 16 << 20, ("xmr_aes128_enc_nc2_inj0", 512, 1024)),
    (K_QSORT, 3, 5000, 2320, 5000 * 2320, 5000 * 2320, ("xmr_qsort_nc3_inj0", 128, None)),
    (K_CHSTONE_SHA, 3, 300, 16384, 300 * 16384, 300 * 20, ("xmr_chsha_nc3_inj0", 256, None)),
])
def test_launch_geometry_and_argument_block(mock_dir, tmp_path, kernel, nc, n, ub, in_b, out_b, want):
    res, ev = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=kernel, nc=nc, n=n, unit_bytes=ub, in_bytes=in_b, out_bytes=out_b,
                                                  flags=3), dict(op="shutdown")])
    assert res["init"] == 0 and res["ops"][0]["rc"] == 0, res
    assert not [e for e in ev if e["op"] == "error"], ev
    launches = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert len(launches) == 1
    la = launches[0]
    name, block, tile_rows = want
    assert la["name"] == name and la["block"] == block and la["smem"] <= 232448 and 1 <= la["grid"] <= 148 * 32 * 4
    a = args_of(la)
    assert a.n_units == n and a.unit_base == 0 and a.unit_bytes == ub and a.flags == 3 and a.plan_mode == 0
    if tile_rows:                                           # TMA-tiled kernels: one tensor map over exactly the caller's rows
        assert a.n_tiles == -(-n // tile_rows) and la["grid"] <= 148 * 8
        tm = [e for e in ev if e["op"] == "tmap"]
        pack = tm[0]["dim0"] * 4 // (16 if kernel == K_AES128 else ub)      # AES: the same dense bytes as 64- or 256-byte rows
        assert (pack == 16 and (a.mode >> 8) & 15 == 4) if kernel == K_AES128 else pack == 1
        assert len(tm) == 1 and tm[0]["dim1"] * pack == n and tm[0]["box1"] <= 256 and tile_rows % (tm[0]["box1"] * pack) == 0
        assert tm[0]["box_bytes"] * (tile_rows // (tm[0]["box1"] * pack)) * 2 + 64 <= la["smem"]     # two ring stages fit
    if kernel == K_QSORT:                                   # per-unit scratch from the pool, released after the launch
        big = [e for e in ev if e["op"] == "alloc" and e["bytes"] >= la["grid"] * 4 * 32 * ub]
        assert big and a.aux != 0
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_injector_variant_and_plan_fields(mock_dir, tmp_path):
    res, ev = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=K_AES128, nc=2, n=4096, in_bytes=65536, out_bytes=65536, p=2 ** -10)])
    la = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]][0]
    a = args_of(la)
    assert la["name"] == "xmr_aes128_enc_nc2_inj1" and a.plan_mode == 1 and a.threshold == 1 << 22 and a.n_sites == 176


@pytest.mark.parametrize("kernel,ub,ob,n", [(K_SHA256, 64, 32, 1), (K_SHA256, 64, 32, 1000), (K_SHA256, 64, 32, (1 << 20) + 123),
                                            (K_CRC16, 13, 2, 7), (K_AES128, 16, 16, 300001), (K_CHSTONE_SHA, 16384, 20, 3)])
def test_run_host_chunk_schedule_copies_every_byte_once(mock_dir, tmp_path, kernel, ub, ob, n):
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host", kernel=kernel, nc=3 if kernel != K_AES128 else 2, n=n, unit_bytes=ub if kernel != K_AES128 else 0,
                                                  in_bytes=n * ub, out_bytes=n * ob, unit_base=1000), dict(op="shutdown")])
    r = res["ops"][0]
    assert r["rc"] == 0, r
    assert not [e for e in ev if e["op"] == "error"], [e for e in ev if e["op"] == "error"]
    h2d = sorted((e["host"] - r["host_in"], e["bytes"]) for e in ev if e["op"] == "h2d")
    d2h = sorted((e["host"] - r["host_out"], e["bytes"]) for e in ev if e["op"] == "d2h" and 0 <= e["host"] - r["host_out"] < n * ob)
    for spans, total in ((h2d, n * ub), (d2h, n * ob)):
        pos = 0
        for off, nb in spans:
            assert off == pos, (spans[:5], total)          # contiguous, no gap, no overlap
            pos += nb
        assert pos == total
    launches = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    done = 0
    for la in launches:                                     # every chunk is keyed by its GLOBAL unit index
        a = args_of(la)
        assert a.unit_base == 1000 + done
        done += a.n_units
    assert done == n and len({la["stream"] for la in launches}) <= 3
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


@pytest.mark.parametrize("op,needle", [
    (dict(op="launch", kernel=K_CRC16, nc=3, n=10, unit_bytes=0, in_bytes=64, out_bytes=64), "crc16 length"),
    (dict(op="launch", kernel=K_CRC16, nc=4, n=10, unit_bytes=8, in_bytes=80, out_bytes=64), "num_clones"),
    (dict(op="launch", kernel=9, nc=3, n=10, unit_bytes=8, in_bytes=80, out_bytes=64), "unknown kernel"),
    (dict(op="launch", kernel=K_CHSTONE_SHA, nc=3, n=2, unit_bytes=100, in_bytes=200, out_bytes=40), "64-byte blocks"),
    (dict(op="launch", kernel=K_QSORT, nc=3, n=2, unit_bytes=4100, in_bytes=8200, out_bytes=8200), "quicksort arrays"),
    (dict(op="launch", kernel=K_MM_U32, nc=3, n=81, M=9, N=9, K=9, in_bytes=324, out_bytes=324), "MM needs"),
    (dict(op="launch", kernel=K_AES128, nc=2, n=4, in_bytes=80, out_bytes=64, misalign=4), "16-byte aligned"),
])
def test_bad_arguments_fail_loudly(mock_dir, tmp_path, op, needle):
    res, ev = run_child(mock_dir, tmp_path, [op])
    r = res["ops"][0]
    assert r["rc"] != 0 and needle in r["err"], r
    assert not [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]


def test_unaligned_sha_input_takes_the_general_kernel(mock_dir, tmp_path):
    res, ev = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=K_SHA256, nc=3, n=100, unit_bytes=64, in_bytes=6500, out_bytes=3200, misalign=4)])
    assert res["ops"][0]["rc"] == 0
    assert [e["name"] for e in ev if e["op"] == "launch" and "_nc" in e["name"]] == ["xmr_sha256_gen_nc3_inj0"]
    assert not [e for e in ev if e["op"] == "tmap"]


def test_a_device_that_is_not_sm100_is_refused(mock_dir, tmp_path):
    res, ev = run_child(mock_dir, tmp_path, [], env_extra={"MOCK_CUDA_CC_MAJOR": "9"})
    assert res["init"] != 0 and "sm_100a code only" in res["error"]


@pytest.mark.parametrize("M,N,K,nc,env,want", [
    (256, 128, 256, 3, {}, ["xmr_mm_split_a", "xmr_mm_split_bt", "xmr_mm_u32_tct_nc3_inj0"]),       # TMR: A limb planes staged in TMEM
    (256, 128, 256, 2, {}, ["xmr_mm_split_a", "xmr_mm_split_bt", "xmr_mm_u32_tc_nc2_inj0"]),
    (256, 128, 256, 3, {"COAST_MM_PATH": "tiled"}, ["xmr_mm_u32_tiled_nc3_inj0"]),
    (64, 128, 48, 3, {}, ["xmr_mm_u32_tiled_nc3_inj0"]),                                              # not 128/64/128-aligned
    (9, 9, 9, 3, {}, ["xmr_mm_u32_nc3_inj0"]),                                                        # the reference's own size
])
def test_exact_matmul_path_selection_and_tensor_maps(mock_dir, tmp_path, M, N, K, nc, env, want):
    res, ev = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=K_MM_U32, nc=nc, n=M * N, M=M, N=N, K=K, in_bytes=M * K * 4,
                                                  aux_bytes=K * N * 4, out_bytes=M * N * 4, flags=3), dict(op="shutdown")], env_extra=env)
    assert res["ops"][0]["rc"] == 0, res
    assert not [e for e in ev if e["op"] == "error"], [e for e in ev if e["op"] == "error"]
    names = [e["name"] for e in ev if e["op"] == "launch" and e["name"] not in ("xmr_counters_reset",)]
    assert names == want
    if "split" in want[0]:
        tm = [e for e in ev if e["op"] == "tmap"]
        assert len(tm) == 2 and all(t["elem"] == 1 and t["rank"] == 3 and t["box0"] == 128 for t in tm)   # u8 limb planes, 128-byte k rows
    la = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]][0]
    assert la["smem"] <= 232448 and la["grid"] <= max(148, (M // 64) * (N // 128))
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_tf32_gemm_launch(mock_dir, tmp_path):
    s = 512
    res, ev = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=K_GEMM_TF32, nc=3, n=s * s, M=s, N=s, K=s, in_bytes=s * s * 4,
                                                  aux_bytes=s * s * 4, out_bytes=s * s * 4, flags=3)])
    assert res["ops"][0]["rc"] == 0 and not [e for e in ev if e["op"] == "error"]
    la = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]][0]
    assert la["name"] == "xmr_gemm_tf32_nc3_inj0" and la["block"] == 384 and la["grid"] == 16 and la["smem"] <= 232448
    tm = [e for e in ev if e["op"] == "tmap"]
    assert [t["rank"] for t in tm] == [2, 3] and tm[1]["swizzle"] != tm[0]["swizzle"]      # B: the 32-byte-atom swizzle of the MN-major operand
    bad, _ = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=K_GEMM_TF32, nc=3, n=100 * 128, M=100, N=128, K=64, in_bytes=100 * 64 * 4,
                                                  aux_bytes=64 * 128 * 4, out_bytes=100 * 128 * 4)])
    assert bad["ops"][0]["rc"] != 0 and "multiples of 128" in bad["ops"][0]["err"]


@pytest.mark.parametrize("nc,M,N,want_name,want_grid", [
    (1, 512, 512, "xmr_gemm_tf32p_nc1_inj0", 8),         # unprotected: CTA pairs, 256 x 256 pair tiles -> 4 pairs
    (2, 512, 512, "xmr_gemm_tf32p_nc2_inj0", 16),        # DWC: pairs, 256 x 128
    (3, 512, 512, "xmr_gemm_tf32_nc3_inj0", 16),         # TMR: always the single-CTA kernel
    (1, 384, 512, "xmr_gemm_tf32_nc1_inj0", 6),          # M not a multiple of 256: no pair tile, single-CTA 128 x 256
    (2, 384, 512, "xmr_gemm_tf32_nc2_inj0", 12),         # ... and single-CTA 128 x 128 for DWC
    (1, 512, 384, "xmr_gemm_tf32n_nc1_inj0", 12),        # N % 256 != 0: the narrow single-CTA kernel
    (2, 512, 384, "xmr_gemm_tf32p_nc2_inj0", 12),
    (2, 2048, 2048, "xmr_gemm_tf32p_nc2_inj0", 148),     # more tiles than SMs: one persistent CTA per SM
])
def test_tf32_gemm_kernel_selection_pairs_and_single(mock_dir, tmp_path, nc, M, N, want_name, want_grid):
    """which TF32 GEMM kernel a shape gets (single CTA / CTA pair, wide / narrow), with an EVEN grid for the cluster kernels and the
    B box matching what each kernel loads per TMA (64 columns for pairs, 128 for single CTAs)"""
    res, ev = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=K_GEMM_TF32, nc=nc, n=M * N, M=M, N=N, K=64, in_bytes=M * 64 * 4,
                                                  aux_bytes=64 * N * 4, out_bytes=M * N * 4, flags=3)])
    assert res["ops"][0]["rc"] == 0 and not [e for e in ev if e["op"] == "error"], res
    la = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]][0]
    assert (la["name"], la["grid"], la["block"]) == (want_name, want_grid, 384) and la["smem"] <= 232448
    if "tf32p" in want_name:
        assert la["grid"] % 2 == 0
    tm = [e for e in ev if e["op"] == "tmap"]
    assert tm[1]["box_bytes"] == 32 * 32 * 4 * (2 if "tf32p" in want_name else 4), tm[1]


def test_retired_tuning_variables_change_no_launch(mock_dir, tmp_path):
    """the GEMM, limb-matmul and quicksort experiment switches of earlier releases are gone: with all of them set, every launch
    (kernel, grid, block, shared memory, tensor maps, argument block) is the one made without them"""
    s = 512
    gemm = dict(op="launch", kernel=K_GEMM_TF32, n=s * s, M=s, N=s, K=64, in_bytes=s * 64 * 4, aux_bytes=64 * s * 4, out_bytes=s * s * 4, flags=3)
    ops = [dict(gemm, nc=1), dict(gemm, nc=3),
           dict(op="launch", kernel=K_MM_U32, nc=2, n=s * s, M=s, N=s, K=128, in_bytes=s * 128 * 4, aux_bytes=128 * s * 4,
                out_bytes=s * s * 4, flags=3),
           dict(op="launch", kernel=K_QSORT, nc=3, n=100, unit_bytes=4 * 580, in_bytes=100 * 4 * 580, out_bytes=100 * 4 * 580, flags=3)]
    pointers = ("inp", "out", "aux", "counters", "plan_table", "status")

    def launches(env):
        res, ev = run_child(mock_dir, tmp_path, ops, env_extra=env)
        assert [r["rc"] for r in res["ops"]] == [0] * len(ops) and not [e for e in ev if e["op"] == "error"], res
        log = []
        for e in ev:
            if e["op"] == "tmap":
                log.append(e)
            elif e["op"] == "launch" and "_nc" in e["name"]:
                a = args_of(e)
                log.append((e["name"], e["grid"], e["block"], e["smem"],
                            [(f, getattr(a, f)) for f, _ in XmrArgs._fields_ if f not in pointers and f != "key"] + [("key", bytes(a.key))]))
        return log

    plain = launches({})
    assert [x[0] for x in plain if isinstance(x, tuple)] == ["xmr_gemm_tf32p_nc1_inj0", "xmr_gemm_tf32_nc3_inj0", "xmr_mm_u32_tc_nc2_inj0",
                                                             "xmr_qsort_nc3_inj0"]
    retired = {"COAST_QSORT_PATH": "nested", "COAST_GEMM_PAIR": "1", "COAST_GEMM_GROUP_M": "8", "COAST_GEMM_L2_HINTS": "0",
               "COAST_GEMM_TAIL_SPLIT": "0", "COAST_GEMM_KEEP_A": "0", "COAST_MM_KEEP_A": "0"}
    assert launches(retired) == plain


def test_quicksort_through_the_host_call_uses_one_scratch_slot_per_chunk(mock_dir, tmp_path):
    n, L = 3000, 580
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host", kernel=K_QSORT, nc=3, n=n, unit_bytes=4 * L, in_bytes=n * 4 * L,
                                                  out_bytes=n * 4 * L), dict(op="shutdown")])
    assert res["ops"][0]["rc"] == 0 and not [e for e in ev if e["op"] == "error"]
    launches = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert sum(args_of(la).n_units for la in launches) == n and all(args_of(la).aux for la in launches)
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_host_call_staging_is_bounded_by_the_call_not_by_the_largest_chunk(mock_dir, tmp_path):
    """one 64 MiB CHStone stream, and a 1-unit crc16 call: the staging slots must not be sized for 1024 units"""
    big = 64 << 20
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host", kernel=K_CHSTONE_SHA, nc=3, n=1, unit_bytes=big, in_bytes=big, out_bytes=20),
                                             dict(op="run_host", kernel=K_CRC16, nc=3, n=1, unit_bytes=13, in_bytes=13, out_bytes=2),
                                             dict(op="shutdown")])
    assert [r["rc"] for r in res["ops"]] == [0, 0, 0], res
    assert max(e["bytes"] for e in ev if e["op"] == "alloc") <= big + 4096
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_reference_entry_points_drive_the_host_call(mock_dir, tmp_path):
    """crc16 / sha256_hash (10 bytes and empty) / aes_enc_dec both directions / matrix_multiply 9x9 / sha_stream: one protected
    launch each with the mode of OPT_PASSES, buffers staged and released"""
    res, ev = run_child(mock_dir, tmp_path, [dict(op="entries", passes="-TMR -countErrors"), dict(op="shutdown")])
    assert res["ops"][0]["rc"] == 0 and not [e for e in ev if e["op"] == "error"], [e for e in ev if e["op"] == "error"]
    names = [e["name"] for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert names == ["xmr_crc16_gen_nc3_inj0", "xmr_sha256_gen_nc3_inj0", "xmr_sha256_gen_nc3_inj0", "xmr_aes128_enck_nc3_inj0",
                     "xmr_aes128_deck_nc3_inj0", "xmr_mm_u32_nc3_inj0", "xmr_chsha_nc3_inj0"]
    args = [args_of(e) for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert [a.unit_bytes for a in args[:3]] == [13, 10, 0] and all(a.n_units == 1 for a in args[:5]) and args[5].n_units == 81
    assert args[3].mode == 2 | 4 and args[4].mode == 1 | 2 | 4          # per-unit key + write-back (+ decrypt): key[] is mutated in place
    assert args[6].unit_bytes == 16384 and all(a.flags & 1 for a in args)
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_aes_per_unit_keys_with_write_back_through_the_host_call(mock_dir, tmp_path):
    n = 200000
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host_aux", kernel=K_AES128, nc=2, n=n, mode=2 | 4, in_bytes=16 * n, aux_bytes=16 * n,
                                                  out_bytes=16 * n), dict(op="shutdown")])
    r = res["ops"][0]
    assert r["rc"] == 0 and not [e for e in ev if e["op"] == "error"]
    for key, direction in (("host_in", "h2d"), ("host_aux", "h2d"), ("host_out", "d2h"), ("host_aux", "d2h")):
        spans = sorted((e["host"] - r[key], e["bytes"]) for e in ev if e["op"] == direction and 0 <= e["host"] - r[key] < 16 * n)
        pos = 0
        for off, nb in spans:
            assert off == pos
            pos += nb
        assert pos == 16 * n, (key, direction)
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_large_matmul_through_the_host_call_is_pipelined_by_row_blocks(mock_dir, tmp_path):
    """B once; A rows up / launch / C rows down per block on rotating streams; every block's launch is keyed by its global element index"""
    M, N, K = 1024, 256, 128
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host_aux", kernel=K_GEMM_TF32, nc=3, n=M * N, M=M, N=N, K=K, in_bytes=M * K * 4,
                                                  aux_bytes=K * N * 4, out_bytes=M * N * 4, unit_base=5), dict(op="shutdown")])
    r = res["ops"][0]
    assert r["rc"] == 0 and not [e for e in ev if e["op"] == "error"], (r, [e for e in ev if e["op"] == "error"])
    launches = [(e, args_of(e)) for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert len(launches) == 8 and len({e["stream"] for e, _ in launches}) == 3
    assert [a.M for _, a in launches] == [128] * 8 and [a.unit_base for _, a in launches] == [5 + i * 128 * N for i in range(8)]
    assert len([e for e in ev if e["op"] == "h2d" and e["host"] == r["host_aux"]]) == 1            # B goes up once
    _contiguous([(e["host"] - r["host_in"], e["bytes"]) for e in ev if e["op"] == "h2d" and 0 <= e["host"] - r["host_in"] < M * K * 4], M * K * 4)
    _contiguous([(e["host"] - r["host_out"], e["bytes"]) for e in ev if e["op"] == "d2h" and 0 <= e["host"] - r["host_out"] < M * N * 4], M * N * 4)
    assert len([e for e in ev if e["op"] == "wait_event"]) == 8 and len([e for e in ev if e["op"] == "event_record"]) == 1
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_matmul_through_the_host_call_is_one_shot(mock_dir, tmp_path):
    M = N = K = 128
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host_aux", kernel=K_MM_U32, nc=3, n=M * N, M=M, N=N, K=K, in_bytes=M * K * 4,
                                                  aux_bytes=K * N * 4, out_bytes=M * N * 4), dict(op="shutdown")])
    assert res["ops"][0]["rc"] == 0 and not [e for e in ev if e["op"] == "error"]
    assert [e["bytes"] for e in ev if e["op"] == "h2d"] == [M * K * 4, K * N * 4]
    assert [e["bytes"] for e in ev if e["op"] == "d2h" and e["bytes"] > 64] == [M * N * 4]
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_lifecycle_and_small_api_calls(mock_dir, tmp_path):
    log = tmp_path / "mock.log"
    env = dict(os.environ, LD_LIBRARY_PATH=f"{mock_dir}:" + os.environ.get("LD_LIBRARY_PATH", ""), MOCK_CUDA_LOG=str(log))
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "mock_cuda", "child.py"),
                          json.dumps({"before_init": True, "ops": [dict(op="misc"), dict(op="shutdown")]})],
                         capture_output=True, text=True, env=env, timeout=120)
    assert res.returncode == 0, res.stdout + res.stderr
    out = json.loads(res.stdout.strip().splitlines()[-1])
    assert out["before_init"]["launch"] != 0 and "coast_init" in out["before_init"]["err"]
    r = out["ops"][0]
    assert r["reinit_same"] == 0 and r["reinit_other"] != 0
    assert r["fill0"] == 0 and r["fill"] == 0 and r["snapshot"] == 0
    assert r["run_host_empty"] == 0 and r["stats"] == [0, 0, 0, 0, 2 ** 64 - 1]
    assert r["run_host_table"] != 0 and "TABLE" in r["run_host_table_err"]
    assert r["launch_table_without_table"] != 0 and "d_table" in r["launch_table_err"]
    ev = [json.loads(ln) for ln in open(log)]
    assert not [e for e in ev if e["op"] == "error"] and ev[-1] == {"op": "exit", "live_allocations": 0}


@pytest.mark.parametrize("flags,mode,nc,want", [
    (3 | 0x8, 0, 3, "xmr_sha256_b64_nc3_inj0"),             # -i: replicas on adjacent lanes
    (3 | 0x10, 0, 3, "xmr_sha256_b64_seg_nc3_inj0"),        # -s (also the default)
    (3, 0, 1, "xmr_sha256_b64_nc1_inj0"),
])
def test_sha_layout_flags_select_the_kernel(mock_dir, tmp_path, flags, mode, nc, want):
    res, ev = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=K_SHA256, nc=nc, n=5000, unit_bytes=64, in_bytes=320000, out_bytes=160000,
                                                  flags=flags)])
    assert [e["name"] for e in ev if e["op"] == "launch" and "_nc" in e["name"]] == [want]


def test_aes_decrypt_and_per_unit_keys_select_the_table_kernels(mock_dir, tmp_path):
    res, ev = run_child(mock_dir, tmp_path, [dict(op="launch", kernel=K_AES128, nc=2, n=1000, mode=1, in_bytes=16000, out_bytes=16000),
                                             dict(op="launch", kernel=K_AES128, nc=2, n=1000, mode=2, in_bytes=16000, out_bytes=16000, aux_bytes=16000),
                                             dict(op="launch", kernel=K_AES128, nc=2, n=1000, mode=2, in_bytes=16000, out_bytes=16000)])
    assert [r["rc"] == 0 for r in res["ops"]] == [True, True, False] and "per-unit keys need d_aux" in res["ops"][2]["err"]
    la = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert [e["name"] for e in la] == ["xmr_aes128_dec_nc2_inj0", "xmr_aes128_enck_nc2_inj0"]
    assert [e["smem"] for e in la] == [0x38000, 0x30000] and all(e["block"] == 512 for e in la)   # decrypt adds the 32 KiB (InvS, S) table


def test_sync_folds_counters_into_the_reference_symbols(mock_dir, tmp_path):
    """coast_sync(): device counters -> coast_stats, TMR_ERROR_CNT (an i32 in the reference: wraps, synchronization.cpp:1428-1431),
    __SYNC_COUNT (i64), and the counters start from zero again"""
    res, ev = run_child(mock_dir, tmp_path, [dict(op="sync_fold"), dict(op="sync_fold"), dict(op="shutdown")],
                        env_extra={"MOCK_CUDA_TALLY": f"{2 ** 32 + 5},0,3200,7,41"})
    a, b = res["ops"][0], res["ops"][1]
    assert a["launch"] == 0 and a["sync"] == 0 and a["stats"] == [2 ** 32 + 5, 0, 3200, 7, 41]
    assert a["TMR_ERROR_CNT"] == 5 and a["SYNC_COUNT"] == 3200 and a["second"] == [0, 0, 0, 0, 2 ** 64 - 1]
    assert b["TMR_ERROR_CNT"] == 10 and b["SYNC_COUNT"] == 6400         # the symbols accumulate over the program, like the pass's globals


def test_peer_counter_block_receives_the_tallies_of_an_attached_process(mock_dir, tmp_path):
    """coast_counters_attach(): every later kernel's argument block points at the OWNER's counters (the multi-GPU fold over NVLink
    peer memory, no collective); the attached process's coast_sync() reports zeros and never resets the owner's block; detach
    restores the local block; no peer access -> a loud error, not a silent local tally"""
    res, ev = run_child(mock_dir, tmp_path, [dict(op="peer_counters"), dict(op="shutdown")], env_extra={"MOCK_CUDA_TALLY": "4,0,3200,7,41"})
    r = res["ops"][0]
    assert r["export"] == 0 and r["attach"] == 0 and r["attach_twice"] != 0 and r["launch"] == 0 and r["sync_attached"] == 0
    launches = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert len(launches) == 2
    assert args_of(launches[0]).counters == r["peer_ptr"] != args_of(launches[1]).counters
    assert r["stats_attached"] == [0, 0, 0, 0, 2 ** 64 - 1]
    assert r["peer_block"] == [4, 0, 3200, 7, 41] == r["peer_block_after"]          # attached sync did not reset it; the local run did not touch it
    assert r["detach"] == 0 and r["stats_local"] == [4, 0, 3200, 7, 41]
    opens = [e for e in ev if e["op"] == "ipc_open"]
    assert len(opens) == 1 and opens[0]["flags"] == 1                                # CU_IPC_MEM_LAZY_ENABLE_PEER_ACCESS
    assert [e for e in ev if e["op"] == "ipc_close"]
    res, ev = run_child(mock_dir, tmp_path, [dict(op="peer_counters")], env_extra={"MOCK_IPC_FAIL": "1"})
    r = res["ops"][0]
    assert r["attach"] != 0 and "peer" in r["attach_err"]


def test_dwc_detection_calls_the_handler_which_aborts_by_default(mock_dir, tmp_path):
    """FAULT_DETECTED_DWC() (synchronization.cpp:1251-1266: default = abort()) is called by coast_sync, not by coast_sync_noabort"""
    res, ev = run_child(mock_dir, tmp_path, [dict(op="sync_fold", nc=2)], env_extra={"MOCK_CUDA_TALLY": "0,3,0,3,17"})
    assert res["ops"][0]["stats"][:2] == [0, 3] and res["ops"][0]["stats"][4] == 17
    log = tmp_path / "mock2.log"
    env = dict(os.environ, LD_LIBRARY_PATH=f"{mock_dir}:" + os.environ.get("LD_LIBRARY_PATH", ""), MOCK_CUDA_LOG=str(log), MOCK_CUDA_TALLY="0,3,0,3,17")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "mock_cuda", "child.py"), json.dumps({"ops": [dict(op="sync_fold", nc=2, abort=True)]})],
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == -6 and "FAULT_DETECTED_DWC" in r.stderr          # SIGABRT, as the reference's protected binary


def _contiguous(spans, total):
    pos = 0
    for off, nb in sorted(spans):
        assert off == pos, (sorted(spans)[:5], total)
        pos += nb
    assert pos == total


def test_pinned_buffers_take_the_zero_copy_host_call(mock_dir, tmp_path):
    """pinned (mapped) host buffers + a read-once kernel: ONE launch on the host pointers' device aliases, no staging copies,
    no staging allocations; COAST_HOST_PATH=staged forces the chunked pipeline on the same buffers"""
    n = 300000
    op = dict(op="run_host_pinned", kernel=K_SHA256, nc=3, n=n, unit_bytes=64, in_bytes=64 * n, out_bytes=32 * n, unit_base=77, status=True)
    res, ev = run_child(mock_dir, tmp_path, [op, dict(op="shutdown")], env_extra={"COAST_HOST_PATH": "zerocopy"})
    r = res["ops"][0]
    assert r["rc"] == 0 and not [e for e in ev if e["op"] == "error"], (r, [e for e in ev if e["op"] == "error"])
    launches = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert len(launches) == 1 and launches[0]["name"] == "xmr_sha256_b64_seg_nc3_inj0"
    a = args_of(launches[0])
    assert (a.inp, a.out, a.status, a.n_units, a.unit_base) == (r["host_in"], r["host_out"], r["host_status"], n, 77)
    assert not [e for e in ev if e["op"] == "h2d"] and all(e["bytes"] <= 64 for e in ev if e["op"] == "d2h")     # only the counters come back by copy
    assert ev[-1] == {"op": "exit", "live_allocations": 0}
    for forced in ({"COAST_HOST_PATH": "staged"}, {}):                       # the default is the staged pipeline (r02 measurement)
        res, ev = run_child(mock_dir, tmp_path / "..", [op, dict(op="shutdown")], env_extra=forced)
        r = res["ops"][0]
        assert r["rc"] == 0 and len([e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]) > 1
        _contiguous([(e["host"] - r["host_in"], e["bytes"]) for e in ev if e["op"] == "h2d"], 64 * n)
    # hybrid: chunked launches read the pinned input in place (no upload copies), outputs and status bytes are staged per chunk
    res, ev = run_child(mock_dir, tmp_path / "..", [op, dict(op="shutdown")], env_extra={"COAST_HOST_PATH": "hybrid"})
    r = res["ops"][0]
    launches = [args_of(e) for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert r["rc"] == 0 and len(launches) > 1 and not [e for e in ev if e["op"] == "h2d"]
    done = 0
    for a in launches:
        assert a.inp == r["host_in"] + 64 * done and a.unit_base == 77 + done and a.out != r["host_out"] + 32 * done
        done += a.n_units
    assert done == n
    _contiguous([(e["host"] - r["host_out"], e["bytes"]) for e in ev if e["op"] == "d2h" and 0 <= e["host"] - r["host_out"] < 32 * n], 32 * n)


def test_default_host_path_is_zero_copy_only_for_tiny_outputs(mock_dir, tmp_path):
    """measured policy (profiles/r02_e2e_*.json): staged by default; pinned buffers + an output of at most 1/8 of the input (crc16: 2 of 64
    bytes) -> one zero-copy launch; the same call with pageable memory falls back to the staged pipeline"""
    n = 200000
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host_pinned", kernel=K_CRC16, nc=3, n=n, unit_bytes=64, in_bytes=64 * n, out_bytes=2 * n),
                                             dict(op="shutdown")])
    la = [e for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert res["ops"][0]["rc"] == 0 and len(la) == 1 and args_of(la[0]).inp == res["ops"][0]["host_in"] and not [e for e in ev if e["op"] == "h2d"]
    res, ev = run_child(mock_dir, tmp_path / "..", [dict(op="run_host", kernel=K_CRC16, nc=3, n=n, unit_bytes=64, in_bytes=64 * n, out_bytes=2 * n)])
    assert res["ops"][0]["rc"] == 0 and [e for e in ev if e["op"] == "h2d"]


def test_zero_copy_is_refused_for_pageable_buffers_only_when_forced(mock_dir, tmp_path):
    op = dict(op="run_host", kernel=K_SHA256, nc=3, n=1000, unit_bytes=64, in_bytes=64000, out_bytes=32000)
    res, ev = run_child(mock_dir, tmp_path, [op], env_extra={"COAST_HOST_PATH": "zerocopy"})
    assert res["ops"][0]["rc"] != 0 and "pinned" in res["ops"][0]["err"]
    res, ev = run_child(mock_dir, tmp_path / "..", [op], env_extra={"COAST_HOST_PATH": "hybrid"})
    assert res["ops"][0]["rc"] != 0 and "pinned" in res["ops"][0]["err"]
    res, ev = run_child(mock_dir, tmp_path / "..", [op])                       # default: the staged pipeline
    assert res["ops"][0]["rc"] == 0 and [e for e in ev if e["op"] == "h2d"]


def test_host_call_stages_the_status_bytes_per_chunk(mock_dir, tmp_path):
    """ADVICE r01: kernels index status[] chunk-locally, so the host call must give every chunk its own device status
    buffer and copy it back to (host status + units done)"""
    n = 300001
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host_status", kernel=K_AES128, nc=2, n=n, in_bytes=16 * n, out_bytes=16 * n),
                                             dict(op="shutdown")])
    r = res["ops"][0]
    assert r["rc"] == 0 and not [e for e in ev if e["op"] == "error"]
    launches = [args_of(e) for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert len(launches) > 1 and all(a.status not in (0, r["host_status"]) for a in launches)
    _contiguous([(e["host"] - r["host_status"], e["bytes"]) for e in ev if e["op"] == "d2h" and 0 <= e["host"] - r["host_status"] < n], n)
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_host_call_chunks_are_bounded_in_bytes(mock_dir, tmp_path):
    """ADVICE r01: 1024-unit floor x 48 MiB streams used to ask for hundreds of GiB; a unit above the byte bound is its own chunk"""
    big, n = 48 << 20, 5
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host", kernel=K_CHSTONE_SHA, nc=3, n=n, unit_bytes=big, in_bytes=n * big, out_bytes=n * 20),
                                             dict(op="shutdown")])
    assert res["ops"][0]["rc"] == 0, res
    launches = [args_of(e) for e in ev if e["op"] == "launch" and "_nc" in e["name"]]
    assert [a.n_units for a in launches] == [1] * n and max(e["bytes"] for e in ev if e["op"] == "alloc") <= big + 4096
    assert ev[-1] == {"op": "exit", "live_allocations": 0}


def test_a_failing_chunk_drains_the_copies_already_queued(mock_dir, tmp_path):
    """the host call must not return while earlier chunks' copies are still in flight on the caller's buffers: after a driver failure
    in a later chunk (here: a staging allocation above the mock box's 6 GiB) the streams are synchronised before the error comes back"""
    big, n = 5 << 30, 2                                                         # first slot fits, the second does not
    res, ev = run_child(mock_dir, tmp_path, [dict(op="run_host", kernel=K_CHSTONE_SHA, nc=3, n=n, unit_bytes=1 << 28, in_bytes=n << 28, out_bytes=n * 20)],
                        env_extra={"COAST_HOST_CHUNK_BYTES": str(1 << 28), "MOCK_CUDA_FAIL_ALLOC_AFTER": "6"})
    r = res["ops"][0]
    if r["rc"] != 0:                                                            # the injected failure fired mid-schedule
        syncs = [i for i, e in enumerate(ev) if e["op"] == "stream_sync"]
        last_copy = max(i for i, e in enumerate(ev) if e["op"] in ("h2d", "d2h", "launch"))
        assert syncs and max(syncs) > last_copy, "error returned without draining the host-call streams"


def test_single_caller_guard(mock_dir, tmp_path):
    res, ev = run_child(mock_dir, tmp_path, [dict(op="two_threads", iters=20000)])
    r = res["ops"][0]
    assert set(r["codes"]) <= {0, -100005} and 0 in r["codes"] and r["after"] == 0


def test_sha256_entry_point_writes_the_callers_ctx_scratch(mock_dir, tmp_path):
    """ADVICE r01: sha256_hash leaves ctx_state / ctx_bitlen / ctx_data behind (sha256_common_tmr.c:101-180); ctx_state must be
    the big-endian words of the digest the launch returned, bitlen = 8*len and ctx_data the last padded block"""
    res, ev = run_child(mock_dir, tmp_path, [dict(op="sha_ctx", lens=[10, 55, 56, 64, 119, 200])])
    for rec in res["ops"][0]["recs"]:
        ln = rec["len"]
        assert rec["bitlen"] == [(8 * ln) & 0xFFFFFFFF, ln >> 29]
        assert rec["state"] == [int.from_bytes(bytes(rec["digest"][4 * i:4 * i + 4]), "big") for i in range(8)]
        rem = ln % 64
        want = (bytes((i * 3 + 1) & 0xFF for i in range(ln - rem, ln)) + b"\x80" + bytes(55 - rem)) if rem < 56 else bytes(56)
        want += (8 * ln).to_bytes(8, "big")
        assert bytes(rec["data"]) == want, (ln, rec["data"])
