#!/usr/bin/env python3
"""Generate tests/golden/coast_golden.json from the REFERENCE ITSELF, run here.

Everything in the fixture is produced by executing byuccl/coast's own C sources, compiled
where they lie under /root/reference/tests by oracle/Makefile into oracle/_ref (see
oracle/ref/*.c).  /root/reference does not exist on the GPU box, so the outputs are
committed as a small fixture next to this script:

    python tests/golden/make_golden.py        # needs /root/reference

Contents
  crc16   : the shipped message (crc16.c:14) and crc16() of it, plus 64 random messages
  sha256  : 10-byte KAT (sha256_common/sha_data.inc), 4000-byte KAT (hifive1/sha256.tmr/sha_data.inc),
            reference digests of messages of every length 0..130 (padding edge cases 55/56/63/64/119/120)
  aes     : the 568 NIST AESAVS records of tests/aes/ECB*.h (80 bytes each: key|key2|cipher|plain|input),
            and what aes_enc_dec() leaves in state[] and key[] for each direction
  mm      : mm_tmr.c 9x9 uint32 operands, results_matrix, xor_golden; matrixMultiply.c int operands/results
  chaes   : tests/chstone/aes: the benchmark's FIPS-197 vector through the reference's own encrypt()/decrypt(), 40 random
            (block, key) pairs both directions, DWC/TMR runs of the reference functions with a flipped input byte in one replica
  chsha   : tests/chstone/sha: the golden outData of sha_driver.c and the SHA-256 of its 16 KiB indata, reference
            digests of Philox streams of several lengths, and TMR/DWC runs with input flips
  qsort   : tests/quicksort: the benchmark's own 580-int input (srand(0)) with the SHA-256 of what quick_sort() makes of it,
            and reference outputs for random arrays of several lengths (duplicates, extremes)
  xmr     : TMR/DWC runs of the reference functions with a single-bit flip in ONE replica's private
            copy of its input (the only fault sites reachable without editing reference sources)

Next to it, data the tests would otherwise read out of the reference checkout:
  chstone_sha_indata.bin : the 2 x 8192-byte input of tests/chstone/sha (sha_data.c), as the benchmark hashes it
  reference_programs.json: the OPT_PASSES sweep of unittest/cfg/full.yml, and the scope facts (directives, definitions,
                           calls) the BOARD=b200 pass reads out of tests/matrixMultiply and tests/sha256_common/sha256_tmr.c
"""
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402


def hexs(b):
    return bytes(b).hex()


def main():
    assert os.path.exists("/root/reference/tests/crc16/crc16.c"), "needs the reference checkout"
    po.build()
    rng = np.random.default_rng(20260922)
    g = {"generator": "tests/golden/make_golden.py", "reference_commit": "397a26e"}

    # ---------------------------------------------------------------- crc16
    rc = po.ref("crc16")
    rc.ref_crc16.restype = C.c_ushort
    rc.ref_crc16.argtypes = [C.c_char_p, C.c_ubyte]
    msg = b"Automated TMR"
    crc = {"shipped_msg": hexs(msg), "shipped_crc": rc.ref_crc16(msg, len(msg)), "random": []}
    for i in range(64):
        n = int(rng.integers(1, 256))
        m = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        crc["random"].append([hexs(m), rc.ref_crc16(m, n)])
    g["crc16"] = crc

    # ---------------------------------------------------------------- sha256
    rs = po.ref("sha256")
    rs.ref_sha256_kat10_msg.restype = C.POINTER(C.c_uint8)
    rs.ref_sha256_kat10_golden.restype = C.POINTER(C.c_uint8)
    rs.ref_sha256.argtypes = [C.c_char_p, C.c_uint32, C.c_char_p]
    assert rs.ref_sha256_kat10() == 0
    r4 = po.ref("sha4000")
    r4.ref_sha4000_msg.restype = C.POINTER(C.c_uint8)
    r4.ref_sha4000_golden.restype = C.POINTER(C.c_uint8)
    r4.ref_sha4000_len.restype = C.c_uint32
    assert r4.ref_sha4000_kat() == 0
    n4 = r4.ref_sha4000_len()

    def ref_sha(m):
        out = C.create_string_buffer(32)
        rs.ref_sha256(m if m else b"\0", len(m), out)
        return out.raw

    sha = {
        "kat10_msg": hexs(rs.ref_sha256_kat10_msg()[:10]), "kat10_digest": hexs(rs.ref_sha256_kat10_golden()[:32]),
        "kat4000_msg": hexs(r4.ref_sha4000_msg()[:n4]), "kat4000_digest": hexs(r4.ref_sha4000_golden()[:32]),
        "by_length": [],
    }
    assert ref_sha(bytes.fromhex(sha["kat10_msg"])) == bytes.fromhex(sha["kat10_digest"])
    assert ref_sha(bytes.fromhex(sha["kat4000_msg"])) == bytes.fromhex(sha["kat4000_digest"])
    for n in range(0, 131):
        m = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        sha["by_length"].append([hexs(m), hexs(ref_sha(m))])
    g["sha256"] = sha

    # ---------------------------------------------------------------- aes
    ra = po.ref("aes")
    assert ra.ref_aes_kat_errors() == 0
    ra.ref_aes_kat_table.restype = C.POINTER(C.c_ubyte)
    ra.ref_aes_kat_table.argtypes = [C.c_int, C.POINTER(C.c_uint)]
    recs = []
    for k in range(4):
        cnt = C.c_uint()
        p = ra.ref_aes_kat_table(k, C.byref(cnt))
        recs.append(bytes(p[: cnt.value * 80]))
    allrec = b"".join(recs)
    assert len(allrec) == 568 * 80
    key_after_enc, key_after_dec = [], []
    for i in range(0, len(allrec), 80):
        r = allrec[i:i + 80]
        key, key2, cipher, plain, inp = r[0:16], r[16:32], r[32:48], r[48:64], r[64:80]
        st = C.create_string_buffer(inp, 16)
        kk = C.create_string_buffer(key, 16)
        ra.ref_aes_enc_dec(st, kk, 0)
        assert st.raw == cipher
        key_after_enc.append(kk.raw)
        kk2 = C.create_string_buffer(key2, 16)
        ra.ref_aes_enc_dec(st, kk2, 1)
        assert st.raw == plain
        key_after_dec.append(kk2.raw)
    g["aes"] = {"table_counts": [len(x) // 80 for x in recs], "records": hexs(allrec),
                "key_after_enc": hexs(b"".join(key_after_enc)), "key_after_dec": hexs(b"".join(key_after_dec))}

    # ---------------------------------------------------------------- mm
    rm = po.ref("mm")
    assert rm.ref_mm_error() == 0
    for f in ("ref_mm_first", "ref_mm_second", "ref_mm_results"):
        getattr(rm, f).restype = C.POINTER(C.c_uint32)
    rm.ref_mm_xor_golden.restype = C.c_uint32
    side = rm.ref_mm_side()
    ri = po.ref("mmint")
    assert ri.ref_mmint_run_main() == 0
    for f in ("ref_mmint_first", "ref_mmint_second"):
        getattr(ri, f).restype = C.POINTER(C.c_int32)
    ri.ref_mmint_results.restype = C.POINTER(C.c_uint32)
    g["mm"] = {
        "side": side,
        "u32_first": list(rm.ref_mm_first()[: side * side]), "u32_second": list(rm.ref_mm_second()[: side * side]),
        "u32_results": list(rm.ref_mm_results()[: side * side]), "xor_golden": rm.ref_mm_xor_golden(),
        "int_first": list(ri.ref_mmint_first()[: side * side]), "int_second": list(ri.ref_mmint_second()[: side * side]),
        "int_results": list(ri.ref_mmint_results()[: side * side]),
    }

    # ---------------------------------------------------------------- xMR with input-copy faults
    # SHA: 24 messages of 64 bytes; per unit one flip in replica r's private data[] copy.
    n = 24
    msgs = rng.integers(0, 256, (n, 64), dtype=np.uint8)
    faults = (po.RefFault * n)()
    plan = []
    for u in range(n):
        if u % 3 == 2:
            faults[u] = po.RefFault(0, -1, 0)
            plan.append(None)
        else:
            r_, by, bi = int(rng.integers(0, 3)), int(rng.integers(0, 64)), int(rng.integers(0, 8))
            faults[u] = po.RefFault(r_, by, bi)
            plan.append([r_, by, bi])
    xmr = {"sha_msgs": hexs(msgs.tobytes()), "sha_faults": plan, "sha_runs": {}}
    rs.ref_sha256_xmr.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int,
                                  C.c_void_p, C.POINTER(po.RefStats)]
    for nc in (2, 3):
        fl = (po.RefFault * n)()
        for u in range(n):
            fl[u] = faults[u] if (faults[u].byte < 0 or faults[u].replica < nc) else po.RefFault(0, -1, 0)
        out = np.zeros(n * 32, dtype=np.uint8)
        st = po.RefStats()
        st.first_fault_unit = po.NO_FAULT_UNIT
        rs.ref_sha256_xmr(msgs.ctypes.data, out.ctypes.data, n, 64, nc, 1, 1, fl, C.byref(st))
        xmr["sha_runs"][str(nc)] = {"out": hexs(out.tobytes()), "stats": st.as_dict()}
    # AES enc, one key: 32 blocks, flips in the replica's private state copy
    n = 32
    blocks = rng.integers(0, 256, (n, 16), dtype=np.uint8)
    key = rng.integers(0, 256, 16, dtype=np.uint8)
    faults = (po.RefFault * n)()
    plan = []
    for u in range(n):
        if u % 4 == 3:
            faults[u] = po.RefFault(0, -1, 0)
            plan.append(None)
        else:
            r_, by, bi = int(rng.integers(0, 2)), int(rng.integers(0, 16)), int(rng.integers(0, 8))
            faults[u] = po.RefFault(r_, by, bi)
            plan.append([r_, by, bi])
    ra.ref_aes_xmr.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_int,
                               C.c_int, C.c_void_p, C.POINTER(po.RefStats)]
    xmr.update({"aes_blocks": hexs(blocks.tobytes()), "aes_key": hexs(key.tobytes()), "aes_faults": plan, "aes_runs": {}})
    for nc in (2, 3):
        out = np.zeros(n * 16, dtype=np.uint8)
        st = po.RefStats()
        st.first_fault_unit = po.NO_FAULT_UNIT
        ra.ref_aes_xmr(blocks.ctypes.data, out.ctypes.data, n, key.ctypes.data, 0, 0, nc, 1, 1, faults, C.byref(st))
        xmr["aes_runs"][str(nc)] = {"out": hexs(out.tobytes()), "stats": st.as_dict()}
    # CRC16: 30 messages of 13 bytes
    n = 30
    msgs = rng.integers(0, 256, (n, 13), dtype=np.uint8)
    faults = (po.RefFault * n)()
    plan = []
    for u in range(n):
        if u % 5 == 4:
            faults[u] = po.RefFault(0, -1, 0)
            plan.append(None)
        else:
            r_, by, bi = int(rng.integers(0, 3)), int(rng.integers(0, 13)), int(rng.integers(0, 8))
            faults[u] = po.RefFault(r_, by, bi)
            plan.append([r_, by, bi])
    rc.ref_crc16_xmr.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int,
                                 C.c_void_p, C.POINTER(po.RefStats)]
    out = np.zeros(n, dtype=np.uint16)
    st = po.RefStats()
    st.first_fault_unit = po.NO_FAULT_UNIT
    rc.ref_crc16_xmr(msgs.ctypes.data, out.ctypes.data, n, 13, 3, 1, 1, faults, C.byref(st))
    xmr.update({"crc_msgs": hexs(msgs.tobytes()), "crc_faults": plan,
                "crc_run_tmr": {"out": [int(x) for x in out], "stats": st.as_dict()}})
    g["xmr"] = xmr

    # ---------------------------------------------------------------- chstone sha (appended last: the rng stream above is unchanged)
    import hashlib
    rh = po.ref("chsha")
    rh.ref_chsha_indata.restype = C.c_void_p
    rh.ref_chsha_golden.restype = C.POINTER(C.c_uint32)
    rh.ref_chsha.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    klen = int(rh.ref_chsha_len())
    indata = np.frombuffer((C.c_uint8 * klen).from_address(rh.ref_chsha_indata()), dtype=np.uint8).copy()
    dg = np.zeros(5, dtype=np.uint32)
    rh.ref_chsha(indata.ctypes.data, klen, dg.ctypes.data)
    assert [int(x) for x in dg] == [int(rh.ref_chsha_golden()[i]) for i in range(5)]      # sha_driver.c:45-46 outData
    ch = {"kat_len": klen, "kat_input_sha256": hashlib.sha256(indata.tobytes()).hexdigest(),
          "kat_digest": [int(x) for x in dg], "philox": []}
    for seed, ln in [(1, 64), (2, 128), (3, 192), (4, 1024), (5, 4096), (6, 16384), (7, 65536)]:
        d = po.fill_philox(ln // 4, 0, seed).view(np.uint8)
        rh.ref_chsha(d.ctypes.data, ln, dg.ctypes.data)
        ch["philox"].append({"seed": seed, "len": ln, "digest": [int(x) for x in dg]})
    n, ln = 12, 192
    msgs = po.fill_philox(n * ln // 4, 0, 77).view(np.uint8)
    faults = (po.RefFault * n)()
    plan = []
    for u in range(n):
        if u % 4 == 3:
            faults[u] = po.RefFault(0, -1, 0)
            plan.append(None)
        else:
            r_, by, bi = int(rng.integers(0, 3)), int(rng.integers(0, ln)), int(rng.integers(0, 8))
            faults[u] = po.RefFault(r_, by, bi)
            plan.append([r_, by, bi])
    rh.ref_chsha_xmr.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int,
                                 C.c_void_p, C.POINTER(po.RefStats)]
    ch.update({"xmr_seed": 77, "xmr_n": n, "xmr_len": ln, "xmr_faults": plan, "xmr_runs": {}})
    for nc in (3, 2):
        fl = (po.RefFault * n)(*[po.RefFault(f.replica, f.byte if f.replica < nc else -1, f.bit) for f in faults])
        out = np.zeros(5 * n, dtype=np.uint32)
        st = po.RefStats()
        st.first_fault_unit = po.NO_FAULT_UNIT
        rh.ref_chsha_xmr(msgs.ctypes.data, out.ctypes.data, n, ln, nc, 1, 1, fl, C.byref(st))
        ch["xmr_runs"][str(nc)] = {"out": [int(x) for x in out], "stats": st.as_dict()}
    g["chsha"] = ch

    # ---------------------------------------------------------------- quicksort (tests/quicksort/quicksort.c), appended last
    rq = po.ref("qsort")
    rq.ref_qsort_init.restype = C.POINTER(C.c_int)
    L = int(rq.ref_qsort_elements())
    assert rq.ref_qsort_selfcheck(0) == 0
    p_ = rq.ref_qsort_init(0)                               # the benchmark's own input: srand(0), 580 x rand()  (:93-115)
    inp = np.array([p_[i] for i in range(L)], dtype=np.int32)
    srt = inp.copy()
    rq.ref_quick_sort(srt.ctypes.data, L)
    qs = {"elements": L, "seed0_input": [int(v) for v in inp], "seed0_sorted_sha256": hashlib.sha256(srt.tobytes()).hexdigest(),
          "random": []}
    for ln in (1, 2, 3, 17, 100, 580, 1024):
        a_ = rng.integers(-2 ** 31, 2 ** 31 - 1, ln, dtype=np.int64).astype(np.int32)
        if ln == 100:
            a_ = (a_ % 7).astype(np.int32)                  # many duplicates
        b_ = a_.copy()
        rq.ref_quick_sort(b_.ctypes.data, ln)
        qs["random"].append({"input": [int(v) for v in a_], "sorted": [int(v) for v in b_]})
    g["qsort"] = qs

    # ---------------------------------------------------------------- chstone aes (tests/chstone/aes), appended last
    ra = po.ref("chaes")
    ra.ref_chaes.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    assert ra.ref_chaes_run_main() == 0                      # the benchmark as shipped prints RESULT: PASS
    st_ = np.zeros(32, dtype=np.int32); k_ = np.zeros(32, dtype=np.int32)
    st_[:16] = [50, 67, 246, 168, 136, 90, 48, 141, 49, 49, 152, 162, 224, 55, 7, 52]         # aes.c:93-108 = FIPS-197 Appendix B
    k_[:16] = [43, 126, 21, 22, 40, 174, 210, 166, 171, 247, 21, 136, 9, 207, 79, 60]         # aes.c:110-125
    ca = {"kat_plain": [int(v) for v in st_[:16]], "kat_key": [int(v) for v in k_[:16]], "random": []}
    assert ra.ref_chaes(st_.ctypes.data, k_.ctypes.data, 0) == 0                              # encrypt(): main_result unchanged
    ca["kat_cipher"] = [int(v) for v in st_[:16]]
    assert ra.ref_chaes(st_.ctypes.data, k_.ctypes.data, 1) == 0 and [int(v) for v in st_[:16]] == ca["kat_plain"]
    assert [int(v) for v in k_[:16]] == ca["kat_key"]        # the key is never modified
    for _ in range(40):
        blk = rng.integers(0, 256, 16, dtype=np.int64).astype(np.int32); key = rng.integers(0, 256, 16, dtype=np.int64).astype(np.int32)
        rec = {"block": [int(v) for v in blk], "key": [int(v) for v in key]}
        for d_, nm in ((0, "enc"), (1, "dec")):
            a_ = np.zeros(32, dtype=np.int32); kk = np.zeros(32, dtype=np.int32)
            a_[:16] = blk; kk[:16] = key
            ra.ref_chaes(a_.ctypes.data, kk.ctypes.data, d_)
            rec[nm] = [int(v) for v in a_[:16]]
        ca["random"].append(rec)
    n = 12
    blocks = rng.integers(0, 256, 16 * n, dtype=np.int64).astype(np.int32)
    keys = rng.integers(0, 256, 16 * n, dtype=np.int64).astype(np.int32)
    plan = []
    faults = (po.RefFault * n)()
    for u in range(n):
        if u % 4 == 3:
            faults[u] = po.RefFault(0, -1, 0); plan.append(None)
        else:
            r_, by, bi = int(rng.integers(0, 3)), int(rng.integers(0, 16)), int(rng.integers(0, 8))
            faults[u] = po.RefFault(r_, by, bi); plan.append([r_, by, bi])
    ra.ref_chaes_xmr.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_int,
                                 C.c_void_p, C.POINTER(po.RefStats)]
    ca.update({"xmr_n": n, "xmr_blocks": [int(v) for v in blocks], "xmr_keys": [int(v) for v in keys], "xmr_faults": plan, "xmr_runs": {}})
    for d_ in (0, 1):
        for nc in (3, 2):
            fl = (po.RefFault * n)(*[po.RefFault(f.replica, f.byte if f.replica < nc else -1, f.bit) for f in faults])
            out = np.zeros(16 * n, dtype=np.int32)
            st = po.RefStats()
            st.first_fault_unit = po.NO_FAULT_UNIT
            ra.ref_chaes_xmr(blocks.ctypes.data, out.ctypes.data, n, keys.ctypes.data, 1, d_, nc, 1, 1, fl, C.byref(st))
            ca["xmr_runs"][f"{d_}_{nc}"] = {"out": [int(x) for x in out], "stats": st.as_dict()}
    g["chaes"] = ca

    path = os.path.join(ROOT, "tests", "golden", "coast_golden.json")
    with open(path, "w") as f:
        json.dump(g, f, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes")

    path = os.path.join(ROOT, "tests", "golden", "chstone_sha_indata.bin")
    indata.tofile(path)
    print("wrote", path, os.path.getsize(path), "bytes")

    import yaml
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import build_reference_tests as brt
    brt.build_all()
    with open("/root/reference/unittest/cfg/full.yml") as f:
        progs = {"full_yml_opt_passes": yaml.safe_load(f)["OPT_PASSES"], "scope_facts": {}}
    for target in ("matrixMultiply", "sha256_tmr"):
        with open(os.path.join(brt.OUT, target, target + ".scope")) as f:
            progs["scope_facts"][target] = f.read()
    path = os.path.join(ROOT, "tests", "golden", "reference_programs.json")
    with open(path, "w") as f:
        json.dump(progs, f, indent=1)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
