"""GPU (B200): the CUDA path, called through the C ABI (libcoast_rt.so), against the CPU oracle on
the same seeded inputs -- bit-exact outputs AND equal counters, with and without injected faults --
and against the committed golden fixtures.  Integer/byte work: the bar is bit-exact."""
import hashlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

STAT_KEYS = ("errors_corrected", "dwc_detected", "syncs", "injected", "first_fault_unit")


def H(x):
    return bytes.fromhex(x)


def dev(rt, arr):
    import torch
    a = np.ascontiguousarray(arr)
    if a.dtype == np.uint32:
        a = a.view(np.int32)
    elif a.dtype == np.uint16:
        a = a.view(np.int16)
    return torch.from_numpy(a.copy()).cuda()


def host(t):
    return t.cpu().numpy().view(np.uint8) if t.dtype.itemsize == 1 else t.cpu().numpy()


def both(rt, oracle, kernel, nc, inp, n, *, flags=0, mode=0, unit_bytes=0, M=0, N=0, K=0, aux=None, key=None,
         plan_kw=None, table=None, unit_base=0):
    import coast_b200 as cb
    oplan = gplan = None
    if table is not None:
        oplan = oracle.make_plan(oracle.PLAN_TABLE, table=table)
        gplan = cb.FaultPlan(mode=cb.PLAN_TABLE, table=dev(rt, table))
    elif plan_kw:
        oplan = oracle.make_plan(oracle.PLAN_BERNOULLI, **plan_kw)
        gplan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, **plan_kw)     # seed + (p | threshold)
    o_out, o_st = oracle.run(kernel, nc, inp, n, flags=flags, mode=mode, unit_bytes=unit_bytes, M=M, N=N, K=K, aux=aux,
                             key=key, plan=oplan, unit_base=unit_base)
    g_out, g_st = rt.run(kernel, nc, dev(rt, inp), n, flags=flags, mode=mode, unit_bytes=unit_bytes, M=M, N=N, K=K,
                         aux=dev(rt, aux) if aux is not None else None, key=key, plan=gplan, unit_base=unit_base)
    g = host(g_out)
    assert g.tobytes() == o_out.tobytes(), f"output mismatch kernel={kernel} nc={nc} n={n}"
    gd = g_st.as_dict()
    for k in STAT_KEYS:
        assert gd[k] == o_st[k], (k, gd, o_st)
    return g, gd


def msgs(oracle, n, nbytes, seed):
    return oracle.fill_philox((n * nbytes + 3) // 4, 0, seed).view(np.uint8)[: n * nbytes].copy()


# ------------------------------------------------------------------------------------------ fill
def test_fill_philox_matches_oracle(rt, oracle):
    import torch
    for n_words, base in ((1, 0), (4, 0), (1000, 0), (1003, 5), (4096, 2), (7, 3)):
        t = torch.zeros(n_words, dtype=torch.int32, device="cuda")
        rt.fill_philox(t, seed=11, word_base=base)
        torch.cuda.synchronize()
        assert (t.cpu().numpy().view(np.uint32) == oracle.fill_philox(n_words, base, 11)).all()


# ------------------------------------------------------------------------------------------ sha256
@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("n", [1, 9, 10, 11, 79, 80, 81, 257, 5000])
def test_sha256_b64_zero_fault(rt, oracle, nc, n):
    m = msgs(oracle, n, 64, 2)
    g, st = both(rt, oracle, oracle.K_SHA256, nc, m, n, unit_bytes=64, flags=3)
    for u in (0, n // 2, n - 1):
        assert g[32 * u: 32 * u + 32].tobytes() == hashlib.sha256(m[64 * u: 64 * u + 64].tobytes()).digest()
    assert st["errors_corrected"] == 0 and st["dwc_detected"] == 0


@pytest.mark.parametrize("nc", [1, 2, 3])
def test_sha256_b64_bernoulli_faults(rt, oracle, nc):
    n = 4000
    m = msgs(oracle, n, 64, 2)
    g, st = both(rt, oracle, oracle.K_SHA256, nc, m, n, unit_bytes=64, flags=3, plan_kw=dict(seed=77, p=0.2))
    assert st["injected"] > 500
    if nc == 3:
        clean, _ = oracle.run(oracle.K_SHA256, 1, m, n, unit_bytes=64)
        assert g.tobytes() == clean.tobytes()          # every single fault is out-voted
        assert st["errors_corrected"] >= st["injected"]


def test_sha256_every_site_class_table_plan(rt, oracle):
    """one unit per enumerated site class and replica: m[] words, working vars at several rounds, ctx_state, both blocks"""
    sites = [0, 7, 15, 16, 16 + 8 * 5 + 3, 16 + 8 * 63 + 7, 528, 535, 536, 536 + 15, 536 + 16 + 8 * 31 + 4, 536 + 535]
    ent = [(r, s, b) for s in sites for r in range(3) for b in (0, 31)]
    n = len(ent) + 5
    m = msgs(oracle, n, 64, 4)
    for nc in (2, 3):
        tab = np.zeros(n, dtype=np.uint32)
        for u, (r, s, b) in enumerate(ent):
            tab[u] = oracle.fault_entry(r, s, b)       # replica 2 entries are ignored under DWC
        tab[-1] = oracle.fault_entry(0, 2000, 0)        # out-of-range site -> ignored
        tab[-2] = oracle.fault_entry(0, 3, 31) & ~0x80000000 & 0xFFFFFFFF   # valid bit clear -> ignored
        both(rt, oracle, oracle.K_SHA256, nc, m, n, unit_bytes=64, flags=3, table=tab)


@pytest.mark.parametrize("length", [1, 3, 10, 55, 56, 63, 65, 119, 120, 200])
def test_sha256_general_lengths(rt, oracle, length):
    n = 37
    m = msgs(oracle, n, length, 6)
    g, _ = both(rt, oracle, oracle.K_SHA256, 3, m, n, unit_bytes=length, flags=3, plan_kw=dict(seed=length, p=0.3))
    g1, _ = both(rt, oracle, oracle.K_SHA256, 1, m, n, unit_bytes=length)
    for u in range(n):
        assert g1[32 * u: 32 * u + 32].tobytes() == hashlib.sha256(m[length * u: length * u + length].tobytes()).digest()


def test_sha256_reference_kats(rt, oracle, golden):
    g = golden["sha256"]
    for key_m, key_d in (("kat10_msg", "kat10_digest"), ("kat4000_msg", "kat4000_digest")):
        m = np.frombuffer(H(g[key_m]), dtype=np.uint8)
        for nc in (1, 2, 3):
            out, st = rt.run(oracle.K_SHA256, nc, dev(rt, m), 1, unit_bytes=len(m), flags=3)
            assert host(out).tobytes() == H(g[key_d])
            assert st.errors_corrected == 0 and st.dwc_detected == 0     # "C:0 E:0 F:0" (sha256_tmr.c:30)


def test_sha256_unaligned_input_takes_general_path(rt, oracle):
    import torch
    n = 100
    m = msgs(oracle, n, 64, 9)
    buf = torch.zeros(n * 64 + 4, dtype=torch.uint8, device="cuda")
    buf[4:] = torch.from_numpy(m.copy()).cuda()
    out, _ = rt.run(oracle.K_SHA256, 3, buf[4:], n, unit_bytes=64)
    ref, _ = oracle.run(oracle.K_SHA256, 3, m, n, unit_bytes=64)
    assert host(out).tobytes() == ref.tobytes()


def test_sha256_full_size_properties(rt, oracle):
    """BASELINE config 2: 2^20 x 64-byte messages.  Size-independent properties: digests equal hashlib on a
    sample; TMR under a p=2^-6 fault plan gives bit-identical output to the fault-free run; counters equal the
    oracle's on the first 2^15 units' worth of the same plan (prefix run with the same unit_base)."""
    import torch
    import coast_b200 as cb
    n = 1 << 20
    d_in = torch.empty(n * 64, dtype=torch.uint8, device="cuda")
    rt.fill_philox(d_in, seed=2)
    clean, st0 = rt.run(cb.K_SHA256, 3, d_in, n, unit_bytes=64, flags=3)
    assert st0.errors_corrected == 0 and st0.syncs == 32 * n
    plan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=22, p=2 ** -6)
    faulty, st1 = rt.run(cb.K_SHA256, 3, d_in, n, unit_bytes=64, flags=3, plan=plan)
    assert torch.equal(clean, faulty)
    assert abs(st1.injected - n / 64) < 6 * (n / 64) ** 0.5
    unp, _ = rt.run(cb.K_SHA256, 1, d_in, n, unit_bytes=64)
    assert torch.equal(clean, unp)
    h_in = d_in.cpu().numpy()
    h_out = clean.cpu().numpy()
    for u in list(range(0, n, 65537)) + [n - 1]:
        assert h_out[32 * u: 32 * u + 32].tobytes() == hashlib.sha256(h_in[64 * u: 64 * u + 64].tobytes()).digest()
    k = 1 << 15
    _, so = oracle.run(oracle.K_SHA256, 3, h_in[: 64 * k], k, unit_bytes=64, flags=3,
                       plan=oracle.make_plan(oracle.PLAN_BERNOULLI, seed=22, p=2 ** -6), threads=8)
    _, sg = rt.run(cb.K_SHA256, 3, d_in[: 64 * k], k, unit_bytes=64, flags=3, plan=plan)
    assert sg.as_dict() == so


# ------------------------------------------------------------------------------------------ aes
@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("n", [1, 15, 16, 17, 319, 320, 321, 512, 1025, 6000])
def test_aes_enc_zero_fault(rt, oracle, nc, n):
    blocks = msgs(oracle, n, 16, 3)
    both(rt, oracle, oracle.K_AES128, nc, blocks, n, key=bytes(range(16)), flags=3)


@pytest.mark.parametrize("nc", [1, 2, 3])
def test_aes_enc_bernoulli_faults_detect_rate(rt, oracle, nc):
    n = 20000
    blocks = msgs(oracle, n, 16, 3)
    g, st = both(rt, oracle, oracle.K_AES128, nc, blocks, n, key=bytes(16), flags=3, plan_kw=dict(seed=33, p=0.05))
    if nc == 2:
        assert st["dwc_detected"] == st["injected"] > 500    # every state flip propagates (bijective rounds)


def test_aes_every_site_table_plan(rt, oracle):
    ent = [(r, s, b) for s in range(176) for r in (0, 1, 2) for b in (0, 7)]
    n = len(ent)
    blocks = msgs(oracle, n, 16, 5)
    tab = np.array([oracle.fault_entry(r, s, b) for (r, s, b) in ent], dtype=np.uint32)
    for nc in (2, 3):
        both(rt, oracle, oracle.K_AES128, nc, blocks, n, key=bytes(range(1, 17)), flags=3, table=tab)        # T-table kernel
        both(rt, oracle, oracle.K_AES128, nc, blocks, n, key=bytes(range(1, 17)), flags=3, table=tab, mode=1)  # decrypt, byte-wise kernel


def test_aes_568_nist_kats_on_device(rt, oracle, golden):
    """aes_test() (tests/aes/aes.c:29-103) on the GPU: encrypt with key, compare to cipher; decrypt with key2, compare to plain."""
    rec = np.frombuffer(H(golden["aes"]["records"]), dtype=np.uint8).reshape(568, 80)
    keys, keys2, cipher, plain, inp = (np.ascontiguousarray(rec[:, 16 * i: 16 * i + 16]) for i in range(5))
    for nc in (1, 2, 3):
        enc, st = rt.run(oracle.K_AES128, nc, dev(rt, inp), 568, mode=oracle.AES_KEY_PER_UNIT, aux=dev(rt, keys), flags=3)
        assert host(enc).tobytes() == cipher.tobytes()
        dec, st2 = rt.run(oracle.K_AES128, nc, enc, 568, mode=oracle.AES_KEY_PER_UNIT | oracle.AES_DECRYPT, aux=dev(rt, keys2), flags=3)
        assert host(dec).tobytes() == plain.tobytes()
        assert st.errors_corrected == st.dwc_detected == st2.errors_corrected == st2.dwc_detected == 0   # "Number of errors: 0"
    # single-key T-table kernel on the VarTxt table (all-zero key, aes/ECBVarTxt128.h)
    vt = rec[14 + 42 + 256:]
    assert not vt[:, :16].any()
    enc, _ = rt.run(oracle.K_AES128, 2, dev(rt, np.ascontiguousarray(vt[:, 64:80])), 256, key=bytes(16))
    assert host(enc).tobytes() == np.ascontiguousarray(vt[:, 32:48]).tobytes()


def test_aes_decrypt_and_per_unit_keys_with_faults(rt, oracle):
    n = 3000
    blocks = msgs(oracle, n, 16, 3)
    keys = msgs(oracle, n, 16, 8)
    for mode in (oracle.AES_DECRYPT, oracle.AES_KEY_PER_UNIT, oracle.AES_KEY_PER_UNIT | oracle.AES_DECRYPT):
        both(rt, oracle, oracle.K_AES128, 2, blocks, n, key=bytes(range(16)), mode=mode, flags=3,
             aux=keys if mode & oracle.AES_KEY_PER_UNIT else None, plan_kw=dict(seed=5, p=0.1))
        both(rt, oracle, oracle.K_AES128, 3, blocks, n, key=bytes(range(16)), mode=mode, flags=3,
             aux=keys if mode & oracle.AES_KEY_PER_UNIT else None, plan_kw=dict(seed=6, p=0.1))


def test_aes_full_size_roundtrip_and_detect_rate(rt, oracle):
    """BASELINE config 3: 2^24 blocks, DWC, Bernoulli(2^-10) flips.  Properties: decrypt(encrypt(x)) == x over the
    full buffer; dwc_detected == injected (detect-rate parity: 100% of state flips); prefix counters == oracle."""
    import torch
    import coast_b200 as cb
    n = 1 << 24
    d_in = torch.empty(n * 16, dtype=torch.uint8, device="cuda")
    rt.fill_philox(d_in, seed=3)
    key = bytes(16)
    enc, st = rt.run(cb.K_AES128, 2, d_in, n, key=key)
    assert st.dwc_detected == 0
    dec, _ = rt.run(cb.K_AES128, 1, enc, n, key=key, mode=cb.AES_DECRYPT)
    assert torch.equal(dec, d_in)
    plan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=33, p=2 ** -10)
    enc_f, st_f = rt.run(cb.K_AES128, 2, d_in, n, key=key, plan=plan)
    assert st_f.dwc_detected == st_f.injected
    assert abs(st_f.injected - n / 1024) < 6 * (n / 1024) ** 0.5
    k = 1 << 16
    o_out, so = oracle.run(oracle.K_AES128, 2, d_in[: 16 * k].cpu().numpy(), k, key=key,
                           plan=oracle.make_plan(oracle.PLAN_BERNOULLI, seed=33, p=2 ** -10), threads=8)
    g_out, sg = rt.run(cb.K_AES128, 2, d_in[: 16 * k], k, key=key, plan=plan)
    assert sg.as_dict() == so and host(g_out).tobytes() == o_out.tobytes()


# ------------------------------------------------------------------------------------------ crc16
def test_crc16_shipped_message(rt, oracle, golden):
    m = np.frombuffer(H(golden["crc16"]["shipped_msg"]), dtype=np.uint8)
    for nc in (1, 2, 3):
        out, st = rt.run(oracle.K_CRC16, nc, dev(rt, m), 1, unit_bytes=13, flags=3)
        assert int(host(out).view(np.uint16)[0]) == 0x5BA3           # "result: 5ba3"
    for mh, c in golden["crc16"]["random"]:
        mm = np.frombuffer(H(mh), dtype=np.uint8)
        out, _ = rt.run(oracle.K_CRC16, 3, dev(rt, mm), 1, unit_bytes=len(mm))
        assert int(host(out).view(np.uint16)[0]) == c


@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("length,n", [(64, 1), (64, 81), (64, 3000), (13, 500), (1, 40), (255, 100), (48, 77)])
def test_crc16_faults(rt, oracle, nc, length, n):
    m = msgs(oracle, n, length, 1)
    both(rt, oracle, oracle.K_CRC16, nc, m, n, unit_bytes=length, flags=3)
    both(rt, oracle, oracle.K_CRC16, nc, m, n, unit_bytes=length, flags=3, plan_kw=dict(seed=length, p=0.3))


def test_crc16_full_size(rt, oracle):
    import torch
    import coast_b200 as cb
    n = 1 << 20
    d_in = torch.empty(n * 64, dtype=torch.uint8, device="cuda")
    rt.fill_philox(d_in, seed=1)
    a, _ = rt.run(cb.K_CRC16, 1, d_in, n, unit_bytes=64)
    b, st = rt.run(cb.K_CRC16, 3, d_in, n, unit_bytes=64, flags=3, plan=cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=4, p=0.01))
    assert torch.equal(a, b) and st.errors_corrected == st.injected      # one u16 vote per unit; every crc/data flip shows
    k = 1 << 14
    o, _ = oracle.run(oracle.K_CRC16, 1, d_in[: 64 * k].cpu().numpy(), k, unit_bytes=64)
    assert host(a[: 2 * k]).tobytes() == o.tobytes()


# ------------------------------------------------------------------------------------------ matmul (exact)
def test_mm_reference_9x9(rt, oracle, golden):
    g = golden["mm"]
    A, B = np.array(g["u32_first"], dtype=np.uint32), np.array(g["u32_second"], dtype=np.uint32)
    for nc in (1, 2, 3):
        out, st = rt.run(oracle.K_MM_U32, nc, dev(rt, A), 81, M=9, N=9, K=9, aux=dev(rt, B), flags=3)
        C = host(out).view(np.uint32)
        assert list(C) == g["u32_results"] and int(np.bitwise_xor.reduce(C)) == g["xor_golden"]   # "Error?: 0"
    Ai = np.array(g["int_first"], dtype=np.int32).view(np.uint32)
    Bi = np.array(g["int_second"], dtype=np.int32).view(np.uint32)
    out, _ = rt.run(oracle.K_MM_U32, 2, dev(rt, Ai), 81, M=9, N=9, K=9, aux=dev(rt, Bi))
    assert list(host(out).view(np.uint32)) == g["int_results"]                                    # "Number of errors: 0"


@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("M,N,K", [(9, 9, 9), (17, 33, 5), (64, 64, 64), (100, 130, 70)])
def test_mm_faults(rt, oracle, nc, M, N, K):
    A = oracle.fill_philox(M * K, 0, 4)
    B = oracle.fill_philox(K * N, 0, 44)
    both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3)
    both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3, plan_kw=dict(seed=M, p=0.2))


# ------------------------------------------------------------------------------------------ ABI behaviour on the GPU
def test_counters_fold_into_reference_globals(rt, oracle):
    before_e, before_s = rt.tmr_error_cnt, rt.sync_count
    n = 300
    m = msgs(oracle, n, 64, 2)
    _, st = both(rt, oracle, oracle.K_SHA256, 3, m, n, unit_bytes=64, flags=3, plan_kw=dict(seed=1, p=0.5))
    assert rt.tmr_error_cnt == (before_e + st["errors_corrected"]) & 0xFFFFFFFF       # i32 TMR_ERROR_CNT
    assert rt.sync_count == before_s + st["syncs"]                                     # i64 __SYNC_COUNT


def test_majority_voter_extension(rt, oracle):
    n = 500
    m = msgs(oracle, n, 64, 2)
    both(rt, oracle, oracle.K_SHA256, 3, m, n, unit_bytes=64, flags=3 | 0x100, plan_kw=dict(seed=3, p=0.4))


def test_run_host_matches_device_path(rt, oracle):
    import torch
    import coast_b200 as cb
    n = 300000
    h_in = torch.from_numpy(msgs(oracle, n, 64, 2)).pin_memory()
    h_out = torch.empty(n * 32, dtype=torch.uint8).pin_memory()
    plan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=9, p=0.01)
    st = rt.run_host(cb.K_SHA256, 3, h_in, h_out, n, unit_bytes=64, flags=3, plan=plan)
    d_out, st2 = rt.run(cb.K_SHA256, 3, h_in.cuda(), n, unit_bytes=64, flags=3, plan=plan)
    assert torch.equal(d_out.cpu(), h_out) and st.as_dict() == st2.as_dict()
    # AES through the host path, DWC with faults: never aborts in the noabort flavour
    hb = torch.from_numpy(msgs(oracle, n, 16, 3)).pin_memory()
    ho = torch.empty(n * 16, dtype=torch.uint8).pin_memory()
    st = rt.run_host(cb.K_AES128, 2, hb, ho, n, key=bytes(16), plan=plan)
    o, so = oracle.run(oracle.K_AES128, 2, hb.numpy(), n, key=bytes(16), plan=oracle.make_plan(oracle.PLAN_BERNOULLI, seed=9, p=0.01), threads=8)
    assert ho.numpy().tobytes() == o.tobytes() and st.as_dict() == so


@pytest.mark.parametrize("case", ["sha64", "sha100", "sha0", "crc64", "crc13", "aes_enc", "aes_dec_keys", "chsha"])
def test_host_call_zero_copy_and_staged_agree_with_the_oracle(rt, oracle, case):
    """coast_run_host(): pinned buffers -> ONE zero-copy launch on the mapped host memory (TMA / vector loads over PCIe, voted
    output and per-unit status written straight to host memory); pageable buffers -> the staged chunk pipeline.  Same bytes,
    same counters, same per-unit status as the oracle on both, with injected faults."""
    import torch
    import coast_b200 as cb
    n = 70001
    kw, okw = {}, {}
    if case.startswith("sha"):
        ub = {"sha64": 64, "sha100": 100, "sha0": 0}[case]
        kernel, nc, ob = cb.K_SHA256, 3, 32
        inp = msgs(oracle, n, ub, 2) if ub else np.zeros(16, dtype=np.uint8)
        kw = okw = dict(unit_bytes=ub, flags=3)
    elif case.startswith("crc"):
        ub = 64 if case == "crc64" else 13
        kernel, nc, ob = cb.K_CRC16, 3, 2
        inp = msgs(oracle, n, ub, 1)
        kw = okw = dict(unit_bytes=ub, flags=3)
    elif case == "aes_enc":
        kernel, nc, ob = cb.K_AES128, 2, 16
        inp = msgs(oracle, n, 16, 3)
        kw = okw = dict(key=bytes(range(16)))
    elif case == "aes_dec_keys":
        kernel, nc, ob = cb.K_AES128, 3, 16
        inp = msgs(oracle, n, 16, 3)
        keys = msgs(oracle, n, 16, 5)
        kw = dict(mode=cb.AES_DECRYPT | cb.AES_KEY_PER_UNIT, flags=1)
        okw = dict(mode=cb.AES_DECRYPT | cb.AES_KEY_PER_UNIT, flags=1, aux=keys)
    else:
        n = 3001
        kernel, nc, ob = cb.K_CHSTONE_SHA, 3, 20
        inp = msgs(oracle, n, 256, 6)
        kw = okw = dict(unit_bytes=256, flags=3)
    p = 0.02
    o_out, o_st = oracle.run(kernel, nc, inp, n, plan=oracle.make_plan(oracle.PLAN_BERNOULLI, seed=21, p=p), unit_base=123, **okw)
    plan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=21, p=p)
    import os
    for pinned, path in ((True, "zerocopy"), (True, "hybrid"), (True, "staged"), (False, None)):
        if path:
            os.environ["COAST_HOST_PATH"] = path
        else:
            os.environ.pop("COAST_HOST_PATH", None)
        if case == "sha0" and path == "hybrid":
            continue                                        # nothing to read: there is no input to alias
        mk = (lambda a: torch.from_numpy(a.copy()).pin_memory()) if pinned else (lambda a: a.copy())
        h_in = mk(inp)
        h_out = mk(np.zeros(n * ob, dtype=np.uint8))
        h_aux = mk(keys) if case == "aes_dec_keys" else None
        h_status = mk(np.full(n, 0xEE, dtype=np.uint8))
        d = rt.make_desc(kernel, nc, h_in.data_ptr() if pinned else h_in.ctypes.data, h_out.data_ptr() if pinned else h_out.ctypes.data, n,
                         plan=plan, unit_base=123, d_aux=(h_aux.data_ptr() if pinned else h_aux.ctypes.data) if h_aux is not None else None,
                         d_status=h_status.data_ptr() if pinned else h_status.ctypes.data, **kw)
        import ctypes as C
        from coast_b200.runtime import _Stats
        st = _Stats()
        rc = rt.L.coast_run_host_noabort(C.byref(d), C.byref(st))
        os.environ.pop("COAST_HOST_PATH", None)
        assert rc == 0, rt.L.coast_last_error()
        assert rt.last_host_path == (path or "staged")
        got = h_out.numpy() if pinned else h_out
        assert got.tobytes() == o_out.tobytes(), (case, path)
        assert {k: getattr(st, k) for k in STAT_KEYS} == {k: o_st[k] for k in STAT_KEYS}, (case, path)
        status = h_status.numpy() if pinned else h_status
        bad_units = int((status != 0).sum())
        assert int(status.max()) <= 32                              # every byte was written (0xEE poison gone)
        if nc == 2:
            assert bad_units == o_st["dwc_detected"]
        else:
            assert int(status.astype(np.int64).sum()) == o_st["errors_corrected"]


@pytest.mark.parametrize("kernel", ["gemm", "mm"])
def test_matmul_host_call_row_blocks_equal_the_device_launch(rt, oracle, kernel):
    """coast_run_host() pipelines a large matmul by C row blocks (B once, A rows up / launch / C rows down per block on rotating
    streams); the plan is keyed by the global element index, so outputs AND counters equal one launch on device buffers"""
    import torch
    import coast_b200 as cb
    M, N, K = 1024, 256, 256
    if kernel == "gemm":
        A = (oracle.fill_philox(M * K, 0, 4).astype(np.float64) / 2 ** 31 - 1.0).astype(np.float32)
        B = (oracle.fill_philox(K * N, 0, 44).astype(np.float64) / 2 ** 31 - 1.0).astype(np.float32)
        kid = cb.K_GEMM_TF32
    else:
        A, B, kid = oracle.fill_philox(M * K, 0, 4), oracle.fill_philox(K * N, 0, 44), cb.K_MM_U32
    plan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=5, p=0.001)
    d_out, st_dev = rt.run(kid, 3, dev(rt, A), M * N, flags=3, M=M, N=N, K=K, aux=dev(rt, B), plan=plan, unit_base=40)
    h_a, h_b = torch.from_numpy(A.view(np.int32).copy()).pin_memory(), torch.from_numpy(B.view(np.int32).copy()).pin_memory()
    h_c = torch.zeros(M * N, dtype=torch.int32).pin_memory()
    st = rt.run_host(kid, 3, h_a, h_c, M * N, flags=3, M=M, N=N, K=K, h_aux=h_b, plan=plan, unit_base=40)
    assert rt.last_host_path == "row-blocks"
    assert h_c.numpy().tobytes() == d_out.cpu().numpy().tobytes() and st.as_dict() == st_dev.as_dict() and st.injected > 0


@pytest.mark.parametrize("nc", [2, 3])
@pytest.mark.parametrize("flagname", ["F_STORE_DATA_SYNC", "F_NO_MEM_REPLICATION"])
def test_store_votes_crc16_mm_and_sha256_match_the_oracle(rt, oracle, nc, flagname):
    """8f-1: -storeDataSync / -noMemReplication = votes on every assignment inside the loops (oracle: sv_crc16_unit / sv_mm_elem);
    outputs, corrected-error count, __SYNC_COUNT and the per-unit status all equal the oracle, zero-fault and under faults at
    every site class; lengths include 64 (the table kernel must NOT be picked) and the 13-byte reference message"""
    import coast_b200 as cb
    extra = getattr(cb, flagname)
    for L, n in ((13, 777), (64, 5000), (255, 100)):
        m = msgs(oracle, n, L, 1)
        g, st = both(rt, oracle, oracle.K_CRC16, nc, m, n, unit_bytes=L, flags=3 | extra)
        assert st["syncs"] == (n * (3 * L + 1) if nc == 3 else 0)
        g, st = both(rt, oracle, oracle.K_CRC16, nc, m, n, unit_bytes=L, flags=3 | extra, plan_kw=dict(seed=4, p=0.3))
        assert st["injected"] > 0 and (st["errors_corrected"] == st["injected"] if nc == 3 else st["dwc_detected"] > 0)
    sites = np.arange(26, dtype=np.uint32)
    table = np.array([oracle.fault_entry(int(s) % nc, int(s), int(s) % 8) for s in sites], dtype=np.uint32)
    both(rt, oracle, oracle.K_CRC16, nc, msgs(oracle, 26, 13, 1), 26, unit_bytes=13, flags=3 | extra, table=table)
    for (M, N, K) in ((9, 9, 9), (64, 128, 32), (128, 64, 128)):          # the tiled / tensor-core shapes must fall back to the plain kernel
        A, B = oracle.fill_philox(M * K, 0, 4), oracle.fill_philox(K * N, 0, 44)
        g, st = both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, flags=3 | extra, M=M, N=N, K=K, aux=B, plan_kw=dict(seed=6, p=0.2))
        assert st["syncs"] == (M * N * (K + 1) if nc == 3 else 0)
    # -noStoreDataSync switches the in-loop votes off again
    g, st = both(rt, oracle, oracle.K_CRC16, 3, msgs(oracle, 100, 13, 1), 100, unit_bytes=13, flags=3 | extra | cb.F_NO_STORE_DATA_SYNC)
    assert st["syncs"] == 100
    # sha256: len + 720 votes per compression + 32; lengths around the padding edges, aligned (64: NOT the TMA kernel) and ragged
    for L, n in ((64, 700), (10, 300), (55, 100), (56, 100), (119, 64), (128, 200)):
        m = msgs(oracle, n, L, 2)
        g, st = both(rt, oracle, oracle.K_SHA256, nc, m, n, unit_bytes=L, flags=3 | extra)
        assert st["syncs"] == (n * (L + 720 * ((L + 8) // 64 + 1) + 32) if nc == 3 else 0)
        both(rt, oracle, oracle.K_SHA256, nc, m, n, unit_bytes=L, flags=3 | extra, plan_kw=dict(seed=8, p=0.5))
    n = 1072
    table = np.array([oracle.fault_entry(u % nc, u, (u * 7) % 32) for u in range(n)], dtype=np.uint32)
    both(rt, oracle, oracle.K_SHA256, nc, msgs(oracle, n, 64, 2), n, unit_bytes=64, flags=3 | extra, table=table)


def test_reference_entry_points(rt, oracle, golden):
    """the four functions the unchanged reference tests call (BOARD=b200 flow), under -TMR -countErrors"""
    import ctypes as C
    L = rt.L
    assert L.coast_set_opt_passes(b"-TMR -countErrors") == 0
    assert L.coast_xmr_crc16(b"Automated TMR", 13) == 0x5BA3
    g = golden["sha256"]
    msg = C.create_string_buffer(H(g["kat10_msg"]), 10)
    digest = C.create_string_buffer(32)
    cd, bl, stt = C.create_string_buffer(64), (C.c_uint32 * 2)(), (C.c_uint32 * 8)()
    L.coast_xmr_sha256_hash(cd, bl, stt, msg, 10, digest)
    assert digest.raw == H(g["kat10_digest"])
    rec = H(golden["aes"]["records"])[:80]
    state, key = C.create_string_buffer(rec[64:80], 16), C.create_string_buffer(rec[0:16], 16)
    L.coast_xmr_aes_enc_dec(state, key, 0)
    assert state.raw == rec[32:48]
    key2 = C.create_string_buffer(rec[16:32], 16)
    L.coast_xmr_aes_enc_dec(state, key2, 1)
    assert state.raw == rec[48:64]
    mm = golden["mm"]
    A = (C.c_uint32 * 81)(*mm["u32_first"]); B = (C.c_uint32 * 81)(*mm["u32_second"]); R = (C.c_uint32 * 81)()
    L.coast_xmr_matrix_multiply_u32(A, B, R, 9)
    assert list(R) == mm["u32_results"]


# ------------------------------------------------------------------------------------------ edge cases
def test_empty_and_degenerate_inputs(rt, oracle):
    import torch
    import coast_b200 as cb
    dummy = torch.zeros(64, dtype=torch.uint8, device="cuda")
    out = torch.zeros(64, dtype=torch.uint8, device="cuda")
    # n_units == 0 is a no-op, not an error
    d = rt.make_desc(cb.K_SHA256, 3, dummy, out, 0, unit_bytes=64)
    rt.launch(d)
    st = rt.sync()
    assert st.as_dict() == cb.Stats().as_dict()
    # the empty message (unit_bytes == 0)
    o, _ = rt.run(cb.K_SHA256, 3, dummy, 5, unit_bytes=0, flags=3)
    assert host(o)[:32].tobytes() == hashlib.sha256(b"").digest() and host(o)[128:160].tobytes() == hashlib.sha256(b"").digest()
    # crc16's length is an `unsigned char` (crc16.c:21): 0 and >255 are rejected loudly
    for bad in (0, 256):
        with pytest.raises(cb.CoastError):
            rt.run(cb.K_CRC16, 3, dummy, 1, unit_bytes=bad)
    with pytest.raises(cb.CoastError):
        rt.run(cb.K_SHA256, 4, dummy, 1, unit_bytes=64)            # num_clones must be 1, 2 or 3
    with pytest.raises(cb.CoastError):
        rt.run(cb.K_GEMM_TF32, 3, dummy, 100 * 100, M=100, N=100, K=100, aux=dummy)   # tile constraint stated, not silently padded


def test_sha256_long_message_multi_block_faults_in_late_blocks(rt, oracle):
    """4000-byte messages = 63 compressions: fault sites in every block index are reachable and agree with the oracle"""
    n, L = 12, 4000
    m = msgs(oracle, n, L, 12)
    ns = oracle.fault_sites(oracle.K_SHA256, L)
    assert ns == 63 * 536
    tab = np.zeros(n, dtype=np.uint32)
    for u in range(n):
        tab[u] = oracle.fault_entry(u % 3, (u * 2999 + 17) % ns, (u * 7) % 32)
    both(rt, oracle, oracle.K_SHA256, 3, m, n, unit_bytes=L, flags=3, table=tab)
    both(rt, oracle, oracle.K_SHA256, 2, m, n, unit_bytes=L, flags=3, table=tab)


@pytest.mark.parametrize("layout_flag", [0x8, 0x10])      # -i (adjacent lanes) / -s (adjacent warps, the default)
@pytest.mark.parametrize("n", [1, 31, 32, 33, 127, 128, 129, 1000, 4099])
def test_sha256_tmr_layouts_give_identical_results(rt, oracle, layout_flag, n):
    m = msgs(oracle, n, 64, 21)
    both(rt, oracle, oracle.K_SHA256, 3, m, n, unit_bytes=64, flags=3 | layout_flag)
    both(rt, oracle, oracle.K_SHA256, 3, m, n, unit_bytes=64, flags=3 | layout_flag, plan_kw=dict(seed=n, p=0.25))


@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("M,N,K", [(64, 128, 16), (128, 256, 64), (192, 384, 160)])
def test_mm_tiled_kernel_exact_and_faults(rt, oracle, nc, M, N, K):
    """sizes that take the register-tiled kernel (64 x 128 x 16 tiles): bit-exact with the oracle, with and without faults"""
    A = oracle.fill_philox(M * K, 0, 4)
    B = oracle.fill_philox(K * N, 0, 44)
    both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3)
    both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3, plan_kw=dict(seed=K, p=0.1))
    tab = np.zeros(M * N, dtype=np.uint32)
    for u, (r, s, b) in enumerate([(0, 0, 0), (1, K - 1, 31), (2, K // 2, 7), (0, 3, 30), (1, 0, 16)]):
        tab[u * 97 % (M * N)] = oracle.fault_entry(r, s, b)
    both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3, table=tab)


def test_mm_full_size_properties(rt, oracle):
    """4096^3 exact integer TMR (the reference's own arithmetic at BASELINE config-4 size): voted output == unprotected output
    bit for bit under a fault plan; spot elements equal the oracle's dot products; XOR-fold check as mm_common_tmr.c:23-32."""
    import torch
    import coast_b200 as cb
    n = 4096
    A = torch.empty(n * n, dtype=torch.int32, device="cuda")
    B = torch.empty(n * n, dtype=torch.int32, device="cuda")
    rt.fill_philox(A, seed=4)
    rt.fill_philox(B, seed=44)
    o1 = torch.empty(n * n, dtype=torch.int32, device="cuda")
    o3 = torch.empty(n * n, dtype=torch.int32, device="cuda")
    rt.run(cb.K_MM_U32, 1, A, n * n, M=n, N=n, K=n, aux=B, out=o1)
    _, st = rt.run(cb.K_MM_U32, 3, A, n * n, M=n, N=n, K=n, aux=B, flags=3, out=o3, plan=cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=8, p=2 ** -12))
    assert torch.equal(o1, o3) and st.errors_corrected == st.injected > 3000
    hA = oracle.fill_philox(n * n, 0, 4)
    hB = oracle.fill_philox(n * n, 0, 44)
    C = o3.cpu().numpy().view(np.uint32).reshape(n, n)
    for (i, j) in [(0, 0), (1, 4095), (2047, 1234), (4095, 4095), (63, 64), (64, 127)]:
        ref = int(np.sum(hA[i * n:(i + 1) * n].astype(np.uint64) * hB[j::n].astype(np.uint64)) & np.uint64(0xFFFFFFFF)) & 0xFFFFFFFF
        exact = 0
        for k in range(n):
            exact = (exact + int(hA[i * n + k]) * int(hB[k * n + j])) & 0xFFFFFFFF
        assert int(C[i, j]) == exact
    assert int(np.bitwise_xor.reduce(C.ravel())) == int(np.bitwise_xor.reduce(o1.cpu().numpy().view(np.uint32)))


@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("M,N,K", [(128, 64, 128), (256, 192, 256), (384, 256, 640)])
def test_mm_tensor_core_limb_kernel_is_bit_exact(rt, oracle, nc, M, N, K, monkeypatch):
    """tile-aligned sizes take the tcgen05 kind::i8 u8-limb kernel (xmr_mm_tc.cuh): exact modulo 2^32 like the reference loops,
    with full-range u32 operands, with and without faults; the CUDA-core tiled kernel gives the same bits."""
    A = oracle.fill_philox(M * K, 0, 4)
    B = oracle.fill_philox(K * N, 0, 44)
    A[:7] = 0xFFFFFFFF
    B[:5] = 0xFFFFFFFF                                  # worst-case limbs
    monkeypatch.delenv("COAST_MM_PATH", raising=False)
    g_tc, _ = both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3)
    both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3, plan_kw=dict(seed=K + nc, p=0.05))
    tab = np.zeros(M * N, dtype=np.uint32)
    for u, (r, s, b) in enumerate([(0, 0, 0), (1, K - 1, 31), (2, K // 2, 7), (0, 3, 30), (1, 0, 16)]):
        tab[u * 89 % (M * N)] = oracle.fault_entry(r, s, b)
    both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3, table=tab)
    for variant in ("tc", "tct"):                       # A operand from shared memory / staged in TMEM (tcgen05.cp + TS-mode MMA)
        monkeypatch.setenv("COAST_MM_PATH", variant)
        g_v, _ = both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3, plan_kw=dict(seed=K, p=0.02))
    monkeypatch.setenv("COAST_MM_PATH", "tiled")
    if N % 128 == 0:
        g_tiled, _ = both(rt, oracle, oracle.K_MM_U32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3)
        assert g_tiled.tobytes() == g_tc.tobytes()


def test_aes_key_mutation_matches_the_reference(rt, oracle, golden):
    """aes_enc_dec() leaves the last round key in key[] after encrypt and the original key after decrypt
    (TI_aes_128.c:214-221,133-141); pinned by running the reference (tests/golden: key_after_enc/dec)."""
    import ctypes as C
    import coast_b200 as cb
    rec = np.frombuffer(H(golden["aes"]["records"]), dtype=np.uint8).reshape(568, 80)
    kenc = np.frombuffer(H(golden["aes"]["key_after_enc"]), dtype=np.uint8)
    kdec = np.frombuffer(H(golden["aes"]["key_after_dec"]), dtype=np.uint8)
    keys = dev(rt, np.ascontiguousarray(rec[:, 0:16]))
    enc, _ = rt.run(cb.K_AES128, 3, dev(rt, np.ascontiguousarray(rec[:, 64:80])), 568, aux=keys,
                    mode=cb.AES_KEY_PER_UNIT | cb.AES_KEY_WRITEBACK, flags=3)
    assert host(enc).tobytes() == np.ascontiguousarray(rec[:, 32:48]).tobytes() and host(keys).tobytes() == kenc.tobytes()
    keys2 = dev(rt, np.ascontiguousarray(rec[:, 16:32]))
    dec, _ = rt.run(cb.K_AES128, 2, enc, 568, aux=keys2, mode=cb.AES_KEY_PER_UNIT | cb.AES_KEY_WRITEBACK | cb.AES_DECRYPT)
    assert host(dec).tobytes() == np.ascontiguousarray(rec[:, 48:64]).tobytes() and host(keys2).tobytes() == kdec.tobytes()
    # and through the reference-facing entry point
    L = rt.L
    assert L.coast_set_opt_passes(b"-TMR") == 0
    r = rec[300].tobytes()
    state, key = C.create_string_buffer(r[64:80], 16), C.create_string_buffer(r[0:16], 16)
    L.coast_xmr_aes_enc_dec(state, key, 0)
    assert state.raw == r[32:48] and key.raw == kenc[16 * 300: 16 * 301].tobytes()


# ------------------------------------------------------------------------------------------ quicksort (SURVEY 8f-4)
@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("L,n", [(580, 64), (1, 5), (2, 33), (17, 100), (1024, 21)])
def test_quicksort_branch_votes_match_oracle(rt, oracle, nc, L, n):
    a = oracle.fill_philox(n * L, 0, 9 + L).view(np.int32)
    g, _ = both(rt, oracle, oracle.K_QSORT, nc, a, n, unit_bytes=4 * L, flags=3)
    assert (g.view(np.int32).reshape(n, L) == np.sort(a.reshape(n, L), axis=1)).all()
    both(rt, oracle, oracle.K_QSORT, nc, a, n, unit_bytes=4 * L, flags=3, plan_kw=dict(seed=L, threshold=0xFFFFFFFF))
    both(rt, oracle, oracle.K_QSORT, nc, a, n, unit_bytes=4 * L, flags=3 | 0x100, plan_kw=dict(seed=L + 1, p=0.5))


def test_quicksort_already_sorted_and_duplicates(rt, oracle):
    L, n = 580, 30
    a = np.sort(oracle.fill_philox(n * L, 0, 3).view(np.int32).reshape(n, L), axis=1)      # sorted input (the reference re-sorts sorted arrays)
    a[10:20] = a[10:20, ::-1]                                                               # reverse-sorted
    a[20:] = (a[20:] & 7)                                                                   # many duplicates
    a = np.ascontiguousarray(a).ravel()
    for nc in (2, 3):
        both(rt, oracle, oracle.K_QSORT, nc, a, n, unit_bytes=4 * L, flags=3, plan_kw=dict(seed=77, threshold=0xFFFFFFFF))


def test_dwc_default_handler_aborts_like_the_reference(built_lib):
    """-DWC mismatch with no user FAULT_DETECTED_DWC: the synthesised handler calls abort() (synchronization.cpp:1251-1266),
    here after kernel completion.  Run in a child process and expect SIGABRT."""
    import subprocess
    import sys
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import torch, coast_b200 as cb\n"
        "rt = cb.Runtime(0)\n"
        "d = torch.zeros(4096 * 16, dtype=torch.uint8, device='cuda')\n"
        "o = torch.empty_like(d)\n"
        "desc = rt.make_desc(cb.K_AES128, 2, d, o, 4096, key=bytes(16), plan=cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=1, p=0.5))\n"
        "rt.launch(desc)\n"
        "print('before sync', flush=True)\n"
        "rt.sync(abort_on_dwc=True)\n"
        "print('NOT REACHED', flush=True)\n" % __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__))))
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=180)
    assert res.returncode == -6, (res.returncode, res.stdout, res.stderr)          # SIGABRT
    assert "before sync" in res.stdout and "NOT REACHED" not in res.stdout and "FAULT_DETECTED_DWC" in res.stderr


def test_quicksort_reference_golden_vectors_on_device(rt, oracle, golden):
    """the benchmark's own 580-int input and the reference outputs of tests/golden (quicksort.c compiled in place)"""
    g = golden["qsort"]
    inp = np.array(g["seed0_input"], dtype=np.int32)
    for nc in (1, 2, 3):
        out, st = both(rt, oracle, oracle.K_QSORT, nc, inp, 1, unit_bytes=4 * len(inp), flags=1)
        assert hashlib.sha256(out.tobytes()).hexdigest() == g["seed0_sorted_sha256"]
        assert st["errors_corrected"] == 0 and st["dwc_detected"] == 0
    for rec in g["random"]:
        a = np.array(rec["input"], dtype=np.int32)
        out, _ = both(rt, oracle, oracle.K_QSORT, 3, a, 1, unit_bytes=4 * len(a))
        assert np.frombuffer(out.tobytes(), dtype=np.int32).tolist() == rec["sorted"]


def test_empty_message_through_the_reference_entry_point(rt):
    """sha256_hash(len = 0) (sha256_common_tmr.c:101-180 hashes one padded block): the host call has nothing to stage"""
    import ctypes as C
    L = rt.L
    assert L.coast_set_opt_passes(b"-TMR -countErrors") == 0
    digest = C.create_string_buffer(32)
    cd, bl, stt, msg = C.create_string_buffer(64), (C.c_uint32 * 2)(), (C.c_uint32 * 8)(), C.create_string_buffer(4)
    L.coast_xmr_sha256_hash(cd, bl, stt, msg, 0, digest)
    assert digest.raw == hashlib.sha256(b"").digest()
