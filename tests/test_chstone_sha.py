"""tests/chstone/sha of byuccl/coast behind the same ABI (SURVEY.md 8f-4): oracle pinned on the reference's golden
outData and on reference digests of Philox streams; the CUDA kernel against the oracle (bit-exact), through the C ABI."""
import hashlib
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def benchmark_indata():
    """indata[2][8192] of tests/chstone/sha, stored by tests/golden/make_golden.py"""
    return np.fromfile(os.path.join(ROOT, "tests", "golden", "chstone_sha_indata.bin"), dtype=np.uint8)


def _table(oracle, faults, nc, n):
    tab = np.zeros(n, dtype=np.uint32)
    for u, f in enumerate(faults):
        if f is not None and f[0] < nc:
            site, bit = oracle.chstone_site_of_input_bit(f[1], f[2])
            tab[u] = oracle.fault_entry(f[0], site, bit)
    return tab


# ------------------------------------------------------------------ CPU: the oracle is pinned
def test_oracle_matches_reference_digests_of_philox_streams(oracle, golden):
    for rec in golden["chsha"]["philox"]:
        data = oracle.fill_philox(rec["len"] // 4, 0, rec["seed"]).tobytes()
        assert oracle.chstone_sha(data) == rec["digest"], rec["len"]


def test_oracle_matches_the_benchmark_golden(oracle, golden):
    g = golden["chsha"]
    indata = benchmark_indata()
    assert len(indata) == g["kat_len"] and hashlib.sha256(indata.tobytes()).hexdigest() == g["kat_input_sha256"]
    assert oracle.chstone_sha(indata.tobytes()) == g["kat_digest"]                # sha_driver.c:45-46 outData
    assert g["kat_digest"] == [0x006a5a37, 0x93dc9485, 0x2c412112, 0x63f7ba43, 0xad73f922]


def test_oracle_xmr_runs_match_the_reference_under_input_flips(oracle, golden):
    g = golden["chsha"]
    n, ln = g["xmr_n"], g["xmr_len"]
    msgs = oracle.fill_philox(n * ln // 4, 0, g["xmr_seed"]).view(np.uint8)
    for nc in (3, 2):
        plan = oracle.make_plan(oracle.PLAN_TABLE, table=_table(oracle, g["xmr_faults"], nc, n))
        out, st = oracle.run(oracle.K_CHSTONE_SHA, nc, msgs, n, unit_bytes=ln, plan=plan,
                             flags=oracle.F_COUNT_ERRORS | oracle.F_COUNT_SYNCS)
        ref = g["xmr_runs"][str(nc)]
        assert [int(v) for v in out.view(np.uint32)] == ref["out"]
        for k in ("errors_corrected", "dwc_detected", "syncs", "injected", "first_fault_unit"):
            assert st[k] == ref["stats"][k], (nc, k)


def test_oracle_site_geometry_and_bad_lengths(oracle):
    assert oracle.fault_sites(oracle.K_CHSTONE_SHA, 16384) == 421 * 257
    assert oracle.out_bytes_per_unit(oracle.K_CHSTONE_SHA) == 20 and oracle.votes_per_unit(oracle.K_CHSTONE_SHA) == 5
    for bad in (0, 63, 100):
        with pytest.raises(ValueError):
            oracle.run(oracle.K_CHSTONE_SHA, 1, np.zeros(128, dtype=np.uint8), 1, unit_bytes=bad)
    # every site class changes the digest of the faulted replica, and TMR outvotes it
    data = oracle.fill_philox(32, 0, 9).view(np.uint8)
    clean = oracle.chstone_sha(data.tobytes())
    for site in (0, 15, 16, 20, 415, 416, 420, 421 + 3, 2 * 421 + 418):
        tab = np.array([oracle.fault_entry(1, site, 5)], dtype=np.uint32)
        out, st = oracle.run(oracle.K_CHSTONE_SHA, 3, data, 1, unit_bytes=128, flags=oracle.F_COUNT_ERRORS,
                             plan=oracle.make_plan(oracle.PLAN_TABLE, table=tab))
        assert [int(v) for v in out.view(np.uint32)] == clean and st["errors_corrected"] >= 1, site
        out, st = oracle.run(oracle.K_CHSTONE_SHA, 2, data, 1, unit_bytes=128,
                             plan=oracle.make_plan(oracle.PLAN_TABLE, table=tab))
        assert st["dwc_detected"] == 1, site


# ------------------------------------------------------------------ GPU: the kernel against the oracle
def _both(rt, oracle, nc, data, n, ln, plan_kw=None, flags=0):
    from test_gpu_parity import both
    kw = {}
    if plan_kw is not None:
        if "table" in plan_kw:
            kw["table"] = plan_kw["table"]
        else:
            kw["plan_kw"] = plan_kw
    _, st = both(rt, oracle, oracle.K_CHSTONE_SHA, nc, data, n, unit_bytes=ln, flags=flags, **kw)
    return st


def _run(rt, nc, data, n, ln, table=None, flags=0):
    import coast_b200 as cb
    from test_gpu_parity import dev, host
    plan = cb.FaultPlan(mode=cb.PLAN_TABLE, table=dev(rt, table)) if table is not None else None
    out, st = rt.run(cb.K_CHSTONE_SHA, nc, dev(rt, data), n, unit_bytes=ln, plan=plan, flags=flags)
    return [int(v) for v in host(out).view(np.uint32)], st.as_dict()


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("n,ln", [(1, 64), (7, 128), (333, 192), (1000, 1024), (64, 16384)])
def test_chsha_zero_fault(rt, oracle, nc, n, ln):
    data = oracle.fill_philox(n * ln // 4, 0, 100 + ln).view(np.uint8)
    _both(rt, oracle, nc, data, n, ln, flags=oracle.F_COUNT_ERRORS | oracle.F_COUNT_SYNCS)


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [2, 3])
def test_chsha_bernoulli_faults(rt, oracle, nc):
    n, ln = 4096, 320
    data = oracle.fill_philox(n * ln // 4, 0, 5).view(np.uint8)
    st = _both(rt, oracle, nc, data, n, ln, plan_kw={"seed": 31 + nc, "p": 0.05},
               flags=oracle.F_COUNT_ERRORS | oracle.F_COUNT_SYNCS)
    assert st["injected"] > 100
    assert (st["errors_corrected"] if nc == 3 else st["dwc_detected"]) > 0


@pytest.mark.gpu
def test_chsha_every_site_of_every_compression(rt, oracle):
    """TABLE plan: unit u gets site u of a 3-compression stream (2 data blocks + the final block), rotating replica and bit"""
    ln = 128
    ns = oracle.fault_sites(oracle.K_CHSTONE_SHA, ln)
    assert ns == 3 * 421
    data = np.tile(oracle.fill_philox(ln // 4, 0, 6).view(np.uint8), ns)
    for nc in (3, 2):
        tab = np.array([oracle.fault_entry(u % nc, u, (7 * u) % 32) for u in range(ns)], dtype=np.uint32)
        st = _both(rt, oracle, nc, data, ns, ln, plan_kw={"table": tab}, flags=oracle.F_COUNT_ERRORS)
        assert st["injected"] == ns


@pytest.mark.gpu
def test_chsha_reference_golden_vectors_on_device(rt, oracle, golden):
    import coast_b200 as cb
    g = golden["chsha"]
    for rec in g["philox"]:
        data = oracle.fill_philox(rec["len"] // 4, 0, rec["seed"]).view(np.uint8)
        got, _ = _run(rt, 3, data, 1, rec["len"])
        assert got == rec["digest"], rec["len"]
    n, ln = g["xmr_n"], g["xmr_len"]
    msgs = oracle.fill_philox(n * ln // 4, 0, g["xmr_seed"]).view(np.uint8)
    for nc in (3, 2):
        tab = _table(oracle, g["xmr_faults"], nc, n)
        got, st = _run(rt, nc, msgs, n, ln, table=tab, flags=cb.F_COUNT_ERRORS | cb.F_COUNT_SYNCS)
        ref = g["xmr_runs"][str(nc)]
        assert got == ref["out"]
        for k in ("errors_corrected", "dwc_detected", "syncs", "injected", "first_fault_unit"):
            assert st[k] == ref["stats"][k], (nc, k)


@pytest.mark.gpu
def test_chsha_benchmark_input_gives_outdata_through_the_entry_point(rt, oracle, golden, built_lib):
    """sha_stream() as the make flow binds it: indata[2][8192], in_i = {8192, 8192} -> sha_info_digest == outData"""
    import ctypes as C
    lib = C.CDLL(built_lib)
    lib.coast_set_opt_passes(b"-TMR -countErrors")
    indata = benchmark_indata()
    assert hashlib.sha256(indata.tobytes()).hexdigest() == golden["chsha"]["kat_input_sha256"]
    in_i = (C.c_int * 2)(8192, 8192)
    dig = (C.c_uint32 * 5)()
    lib.coast_xmr_chstone_sha_stream(indata.ctypes.data_as(C.c_void_p), in_i, 2, 8192, dig)
    assert list(dig) == golden["chsha"]["kat_digest"]


@pytest.mark.gpu
def test_chsha_rejects_ragged_streams(rt):
    import coast_b200 as cb
    from test_gpu_parity import dev
    with pytest.raises(cb.CoastError):
        rt.run(cb.K_CHSTONE_SHA, 3, dev(rt, np.zeros(100, dtype=np.uint8)), 1, unit_bytes=100)
