"""tests/chstone/aes of byuccl/coast behind the same ABI (SURVEY.md 8f-4): the oracle restatement (oracle/coast_oracle.c
orc_chstone_aes) pinned on the reference's own encrypt()/decrypt() -- the benchmark's FIPS-197 vector, 40 random blocks both
directions, DWC/TMR runs with an input-copy flip -- and the CUDA kernel against the oracle (bit-exact, every fault site),
through the C ABI and through the unchanged benchmark built by the BOARD=b200 flow."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAT_KEYS = ("errors_corrected", "dwc_detected", "syncs", "injected", "first_fault_unit")


def i32(x):
    return np.asarray(x, dtype=np.int32)


# ------------------------------------------------------------------ CPU: the oracle is pinned
def test_oracle_matches_the_reference_vectors(oracle, golden):
    g = golden["chaes"]
    assert bytes(g["kat_cipher"]).hex() == "3925841d02dc09fbdc118597196a0b32"                # FIPS-197 Appendix B, aes_enc.c:77-80
    out, _ = oracle.run(oracle.K_CHSTONE_AES, 1, i32(g["kat_plain"]), 1, mode=2, aux=i32(g["kat_key"]))
    assert list(out.view(np.int32)) == g["kat_cipher"]
    out, _ = oracle.run(oracle.K_CHSTONE_AES, 1, i32(g["kat_cipher"]), 1, mode=3, aux=i32(g["kat_key"]))
    assert list(out.view(np.int32)) == g["kat_plain"]
    for rec in g["random"]:
        for mode, nm in ((2, "enc"), (3, "dec")):
            out, _ = oracle.run(oracle.K_CHSTONE_AES, 1, i32(rec["block"]), 1, mode=mode, aux=i32(rec["key"]))
            assert list(out.view(np.int32)) == rec[nm]
    # one shared key through desc.key == the same key per unit
    key = bytes(g["kat_key"])
    out, _ = oracle.run(oracle.K_CHSTONE_AES, 1, i32(g["kat_plain"]), 1, mode=0, key=key)
    assert list(out.view(np.int32)) == g["kat_cipher"]


def test_oracle_xmr_runs_match_the_reference_under_input_flips(oracle, golden):
    g = golden["chaes"]
    n = g["xmr_n"]
    for d in (0, 1):
        for nc in (3, 2):
            tab = np.zeros(n, dtype=np.uint32)
            for u, f in enumerate(g["xmr_faults"]):
                if f is not None and f[0] < nc:
                    tab[u] = oracle.fault_entry(f[0], f[1], f[2])            # sites 0..15 = statemt[i] as loaded
            out, st = oracle.run(oracle.K_CHSTONE_AES, nc, i32(g["xmr_blocks"]), n, mode=2 | d, aux=i32(g["xmr_keys"]),
                                 flags=3, plan=oracle.make_plan(oracle.PLAN_TABLE, table=tab))
            ref = g["xmr_runs"][f"{d}_{nc}"]
            assert list(out.view(np.int32)) == ref["out"]
            for k in STAT_KEYS:
                assert st[k] == ref["stats"][k], (d, nc, k)


def test_chstone_and_ti_formulations_agree_site_by_site(oracle):
    """the CHStone sites (after each round-key addition) are where the TI enumeration puts its flips, modulo the XOR-linear key add:
    same block, same key, same (site, bit) => same bytes out of both restatements"""
    rng = np.random.default_rng(5)
    n = 176
    blocks = rng.integers(0, 256, 16 * n, dtype=np.int64).astype(np.uint8)
    keys = rng.integers(0, 256, 16 * n, dtype=np.int64).astype(np.uint8)
    table = np.array([oracle.fault_entry(0, s, s % 8) for s in range(n)], dtype=np.uint32)
    for d in (0, 1):
        ti, _ = oracle.run(oracle.K_AES128, 1, blocks, n, mode=2 | d, aux=keys, plan=oracle.make_plan(oracle.PLAN_TABLE, table=table))
        ch, _ = oracle.run(oracle.K_CHSTONE_AES, 1, blocks.astype(np.int32), n, mode=2 | d, aux=keys.astype(np.int32),
                           plan=oracle.make_plan(oracle.PLAN_TABLE, table=table))
        assert ch.view(np.int32).astype(np.uint8).tobytes() == ti.tobytes(), d


def test_geometry(oracle):
    assert oracle.fault_sites(oracle.K_CHSTONE_AES) == 176 and oracle.out_bytes_per_unit(oracle.K_CHSTONE_AES) == 64
    assert oracle.votes_per_unit(oracle.K_CHSTONE_AES) == 16


# ------------------------------------------------------------------ GPU
def _both(rt, oracle, nc, blocks, keys, n, mode, **kw):
    import torch
    import coast_b200 as cb
    plan_kw, table = kw.get("plan_kw"), kw.get("table")
    oplan = gplan = None
    if table is not None:
        oplan = oracle.make_plan(oracle.PLAN_TABLE, table=table)
        gplan = cb.FaultPlan(mode=cb.PLAN_TABLE, table=torch.from_numpy(table.view(np.int32).copy()).cuda())
    elif plan_kw:
        oplan = oracle.make_plan(oracle.PLAN_BERNOULLI, **plan_kw)
        gplan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, **plan_kw)
    o_out, o_st = oracle.run(oracle.K_CHSTONE_AES, nc, blocks, n, mode=mode, aux=keys, flags=3, plan=oplan, unit_base=9)
    g_out, g_st = rt.run(cb.K_CHSTONE_AES, nc, torch.from_numpy(blocks.copy()).cuda(), n, mode=mode,
                         aux=torch.from_numpy(keys.copy()).cuda(), flags=3, plan=gplan, unit_base=9)
    assert g_out.cpu().numpy().tobytes() == o_out.tobytes(), (nc, mode)
    assert {k: g_st.as_dict()[k] for k in STAT_KEYS} == {k: o_st[k] for k in STAT_KEYS}
    return g_st.as_dict()


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [1, 2, 3])
@pytest.mark.parametrize("dec", [0, 1])
def test_chaes_matches_the_oracle(rt, oracle, nc, dec):
    rng = np.random.default_rng(11 + nc + 4 * dec)
    for n in (1, 10, 11, 333, 20000):
        blocks = rng.integers(0, 256, 16 * n, dtype=np.int64).astype(np.int32)
        keys = rng.integers(0, 256, 16 * n, dtype=np.int64).astype(np.int32)
        _both(rt, oracle, nc, blocks, keys, n, 2 | dec)
        st = _both(rt, oracle, nc, blocks, keys, n, 2 | dec, plan_kw=dict(seed=3, p=0.2))
        if n >= 333 and nc > 1:
            assert st["injected"] > 0 and (st["errors_corrected"] if nc == 3 else st["dwc_detected"]) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("dec", [0, 1])
def test_chaes_every_site_every_replica(rt, oracle, dec):
    rng = np.random.default_rng(2)
    n = 176 * 3
    blocks = rng.integers(0, 256, 16 * n, dtype=np.int64).astype(np.int32)
    keys = rng.integers(0, 256, 16 * n, dtype=np.int64).astype(np.int32)
    table = np.array([oracle.fault_entry(u % 3, u // 3, (u * 5) % 8) for u in range(n)], dtype=np.uint32)
    st = _both(rt, oracle, 3, blocks, keys, n, 2 | dec, table=table)
    assert st["injected"] == n and st["errors_corrected"] >= n          # a flipped byte disagrees in at least one of the 16 votes


@pytest.mark.gpu
def test_chaes_reference_vectors_on_device_and_shared_key(rt, oracle, golden):
    import torch
    import coast_b200 as cb
    g = golden["chaes"]
    recs = g["random"]
    blocks = i32([v for r in recs for v in r["block"]])
    keys = i32([v for r in recs for v in r["key"]])
    for mode, nm in ((2, "enc"), (3, "dec")):
        out, st = rt.run(cb.K_CHSTONE_AES, 3, torch.from_numpy(blocks).cuda(), len(recs), mode=mode, aux=torch.from_numpy(keys).cuda(), flags=3)
        assert list(out.cpu().numpy().view(np.int32)) == [v for r in recs for v in r[nm]] and st.errors_corrected == 0
    out, _ = rt.run(cb.K_CHSTONE_AES, 2, torch.from_numpy(i32(g["kat_plain"])).cuda(), 1, key=bytes(g["kat_key"]))
    assert list(out.cpu().numpy().view(np.int32)) == g["kat_cipher"]


@pytest.mark.gpu
def test_chaes_entry_point_and_host_call(rt, oracle, golden):
    import ctypes as C
    g = golden["chaes"]
    L = rt.L
    assert L.coast_set_opt_passes(b"-TMR -countErrors") == 0
    st = (C.c_int * 32)(*g["kat_plain"]); key = (C.c_int * 32)(*g["kat_key"])
    L.coast_xmr_chstone_aes.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.coast_xmr_chstone_aes.restype = None
    L.coast_xmr_chstone_aes(st, key, 128128, 0)
    assert list(st)[:16] == g["kat_cipher"] and list(key)[:16] == g["kat_key"]
    L.coast_xmr_chstone_aes(st, key, 128128, 1)
    assert list(st)[:16] == g["kat_plain"]


@pytest.mark.gpu
def test_unchanged_chstone_aes_benchmark_runs_on_the_gpu():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from build_reference_tests import run_env
    exe = os.path.join(ROOT, "oracle", "_ref", "b200", "chstone_aes", "aes.out")
    if not os.path.exists(exe):
        pytest.skip("binary was not built on the CPU box (needs the reference checkout)")
    for passes in ("-TMR", "-DWC", ""):
        res = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=run_env(COAST_OPT_PASSES_OVERRIDE=passes + " -verbose"))
        assert res.returncode == 0, res.stdout + res.stderr
        assert re.search(r"encrypted message \t3925841d02dc09fbdc118597196a0b32\ndecrypto message\t3243f6a8885a308d313198a2e0370734RESULT: PASS", res.stdout)
        assert ("xmr_chaes_enc_nc%d" % (3 if "TMR" in passes else 2 if "DWC" in passes else 1)) in res.stderr and "xmr_chaes_dec_" in res.stderr
