"""GPU (two B200s of one box): the multi-GPU fold of TMR_ERROR_CNT / __SYNC_COUNT / DWC / injected / first_fault_unit done BY THE
KERNELS over peer memory (coast_counters_export / _attach, include/coast_rt.h) instead of a collective: a second process on GPU 1
tallies into GPU 0's counter block, and GPU 0's coast_sync() reads what the oracle counts for the WHOLE unit range."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAT_KEYS = ("errors_corrected", "dwc_detected", "syncs", "injected", "first_fault_unit")


@pytest.mark.parametrize("nc", [2, 3])
def test_second_gpu_tallies_into_the_owners_counter_block(rt, oracle, tmp_path, nc):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs of one box")
    n, half, seed, threshold = 6000, 2500, 5, 2 ** 32 // 40
    m = oracle.fill_philox(n * 16, 0, 9).view(np.uint8).copy()
    oplan = oracle.make_plan(oracle.PLAN_BERNOULLI, seed=seed, threshold=threshold)
    o_out, o_st = oracle.run(oracle.K_SHA256, nc, m, n, flags=3, unit_bytes=64, plan=oplan, unit_base=0)
    o_hi_out, o_hi = oracle.run(oracle.K_SHA256, nc, m[half * 64:], n - half, flags=3, unit_bytes=64, plan=oplan, unit_base=half)
    assert o_st["injected"] > 20 and o_hi["injected"] > 5

    rt.sync()                                               # counters start from zero
    handle = rt.counters_export()
    fin, fout = str(tmp_path / "in.npy"), str(tmp_path / "out.npy")
    np.save(fin, m[half * 64:])
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "peer_counters_child.py"), "1", handle.hex(), fin, fout,
                        str(half), str(nc), str(seed), str(threshold)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    child = json.loads(r.stdout.strip().splitlines()[-1])
    assert child["attached"] == dict(errors_corrected=0, dwc_detected=0, syncs=0, injected=0, first_fault_unit=2 ** 64 - 1)
    assert child["same_out"] and all(child["detached"][k] == o_hi[k] for k in STAT_KEYS)     # detached: the local block again
    assert np.load(fout).tobytes() == o_out[half * 32:].tobytes()

    import coast_b200 as cb
    gplan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=seed, threshold=threshold)
    g_lo, st = rt.run(cb.K_SHA256, nc, torch.from_numpy(m[: half * 64]).cuda(), half, flags=3, unit_bytes=64, plan=gplan, unit_base=0)
    assert g_lo.cpu().numpy().tobytes() == o_out[: half * 32].tobytes()
    got = st.as_dict()
    for k in STAT_KEYS:                                     # GPU 0's own shard + what GPU 1's kernels added over the link
        assert got[k] == o_st[k], (k, got, o_st)
