#!/usr/bin/env python3
"""bench.py -- measurement of the protected-region hot path on B200.

Headline workload (BASELINE.json configs[1]): SHA-256 under TMR, 2^20 x 64-byte messages per GPU, warp-shuffle
select voter, -countErrors -countSyncs.  Metric: MB/s of VOTED OUTPUT.  One "step" = one protected launch over the
whole batch.  The same JSON line carries the other BASELINE configs under "also" (each timed in the same process
with its own roofline / e2e / cpu_baseline):
    N = 1 : aes (configs[2]), gemm (configs[3]), crc16 (config-1 timing shape), crc16_cpu_1thread (configs[0]),
            sha256_2p30 (configs[4] on one GPU)
    N > 1 : sha256_2p30 strong-scaled over the ranks (configs[4]), gemm sharded by C row-blocks (configs[3])

  python bench.py [--gpus N --steps K --warmup W]          # this repo's CUDA path
  python bench.py --workload aes|gemm|crc16|sha256_2p30     # one workload as its own line
  python bench.py --impl reference ...                      # the reference's own C sources (oracle/_ref, else the
                                                            # oracle port) under CPU xMR, all host threads
Under torchrun (N>1) every rank works on its own shard (no data-path collective).  The ranks rendezvous ON THE GPU
(a 1-element all-reduce on the compute stream) right before the start event.  The only exchange of the path -- the fault
counters -- is done BY THE KERNELS: ranks 1..N-1 map rank 0's counter block over NVLink (coast_counters_attach) and every
kernel's closing tally is a handful of system-scope atomics into it, so the timed region holds no collective at all and
rank 0's coast_sync() reads the whole job's TMR_ERROR_CNT / __SYNC_COUNT.  (Without peer access the fallback is ONE NCCL
all-reduce of the 4 counters per timed region, inside the region; `collectives.counter_fold` says which ran.)
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "protected-kernel throughput (MB/s voted output), sha256 TMR"
SM_COUNT = 148

# one name per workload, shared by both arms so that `config` is identical in the two JSON lines the driver compares
WORKLOAD_NAMES = {
    "sha256": "sha256 TMR, 2^20 x 64-byte messages per GPU (BASELINE configs[1])",
    "sha256_2p30": "batched sha256 TMR, 2^30 x 64-byte messages sharded over the GPUs (BASELINE configs[4])",
    "aes": "aes-128 ECB encrypt DWC, 2^24 x 16-byte blocks, Bernoulli(2^-10) single-bit flips (BASELINE configs[2])",
    "crc16": "crc16 TMR, 2^20 x 64-byte messages (SURVEY.md 8d config 1 timing shape)",
    "gemm": "matmul TMR 4096x4096x4096 fp32 on tcgen05 kind::tf32, three TMEM accumulator replicas + voter (BASELINE configs[3])",
}
PROTECTION = {"sha256": "-TMR -countErrors -countSyncs", "sha256_2p30": "-TMR -countErrors -countSyncs",
              "aes": "-DWC + single-bit-flip injector", "crc16": "-TMR -countErrors -countSyncs",
              "gemm": "-TMR -countErrors -countSyncs"}
FULL_UNITS = {"sha256": 1 << 20, "sha256_2p30": 1 << 30, "aes": 1 << 24, "crc16": 1 << 20, "gemm": 4096 * 4096}
OUT_B = {"sha256": 32, "sha256_2p30": 32, "aes": 16, "crc16": 2, "gemm": 4}
DTYPE = {"sha256": "u32", "sha256_2p30": "u32", "aes": "u8", "crc16": "u16", "gemm": "f32(tf32 mma)"}
STRONG = {"sha256_2p30", "gemm"}


def metric_name(wl):
    return METRIC if wl.startswith("sha256") else f"protected-kernel throughput (MB/s voted output), {wl}"


def config_for(wl: str, n_gpus: int) -> dict:
    """The `config` object.  A pure function of (workload, GPU count): both arms print the same bytes."""
    return {"workload": WORKLOAD_NAMES[wl],
            "units": FULL_UNITS[wl], "units_are": "in total, sharded over the GPUs" if wl in STRONG else "per GPU",
            "protection": PROTECTION[wl], "voter": "select (r0==r1?r0:r2), one vote per stored element",
            "inputs": "Philox4x32-10 counter stream, identical bytes in both arms",
            "l2": "rotating in/out buffer sets larger than the 126 MB L2 (one set when a set alone is larger)",
            "parallelism": f"shard{n_gpus}" if n_gpus > 1 else "1gpu"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


def hbm_peak():
    pj = measured_peaks()
    if "hbm_gbs" in pj:
        return float(pj["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons via NVML while the timed regions run."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self.power = [], set(), None, []
        self.want_power = False
        self.period = 0.002
        self._stop = threading.Event()
        self._th = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                if self.want_power:                        # a slow NVML query that holds the driver lock: never inside a timed region
                    try:
                        self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)  # W (board power, NVML's ~100 ms window)
                    except Exception:
                        pass
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(self.period)

    def reset(self):
        self.samples, self.reasons, self.power = [], set(), []

    def start(self, period=0.002):
        """period: NVML polling interval.  2 ms inside the device-timed region (GPU-bound, launches are cheap); 25 ms inside
        the host-call region, where NVML queries contend with the copy/launch submissions on the driver lock and were
        measured to slow the pipeline by up to 1.8x."""
        self.period = period
        if self.nv:
            self._stop.clear()
            self._th = threading.Thread(target=self._run, daemon=True)
            self._th.start()

    def stop(self):
        if self._th:
            self._stop.set()
            self._th.join()
            self._th = None

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "power_w_max_single_launch_loop": round(max(self.power), 1) if self.power else None,
                "sampled_over": "the timed region and the back-to-back single-launch loop that follows it (same kernel, GPU busy)"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own C functions under the restated xMR wrapper (oracle/_ref), or the port
# ------------------------------------------------------------------------------------------------
class CpuArm:
    """One workload on the host cores.  `one()` runs one pass over n units; inputs are built once."""

    def __init__(self, wl: str, n_units: int, threads: int):
        import ctypes as C
        import numpy as np
        from oracle import pyoracle as po
        po.build()
        self.wl, self.threads = wl, threads
        self.ob = OUT_B[wl]
        self.n = n_units
        have_ref = po.ref_available()
        if wl.startswith("sha256"):
            msgs = po.fill_philox(n_units * 16, 0, 2).view(np.uint8)
            out = np.zeros(n_units * 32, dtype=np.uint8)
            if have_ref:
                lib = po.ref("sha256")
                lib.ref_sha256_xmr_mt.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int,
                                                  C.c_int, C.POINTER(po.RefStats)]
                self.kind = "reference"

                def one():
                    st = po.RefStats()
                    lib.ref_sha256_xmr_mt(msgs.ctypes.data, out.ctypes.data, n_units, 64, 3, 1, 1, threads, C.byref(st))
            else:
                self.kind = "port"

                def one():
                    po.run(po.K_SHA256, 3, msgs, n_units, unit_bytes=64, flags=3, threads=threads)
        elif wl == "crc16":
            inp = po.fill_philox(n_units * 16, 0, 2).view(np.uint8)
            out = np.zeros(n_units, dtype=np.uint16)
            if have_ref:                                     # the reference's own crc16() under the restated TMR wrapper
                lib = po.ref("crc16")
                lib.ref_crc16_xmr_mt.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int,
                                                 C.c_int, C.POINTER(po.RefStats)]
                self.kind = "reference"

                def one():
                    st = po.RefStats()
                    lib.ref_crc16_xmr_mt(inp.ctypes.data, out.ctypes.data, n_units, 64, 3, 1, 1, threads, C.byref(st))
            else:
                self.kind = "port"

                def one():
                    po.run(po.K_CRC16, 3, inp, n_units, unit_bytes=64, flags=3, threads=threads)
        elif wl == "aes":
            inp = po.fill_philox(n_units * 4, 0, 2).view(np.uint8)
            if have_ref:
                # the reference's own aes_enc_dec() under the restated DWC wrapper.  Its flips can only go into a replica's private
                # copy of the INPUT (mid-round sites need edited sources): Bernoulli(2^-10) per block, as in the GPU arm's plan.
                lib = po.ref("aes")
                lib.ref_aes_xmr_mt.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_int,
                                               C.c_int, C.c_void_p, C.c_int, C.POINTER(po.RefStats)]
                rng = np.random.default_rng(33)
                hit = rng.random(n_units) < 2.0 ** -10
                faults = np.zeros((n_units, 3), dtype=np.int32)           # ref_fault {replica, byte, bit}
                faults[:, 1] = -1
                k = int(hit.sum())
                faults[hit] = np.stack([rng.integers(0, 2, k), rng.integers(0, 16, k), rng.integers(0, 8, k)], axis=1)
                key = np.zeros(16, dtype=np.uint8)
                out = np.zeros(n_units * 16, dtype=np.uint8)
                self.kind = "reference"

                def one():
                    st = po.RefStats()
                    lib.ref_aes_xmr_mt(inp.ctypes.data, out.ctypes.data, n_units, key.ctypes.data, 0, 0, 2, 0, 0, faults.ctypes.data,
                                       threads, C.byref(st))
                    assert st.dwc_detected == st.injected == k      # detect-rate parity holds on the CPU arm too
            else:
                self.kind = "port"
                plan = po.make_plan(po.PLAN_BERNOULLI, seed=33, p=2.0 ** -10)

                def one():
                    po.run(po.K_AES128, 2, inp, n_units, flags=0, key=bytes(16), plan=plan, threads=threads)
        else:  # gemm: a row-block sample of the 4096^3 problem (n_units = rows * 4096); a shape the reference has no code for
            side = 4096
            rows = max(1, n_units // side)
            self.n = rows * side
            A = (po.fill_philox(rows * side, 0, 4).astype(np.float64) / 2 ** 31 - 1.0).astype(np.float32)
            B = (po.fill_philox(side * side, 0, 44).astype(np.float64) / 2 ** 31 - 1.0).astype(np.float32)
            self.kind = "port"

            def one():
                po.run(po.K_GEMM_TF32, 3, A, rows * side, flags=3, threads=threads, M=rows, N=side, K=side, aux=B)
        self.one = one

    def time_passes(self, passes: int, warm: int = 1):
        """seconds of each pass (after `warm` untimed ones): thread creation, page faults and cold caches stay out."""
        for _ in range(warm):
            self.one()
        ts = []
        for _ in range(passes):
            t0 = time.perf_counter()
            self.one()
            ts.append(time.perf_counter() - t0)
        return ts


def cpu_sample_units(wl: str, threads: int, budget_s: float, passes: int):
    """units per pass such that (passes + 1 warm) passes take about budget_s on this box (calibrated on a small pass)."""
    cal_n = {"gemm": 4096 * 2, "aes": 1 << 16}.get(wl, 1 << 14)
    arm = CpuArm(wl, cal_n, threads)
    t_cal = min(arm.time_passes(2, warm=1))
    rate = arm.n / max(t_cal, 1e-6)
    n = int(max(cal_n, min(FULL_UNITS[wl], rate * budget_s / (passes + 1))))
    return (n // 4096) * 4096 if wl == "gemm" else 1 << (n.bit_length() - 1)


def cpu_baseline_block(wl: str, budget_s: float, passes: int = 5, threads: int = 0):
    threads = threads or (os.cpu_count() or 1)
    n = cpu_sample_units(wl, threads, budget_s, passes)
    arm = CpuArm(wl, n, threads)
    ts = arm.time_passes(passes, warm=1)
    med = statistics.median(ts)
    return {"value": round(arm.n * arm.ob / med / 1e6, 3), "unit": "MB/s", "cores": threads, "kind": arm.kind,
            "sample": f"{arm.n} units per pass of the same Philox inputs, median of {passes} passes after 1 warm-up, {threads} pinned pthreads",
            "spread": round(max(ts) / min(ts), 3)}


def crc16_config1_block(budget_s: float = 3.0):
    """BASELINE configs[0]: tests/crc16 under TMR on the host CPU, ONE thread (plumbing, no GPU): the literal program's
    `result: 5ba3`, and the 2^20 x 64-byte timing shape of SURVEY.md 8d row 1 (a bounded sample of it)."""
    import ctypes as C
    import numpy as np
    from oracle import pyoracle as po
    po.build()
    res = None
    if po.ref_available():
        lib = po.ref("crc16")
        lib.ref_crc16_xmr.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_void_p,
                                      C.POINTER(po.RefStats)]
        msg = np.frombuffer(b"Automated TMR", dtype=np.uint8).copy()
        out = np.zeros(1, dtype=np.uint16)
        st = po.RefStats()
        lib.ref_crc16_xmr(msg.ctypes.data, out.ctypes.data, 1, 13, 3, 1, 1, None, C.byref(st))
        res = f"{int(out[0]):04x}"
        assert res == "5ba3", res
    blk = cpu_baseline_block("crc16", budget_s, passes=5, threads=1)
    blk.update({"metric": metric_name("crc16"), "result_of_the_literal_program": res,
                "config": {"workload": "tests/crc16 under TMR on the host CPU, 1 thread (BASELINE configs[0])", "gpu": "none"}})
    return blk


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path on this box's host cores, same metric/config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = args.threads or (os.cpu_count() or 1)
    wl = args.workload
    n = cpu_sample_units(wl, threads, args.ref_budget_s, args.steps + args.warmup)
    arm = CpuArm(wl, n, threads)
    ts = arm.time_passes(args.steps, warm=args.warmup)
    t = statistics.median(ts)
    val = arm.n * arm.ob / t / 1e6
    line = {
        "impl": "reference",
        "metric": metric_name(wl),
        "value": round(val, 3), "unit": "MB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t * 1e3, 3), "higher_is_better": True,
        "scaling": "strong" if wl in STRONG else "weak", "vs_baseline": None,
        "dtype": DTYPE[wl], "data": "synthetic",
        "config": config_for(wl, args.gpus),
        "cpu_baseline": {"value": round(val, 3), "unit": "MB/s", "cores": threads, "kind": arm.kind,
                         "sample": f"{arm.n} units per step (a bounded sample of the workload), median of {args.steps} steps, "
                                   f"{threads} pinned pthreads",
                         "spread": round(max(ts) / min(ts), 3)},
        "e2e": {"value": round(val, 3), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "notes": "reference C sources compiled in place (oracle/_ref) + restated xMR wrapper (sha256, crc16, aes; aes flips go into a "
                 "replica's input copy); oracle port for the fp32 matmul; the real opt -TMR binary needs LLVM 7 (absent). "
                 "value = units x output bytes / MEDIAN step time.",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def workload_table(cb):
    F = cb.F_COUNT_ERRORS | cb.F_COUNT_SYNCS
    return {
        "sha256": dict(kernel=cb.K_SHA256, nc=3, flags=F, unit_bytes=64, in_b=64, alg_b=96, plan=None,
                       kname="xmr_sha256_b64_seg_nc3_inj0", bound="hbm", sets=4, profile="r01_sha256_tmr_seg.json",
                       profile_units=1 << 20, traffic="r01_sha256_tmr_traffic.json"),
        "sha256_2p30": dict(kernel=cb.K_SHA256, nc=3, flags=F, unit_bytes=64, in_b=64, alg_b=96, plan=None,
                            kname="xmr_sha256_b64_seg_nc3_inj0", bound="hbm", sets=1, profile="r01_sha256_tmr_seg.json",
                            profile_units=1 << 20, traffic=None),
        "aes": dict(kernel=cb.K_AES128, nc=2, flags=0, unit_bytes=0, in_b=16, alg_b=32,
                    plan=dict(seed=33, p=2.0 ** -10), key=bytes(16),
                    kname="xmr_aes128_enc_nc2_inj1", bound="hbm", sets=2, profile="r02_aes_nc2_inj1.json", profile_units=1 << 24,
                    traffic="r02_aes_traffic.json"),
        "crc16": dict(kernel=cb.K_CRC16, nc=3, flags=F, unit_bytes=64, in_b=64, alg_b=66, plan=None,
                      kname="xmr_crc16_b64_nc3_inj0", bound="hbm", sets=4, profile="r01_crc16_nc3_v2.json", profile_units=1 << 20,
                      traffic="r01_crc16_traffic.json"),
        "gemm": dict(kernel=cb.K_GEMM_TF32, nc=3, flags=F, side=4096, plan=None,
                     kname="xmr_gemm_tf32_nc3_inj0", bound="tensor", sets=2, profile="r02_gemm_nc3.json", profile_units=4096 * 4096,
                     traffic="r02_gemm_traffic.json"),
    }


def static_profile(name):
    """ncu numbers that are properties of the CODE (instruction count per launch, pipe shares), read from the committed
    summary under profiles/ and labelled as static wherever they are used."""
    if not name:
        return None
    fallbacks = {"r02_aes_nc2_inj1.json": "r01_aes_nc2_inj.json", "r02_gemm_nc3.json": "r01_gemm_nc3_final.json"}
    for cand in (name, fallbacks.get(name, name)):
        p = os.path.join(ROOT, "profiles", cand)
        if os.path.exists(p):
            try:
                with open(p) as f:
                    d = json.load(f)
                d = d[0] if isinstance(d, list) else d
                d["_file"] = f"profiles/{cand}"
                return d
            except Exception:
                return None
    return None


class Ctx:
    pass


DUMP_UNITS = 1 << 16                     # --dump-outputs: output units kept per workload (a fixed sample of larger outputs)
DUMP_WORD = {"sha256": "<u4", "sha256_2p30": "<u4", "aes": "u1", "crc16": "<u2", "gemm": "<f4"}
DUMP_MAX_BYTES = 64 << 20


def output_sample(torch, out, n: int, unit_base: int, wl: str):
    """The voted output of one launch as its caller reads it, for --dump-outputs: at most DUMP_UNITS units, drawn with a
    fixed seed so that two runs with the same arguments sample the same units.  One row per unit, one column per output
    word (digest word, byte, crc or fp32 element), widened exactly to float64 (u32 words) or float32.  Returns
    (values, global unit indices as float64)."""
    import numpy as np
    k = min(n, DUMP_UNITS)
    idx = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False)) if k < n else np.arange(n)
    rows = out.view(torch.uint8)[: n * OUT_B[wl]].view(n, OUT_B[wl])[torch.from_numpy(idx).to(out.device)]
    vals = rows.cpu().numpy().view(DUMP_WORD[wl])
    return vals.astype(np.float64 if DUMP_WORD[wl] == "<u4" else np.float32), (unit_base + idx).astype(np.float64)


def write_dump(path: str, arrays: dict) -> None:
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs: {total} bytes exceed {DUMP_MAX_BYTES}"
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def measure(cx, wl: str, steps: int, warmup: int, *, cpu_budget_s: float = 0.0, e2e_cap_units: int = 1 << 24, dump=None):
    """One workload on this rank's GPU: device-timed region, single-launch loop, end-to-end host call.  Returns the
    JSON-line dict on rank 0 (None elsewhere).  Every rank must call it with the same arguments.  With a `dump` dict,
    rank 0 adds to it a sample of the output of the last timed step (`<wl>`, `<wl>_units`) and the counters its
    coast_sync() returned after the timed region (`<wl>_counters`)."""
    torch, cb, rt, dist = cx.torch, cx.cb, cx.rt, cx.dist
    world, rank, dev = cx.world, cx.rank, cx.dev
    from coast_b200.shard import shard_range
    W = workload_table(cb)[wl]
    is_gemm = W["kernel"] == cb.K_GEMM_TF32
    plan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, **W["plan"]) if W.get("plan") else None
    nsets = W["sets"]
    out_b = OUT_B[wl]
    flops_issued = 0.0

    if is_gemm:
        # strong scaling (SURVEY.md 8e): C row-blocks of side/world rows per GPU, A row-block local, B replicated
        side = W["side"]
        r0, r1 = shard_range(side // 128, rank, world)
        rows = (r1 - r0) * 128
        n = rows * side
        unit_base = r0 * 128 * side
        scaling = "strong"
        in_b = 0
        alg_bytes = (rows * side + side * side + rows * side) * 4
        flops_issued = 3 * 2.0 * rows * side * side
        ins, outs, auxs = [], [], []
        for i in range(nsets):
            A = torch.empty(max(rows, 1) * side, dtype=torch.float32, device=dev)
            B = torch.empty(side * side, dtype=torch.float32, device=dev)
            rt.fill_philox(A, seed=4, word_base=unit_base + i * 0x20000000)
            rt.fill_philox(B, seed=44, word_base=i * 0x20000000)
            # Philox words -> uniform(-1,1) fp32 (SURVEY.md 8d config 4)
            A = (A.view(torch.int32).to(torch.float64) / 2 ** 31).to(torch.float32).contiguous()
            B = (B.view(torch.int32).to(torch.float64) / 2 ** 31).to(torch.float32).contiguous()
            ins.append(A); auxs.append(B); outs.append(torch.empty(max(n, 1), dtype=torch.float32, device=dev))
        descs = [rt.make_desc(W["kernel"], W["nc"], ins[i], outs[i], n, flags=W["flags"], M=rows, N=side, K=side, d_aux=auxs[i],
                              unit_base=unit_base, plan=plan) for i in range(nsets)] if n else []
        total_out_bytes = side * side * 4
    else:
        if wl in STRONG:                                     # config 5: a fixed 2^30-message batch, contiguous shards
            lo, hi = shard_range(FULL_UNITS[wl], rank, world)
            n, unit_base, scaling = hi - lo, lo, "strong"
            if n * 96 > 150 * (1 << 30):
                raise SystemExit(f"{wl}: {n} messages per GPU do not fit 180 GB; use more GPUs")
        else:
            n = FULL_UNITS[wl]                               # weak scaling: the same shard size on every GPU
            unit_base = rank * n
            scaling = "weak"
        in_b = W["in_b"]
        alg_bytes = n * W["alg_b"]
        ins = [torch.empty(n * in_b, dtype=torch.uint8, device=dev) for _ in range(nsets)]
        outs = [torch.empty(n * out_b, dtype=torch.uint8, device=dev) for _ in range(nsets)]
        for i, t in enumerate(ins):
            rt.fill_philox(t, seed=2, word_base=(unit_base * in_b // 4) + i * 0x10000000)
        descs = [rt.make_desc(W["kernel"], W["nc"], ins[i], outs[i], n, flags=W["flags"], unit_bytes=W["unit_bytes"], key=W.get("key"),
                              unit_base=unit_base, plan=plan) for i in range(nsets)]
        total_out_bytes = (FULL_UNITS[wl] if wl in STRONG else world * n) * out_b
    d_stats = torch.zeros(5, dtype=torch.int64, device=dev)
    go = torch.zeros(1, dtype=torch.int32, device=dev)
    launches = 0

    def step(i):
        nonlocal launches
        if descs:
            rt.launch(descs[i % nsets])                    # ONE kernel: replicas + voter + counters (+ injector)
            launches += 1

    def exchange_counters():
        # the only exchange of the path: 32 bytes of counters over NVLink, where the program reads them (coast_sync)
        rt.stats_snapshot(d_stats)                         # D2D copy of the device counters on the compute stream
        dist.all_reduce(d_stats[:4])                       # the compute stream waits for it

    def fence():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = cx.sampler
    sampler.reset()
    peer_fold = dist is not None and cx.peer_handle is not None
    if peer_fold:
        fence()
        if rank != 0:
            rt.counters_attach(cx.peer_handle)             # from here on this rank's kernels tally into rank 0's block over NVLink
    rt.sync()                                              # (rank 0 resets the shared block; an attached rank's sync only drains its stream)
    if peer_fold:
        fence()                                            # nobody launches before the owner's reset has landed
    for i in range(warmup):
        step(i)
    if dist is not None and not peer_fold:
        exchange_counters()
    fence()
    launches = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    n_sm = rt.sm_count()
    probe0 = torch.zeros(2 * n_sm, dtype=torch.int64, device=dev)
    probe1 = torch.zeros(2 * n_sm, dtype=torch.int64, device=dev)
    if dist is not None:
        dist.all_reduce(go)                                # rendezvous ON THE GPU: every rank's clock starts when the last rank arrives
    use_probe = os.environ.get("COAST_BENCH_CLOCK_PROBE", "1") != "0"
    if use_probe:
        rt.clock_probe(probe0)                             # {clock64, globaltimer} per SM, just outside the timed region
    e0.record()
    for i in range(steps):
        step(i)
    if dist is not None and not peer_fold:
        exchange_counters()                                # fallback: inside the timed region, once -- where coast_sync() would fold them
    e1.record()
    if use_probe:
        rt.clock_probe(probe1)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    timed_launches = launches
    if dump is not None and rank == 0 and descs:
        dump[wl], dump[wl + "_units"] = output_sample(torch, outs[(steps - 1) % nsets], n, unit_base, wl)
    # the SM clock the region REALLY ran at: cycles / nanoseconds between the two probes, per SM that answered both, median
    p0, p1 = probe0.view(-1, 2).cpu(), probe1.view(-1, 2).cpu()
    both = (p0[:, 1] > 0) & (p1[:, 1] > p0[:, 1])
    sm_clock_mhz = None
    if int(both.sum()) >= 8:
        ghz = (p1[both, 0] - p0[both, 0]).double() / (p1[both, 1] - p0[both, 1]).double()
        sm_clock_mhz = round(float(ghz.median()) * 1e3, 1)
    if peer_fold:
        dist.barrier()                                     # every rank's kernels (and their remote atomics) have retired
    st = rt.sync()                                         # rank 0: the counters of the whole job (peer fold) / of this rank
    if peer_fold:
        units_all = torch.tensor([n], dtype=torch.int64, device=dev)
        dist.all_reduce(units_all)                         # units of all ranks, for the check below (outside the timed region)
        n_counted = int(units_all[0]) if rank == 0 else 0
        fence()
        if rank != 0:
            rt.counters_detach()                           # the single-launch loop and the host calls below tally locally again
    else:
        n_counted = n
    if dump is not None and rank == 0:
        import numpy as np
        dump[wl + "_counters"] = np.array(list(st.as_dict().values()), dtype=np.float64)
    if wl.startswith("sha256"):
        assert st.errors_corrected == 0 and st.syncs == 32 * n_counted * (steps + warmup), (st, n_counted)
    if wl == "aes" and (rank == 0 or not peer_fold):
        assert st.dwc_detected == st.injected > 0, st      # detect-rate parity: every state flip is detected

    # kernel-only duration (cross-check of the roofline's average) and enough GPU-busy time for >= 20 clock samples:
    # single launches bracketed by events, for at least 20 launches and 60 ms
    kms = []
    sampler.want_power = True                              # board power: sampled in this loop only (same kernel, GPU busy)
    t_loop = time.perf_counter()
    i = 0
    while descs and (i < 20 or time.perf_counter() - t_loop < 0.06) and i < 2000:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rt.launch(descs[i % nsets])
        b.record()
        b.synchronize()
        kms.append(a.elapsed_time(b))
        i += 1
    sampler.stop()
    sampler.want_power = False
    clocks = sampler.summary()
    clocks["sm_mhz_in_timed_region"] = sm_clock_mhz
    clocks["sm_mhz_in_timed_region_how"] = ("clock64() / %globaltimer deltas between two probe kernels bracketing the timed region, median over SMs; "
                                            "NVML (sm_mhz) reports the requested clock, this is the delivered one")
    rt.sync()
    k_ms = statistics.median(kms) if kms else 0.0

    coll_in_value_ms = 0.0
    if dist is not None and not peer_fold:                 # what the one counter exchange costs, measured on its own
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.all_reduce(go)
        a.record()
        for _ in range(5):
            exchange_counters()
        b.record(); b.synchronize()
        coll_in_value_ms = a.elapsed_time(b) / 5

    # end to end through the reference-facing host call: pinned HOST buffers in, voted output in HOST memory out, every step
    e2e_steps = max(3, min(steps, 20))
    if is_gemm:
        h_in = ins[0].cpu().pin_memory(); h_aux = auxs[0].cpu().pin_memory()
        h_out = torch.empty(max(n, 1), dtype=torch.float32).pin_memory()
        call = lambda: rt.run_host(W["kernel"], W["nc"], h_in, h_out, n, flags=W["flags"], M=rows, N=side, K=side, h_aux=h_aux,
                                   unit_base=unit_base, plan=plan)
        h2d, d2h = (rows * side + side * side) * 4, rows * side * 4 + 40
    else:
        ne = min(n, e2e_cap_units)                           # e2e batch: at most 2^24 units of the shard through host memory
        h_in = torch.empty(ne * in_b, dtype=torch.uint8).pin_memory()
        h_in.copy_(ins[0][: ne * in_b].cpu())
        h_out = torch.empty(ne * out_b, dtype=torch.uint8).pin_memory()
        call = lambda: rt.run_host(W["kernel"], W["nc"], h_in, h_out, ne, unit_bytes=W["unit_bytes"], flags=W["flags"],
                                   key=W.get("key"), unit_base=unit_base, plan=plan)
        h2d, d2h = ne * in_b, ne * out_b + 40
    for _ in range(3):
        call()
    fence()
    e2e_ts = []
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        t1 = time.perf_counter()
        call()
        e2e_ts.append(time.perf_counter() - t1)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    host_path = rt.last_host_path
    assert torch.equal(h_out.view(torch.uint8), outs[0].view(torch.uint8)[: h_out.numel() * h_out.element_size()].cpu())
    e2e_units = (h_out.numel() * h_out.element_size()) // out_b      # units per e2e call on this rank

    # context for the e2e number: what a bare pinned copy of the same buffers achieves on this box
    def copy_gbs(dst, src, reps=5):
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(reps):
            dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        return src.numel() * src.element_size() * reps / (time.perf_counter() - t) / 1e9
    pcie_h2d = copy_gbs(ins[1 % nsets].view(torch.uint8)[: h_in.numel() * h_in.element_size()], h_in.view(torch.uint8))
    pcie_d2h = copy_gbs(h_out.view(torch.uint8), outs[0].view(torch.uint8)[: h_out.numel() * h_out.element_size()])

    # SURVEY.md 8e "measured separately": the OPTIONAL data-path collectives a caller may add around the sharded launch --
    # all-gather of the voted outputs; for the matmul also the one distribution step (B from rank 0).  Never part of
    # `value`.  Device-timed, max over ranks.
    coll_ms = [0.0, 0.0]
    coll_note = None
    if dist is not None and world > 1:
        def time_coll(fn, reps=3):
            fn(); torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dist.all_reduce(go); a.record()
            for _ in range(reps):
                fn()
            b.record(); b.synchronize()
            return a.elapsed_time(b) / reps
        try:
            mine = outs[0].view(torch.uint8)
            per = torch.tensor([mine.numel()], dtype=torch.int64, device=dev)
            lo_hi = torch.stack([per, -per]).flatten()
            dist.all_reduce(lo_hi, op=dist.ReduceOp.MIN)
            equal = int(lo_hi[0]) == -int(lo_hi[1])                       # all_gather_into_tensor needs equal shards
            if equal and world * mine.numel() <= (2 << 30):
                gathered = torch.empty(world * mine.numel(), dtype=torch.uint8, device=dev)
                coll_ms[0] = time_coll(lambda: dist.all_gather_into_tensor(gathered, mine))
                assert torch.equal(gathered[rank * mine.numel():(rank + 1) * mine.numel()], mine)
                del gathered
            else:
                coll_note = "all-gather skipped: unequal shards or more than 2 GiB of outputs"
            if is_gemm:
                Bt = auxs[0]
                coll_ms[1] = time_coll(lambda: dist.broadcast(Bt, src=0))
        except Exception as exc:                                          # optional measurement: never lose the bench line
            coll_note = f"collective timing failed: {exc!r}"[:200]

    t = torch.tensor([ms, e2e_s, coll_ms[0], coll_ms[1], coll_in_value_ms, statistics.median(e2e_ts)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)           # max over ranks
    ms, e2e_s, coll_ms, coll_in_value_ms, e2e_med = float(t[0]), float(t[1]), [float(t[2]), float(t[3])], float(t[4]), float(t[5])
    del ins, outs, descs, h_in, h_out
    if is_gemm:
        del auxs, h_aux
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    ms_per_step = ms / steps
    value = total_out_bytes / (ms_per_step * 1e-3) / 1e6
    # the dominant kernel's average launch duration over the TIMED REGION (one launch per step, back to back on the
    # launching stream, CUDA events); the per-launch event pairs measured after it (k_ms) are kept as a cross-check
    k_reg = ms / max(1, timed_launches)
    prof = static_profile(W.get("profile"))
    sm_hz = (clocks.get("sm_mhz_in_timed_region") or clocks.get("sm_mhz") or 1965.0) * 1e6   # the delivered clock when the probes answered
    sm_hz_how = "SM clock delivered in the timed region (clock64/globaltimer probes)" if clocks.get("sm_mhz_in_timed_region") else "NVML-sampled SM clock"
    if W["bound"] == "hbm":
        peak, peak_src = hbm_peak()
        achieved, unit = alg_bytes / (k_reg * 1e-3) / 1e9, "GB/s"
        rl_extra = {"algorithmic_bytes_per_launch": alg_bytes,
                    "note": "integer-issue / shared-memory bound, not HBM bound (DESIGN.md section 5): alu_frac and issue_frac say how "
                            "close the kernel is to the SM's integer ceiling"}
    else:
        pj = measured_peaks()
        peak = float(pj.get("bf16_tflops", 1590.0)) / 2.0
        peak_src = "measured bf16 cuBLAS burst / 2 (TF32 runs at half the bf16 rate)" if pj else "fallback 1590/2"
        achieved, unit = flops_issued / (k_reg * 1e-3) / 1e12, "TFLOP/s"
        hw = 4096.0 * SM_COUNT * sm_hz / 1e12                # tcgen05 kind::tf32: 4096 dense FLOP / clk / SM
        rl_extra = {"issued_flops_per_launch": flops_issued, "useful_flops_per_launch": flops_issued / 3,
                    "frac_of_clock_scaled_hw_rate": round(achieved / hw, 5),
                    "clock_scaled_hw_rate": {"value": round(hw, 1), "unit": "TFLOP/s", "how": "4096 FLOP/clk/SM x 148 SMs x " + sm_hz_how},
                    "note": "issued = 3 replicas x 2MNK; useful = one replica"}
    if prof and prof.get("kernel") == W["kname"] and "warp_insts" in prof:
        # instructions per launch are a property of the CODE (static, from the committed ncu summary, scaled to this launch's
        # unit count); the time is live
        wi = prof["warp_insts"] * (n / float(W["profile_units"]))
        rl_extra["issue_frac"] = round(wi / (k_reg * 1e-3) / (SM_COUNT * 4 * sm_hz), 4)
        rl_extra["issue_frac_how"] = (f"warp instructions per launch ({prof['_file']}, static) / live kernel time / "
                                      "(148 SMs x 4 schedulers x 1 warp instruction per clock x " + sm_hz_how + ")")
        if W["bound"] == "hbm" and "pipe_alu_pct" in prof:
            rl_extra["alu_frac"] = round(prof["pipe_alu_pct"] / 100.0, 4)
            rl_extra["alu_frac_source"] = f"{prof['_file']} (static): ncu sm__inst_executed_pipe_alu, pct of peak sustained active"
    traffic, traffic_src = None, None
    if W.get("traffic"):
        tp = os.path.join(ROOT, "profiles", W["traffic"])
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            if tj.get("kernel", W["kname"]) == W["kname"]:
                traffic = tj.get("dram_bytes_per_launch")
                traffic_src = f"profiles/{W['traffic']} (static: one ncu --set full capture of this kernel at this size, not measured in this run)"
    bound_s = max(h2d / (pcie_h2d * 1e9), d2h / (pcie_d2h * 1e9))
    line = {
        "metric": metric_name(wl),
        "value": round(value, 1), "unit": "MB/s", "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": round(ms_per_step, 5), "higher_is_better": True, "scaling": scaling,
        "vs_baseline": None, "dtype": DTYPE[wl], "data": "synthetic",
        "config": config_for(wl, world),
        "roofline": dict({"bound": W["bound"], "achieved": round(achieved, 2), "peak": peak, "unit": unit,
                          "frac": round(achieved / peak, 5), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                          "kernel": W["kname"], "kernel_ms": round(k_reg, 5),
                          "kernel_ms_source": "timed region / launches (CUDA events on the launching stream)",
                          "kernel_ms_single_launch_events": round(k_ms, 5)}, **rl_extra),
        "e2e": {"value": round(world * e2e_units * out_b / e2e_s / 1e6, 1), "unit": "MB/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": round(e2e_s * 1e3, 4), "ms_per_step_median": round(e2e_med * 1e3, 4),
                "units_per_step_per_gpu": e2e_units, "path": host_path,
                "timer": "host clock around the blocking C-ABI call coast_run_host (pinned host buffers in and out)",
                "pcie_pinned_copy_gbs": {"h2d": round(pcie_h2d, 1), "d2h": round(pcie_d2h, 1)},
                "bound_ms": round(bound_s * 1e3, 4), "frac_of_bound": round(bound_s / e2e_s, 4),
                "bound_how": "max(h2d_bytes / bare pinned H2D copy rate, d2h_bytes / bare pinned D2H copy rate) on this box (full duplex)"
                             + ("; the zero-copy path reads the pinned input from the SMs, not through a copy engine, so it can beat this figure"
                                if host_path == "zerocopy" else ""),
                "numa_node": rt.numa_node},
        "gpu_launches": timed_launches,
        "clocks": clocks,
        "stats_last_sync": st.as_dict(),
    }
    if world > 1:
        line["collectives"] = {"counter_fold": "nvlink-peer-atomics" if peer_fold else "nccl-allreduce",
                               "in_value": ("GPU-side rendezvous before the start event; NO collective in the timed region: ranks 1..N-1 map rank 0's "
                                            "counter block over NVLink (coast_counters_attach) and every kernel's closing tally is a few system-scope "
                                            "atomics into it; stats_last_sync is the whole job's fold read by rank 0's coast_sync()") if peer_fold else
                                           ("GPU-side rendezvous before the start event + ONE all-reduce of the 4 counters per timed region "
                                            "(where coast_sync() folds them); no per-step collective"),
                               "in_value_ms": round(coll_in_value_ms, 4), "in_value_ms_per_step": round(coll_in_value_ms / steps, 5),
                               "allgather_outputs_ms": round(coll_ms[0], 4) if coll_ms[0] else None,
                               "allgather_bytes": world * total_out_bytes // world if coll_ms[0] else None,
                               "broadcast_B_ms": round(coll_ms[1], 4) if coll_ms[1] else None,
                               "note": coll_note or "all-gather / broadcast measured separately, not part of value (SURVEY.md 8e)"}
    if world == 1 and cpu_budget_s > 0:
        line["cpu_baseline"] = cpu_baseline_block("sha256" if wl.startswith("sha256") else wl, cpu_budget_s)
    return line


ALSO_STEPS = {"aes": 20, "gemm": 40, "crc16": 200, "sha256_2p30": 3}


def run_ours(args):
    import torch
    import coast_b200 as cb

    cx = Ctx()
    cx.torch, cx.cb = torch, cb
    cx.world = int(os.environ.get("WORLD_SIZE", "1"))
    cx.rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cx.dist = None
    if args.host_path:
        os.environ["COAST_HOST_PATH"] = args.host_path
    cx.rt = cb.Runtime(local)                              # coast_init first: it places the process on the GPU's NUMA node
    if cx.world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        cx.dist = dist
    cx.dev = f"cuda:{local}"
    cx.sampler = ClockSampler(local)
    cx.peer_handle = None
    if cx.dist is not None and os.environ.get("COAST_BENCH_COUNTER_FOLD", "peer") == "peer":
        # rank 0 exports its counter block (a 64-byte CUDA IPC handle), everyone else maps it over NVLink -- or all ranks fall back
        from coast_b200.shard import negotiate_peer_counter_block

        def probe(handle):
            cx.rt.counters_attach(handle)
            cx.rt.counters_detach()
        cx.peer_handle = negotiate_peer_counter_block(cx.dist, cx.rank, torch, cx.dev, cx.rt.counters_export, probe,
                                                      log=lambda m: print("bench: " + m, file=sys.stderr))

    main_cpu = 0.0 if args.no_cpu_baseline else 10.0
    dump = {} if args.dump_outputs else None
    line = measure(cx, args.workload, args.steps, args.warmup, cpu_budget_s=main_cpu, dump=dump)
    if args.workload == "sha256" and not args.no_also:
        also = {}
        wls = ["aes", "gemm", "crc16", "sha256_2p30"] if cx.world == 1 else ["sha256_2p30", "gemm"]
        for wl in wls:
            t0 = time.perf_counter()
            try:
                sub = measure(cx, wl, ALSO_STEPS[wl], 3, cpu_budget_s=0.0 if args.no_cpu_baseline else 3.0, dump=dump)
            except Exception as exc:                       # an extra workload must never cost the headline line
                sub = {"error": repr(exc)[:300]}
                if cx.dist is not None:
                    raise
            if sub is not None:
                sub["wall_s"] = round(time.perf_counter() - t0, 2)
                also[wl] = sub
        if cx.rank == 0 and cx.world == 1 and not args.no_cpu_baseline:
            try:
                also["crc16_cpu_1thread"] = crc16_config1_block()
            except Exception as exc:
                also["crc16_cpu_1thread"] = {"error": repr(exc)[:300]}
        if line is not None:
            line["also"] = also
    if cx.rank == 0:
        if dump is not None:
            write_dump(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if cx.dist is not None:
        cx.dist.barrier()
        cx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="headline workload only (skip the other BASELINE configs)")
    ap.add_argument("--host-path", choices=["staged", "hybrid", "zerocopy", "one-shot"], default=None, help="force the host-call path of the e2e measurement")
    ap.add_argument("--ref-budget-s", type=float, default=90.0, help="--impl reference: CPU seconds the whole run may take")
    ap.add_argument("--threads", type=int, default=0, help="--impl reference: host threads (default: all; config 1 is 1 thread)")
    ap.add_argument("--workload", choices=["sha256", "sha256_2p30", "aes", "crc16", "gemm"], default="sha256",
                    help="default sha256 = BASELINE configs[1], the headline line (with the other configs under `also`)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of each timed workload's last-step output, and its counters, as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "ours":
            ap.error("--dump-outputs applies to the GPU arm (--impl ours)")
        os.makedirs(args.dump_outputs, exist_ok=True)
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
