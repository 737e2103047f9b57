"""GPU (B200): the tcgen05 TF32 GEMM with NC accumulator replicas in TMEM + voting epilogue (BASELINE config 4).

Floating point on tensor cores: kind::tf32 reads the top 19 bits of each fp32 operand and accumulates in fp32 in an
unspecified order, so CPU parity is a TOLERANCE (|err| <= 2e-6*K absolute for operands in (-1,1); stated here), while
everything the protection layer promises is exact: the NC replicas are bit-identical, the voted output equals the
unprotected kernel's output bit for bit with and without injected faults, and the counters follow the fault plan."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def tf32(x):
    return (x.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def operands(oracle, M, N, K, seed=4):
    # uniform(-1,1) from Philox words (SURVEY.md 8d config 4)
    a = oracle.fill_philox(M * K, 0, seed).astype(np.float64) / 2 ** 31 - 1.0
    b = oracle.fill_philox(K * N, 0, seed + 40).astype(np.float64) / 2 ** 31 - 1.0
    return a.astype(np.float32).reshape(M, K), b.astype(np.float32).reshape(K, N)


def run(rt, nc, A, B, flags=3, plan=None):
    import torch
    import coast_b200 as cb
    M, K = A.shape
    N = B.shape[1]
    dA, dB = torch.from_numpy(A).cuda(), torch.from_numpy(B).cuda()
    out = torch.empty(M * N, dtype=torch.float32, device="cuda")
    _, st = rt.run(cb.K_GEMM_TF32, nc, dA, M * N, M=M, N=N, K=K, aux=dB, flags=flags, plan=plan, out=out)
    return out.cpu().numpy().reshape(M, N), st


@pytest.mark.parametrize("M,N,K", [(128, 128, 32), (128, 128, 64), (256, 128, 96), (128, 384, 256), (384, 256, 512), (512, 512, 1024)])
def test_gemm_tf32_matches_truncated_fp64_reference(rt, oracle, M, N, K):
    A, B = operands(oracle, M, N, K)
    ref = tf32(A).astype(np.float64) @ tf32(B).astype(np.float64)
    outs = {}
    for nc in (1, 2, 3):
        C, st = run(rt, nc, A, B)
        assert np.abs(C - ref).max() <= 2e-6 * K, (nc, np.abs(C - ref).max())
        assert st.errors_corrected == 0 and st.dwc_detected == 0      # replicas are bit-identical
        if nc == 3:
            assert st.syncs == M * N                                   # one fp32 vote per element
        outs[nc] = C
    assert outs[1].tobytes() == outs[2].tobytes() == outs[3].tobytes()
    # the element oracle (oracle/coast_oracle.c orc_gemm_tf32_elem) agrees with the same tolerance
    o, _ = oracle.run(oracle.K_GEMM_TF32, 1, A, M * N, M=M, N=N, K=K, aux=B)
    assert np.abs(o.view(np.float32).reshape(M, N) - outs[3]).max() <= 2e-6 * K


def check_faults_against_clean(rt, oracle, A, B, clean, seed, p):
    """DWC and TMR under a Bernoulli fault plan: TMR votes every fault out (the clean bits); DWC stores replica 0, so its output
    differs from the clean one in exactly the bits the oracle flips in replica 0; counters equal the oracle's"""
    import coast_b200 as cb
    M, K = A.shape
    N = B.shape[1]
    plan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=seed, p=p)
    got, want = {}, {}
    for nc in (2, 3):
        got[nc], st = run(rt, nc, A, B, plan=plan)
        want[nc], so = oracle.run(oracle.K_GEMM_TF32, nc, A, M * N, M=M, N=N, K=K, aux=B, flags=3,
                                  plan=oracle.make_plan(oracle.PLAN_BERNOULLI, seed=seed, p=p))
        assert st.as_dict() == so and st.injected > 0, (nc, st.as_dict(), so)
    assert got[3].tobytes() == clean.tobytes()
    flipped = want[2].view(np.uint32) ^ want[3].view(np.uint32)       # the oracle's TMR output is its clean output
    assert ((got[2].view(np.uint32) ^ clean.view(np.uint32)).ravel() == flipped.ravel()).all() and flipped.any()


@pytest.mark.parametrize("M,N,K", [(2432, 2048, 64), (2560, 2048, 96)])
def test_gemm_unprotected_tail_split_is_bit_identical(rt, oracle, M, N, K):
    """152 single-CTA 128 x 256 tiles on 148 CTAs / 80 pair tiles of 256 x 256 on 74 CTA pairs: the 4 / 6 tiles of the short last round
    run as halves (`decode` in xmr_gemm_tf32*.cuh); every element accumulates over K in the same order, so the output equals the TMR
    kernel's, whose single-CTA 128 x 128 schedule has no split"""
    A, B = operands(oracle, M, N, K, seed=12)
    split, _ = run(rt, 1, A, B)
    tmr, st = run(rt, 3, A, B)
    assert split.tobytes() == tmr.tobytes() and st.errors_corrected == 0
    ref = tf32(A).astype(np.float64) @ tf32(B).astype(np.float64)
    assert np.abs(split - ref).max() <= 2e-6 * K


@pytest.mark.parametrize("M,N,K", [(256, 256, 32), (256, 256, 256), (512, 768, 96), (1024, 512, 2048), (2560, 4096, 64)])
def test_gemm_cta_pair_kernels_are_bit_identical_to_the_single_cta_kernels(rt, oracle, M, N, K):
    """the unprotected and DWC kernels run on CTA pairs (xmr_gemm_tf32p_*, tcgen05 cta_group::2, 256 x BN pair tiles, each CTA stages
    half of B), TMR on single CTAs (xmr_gemm_tf32_*): same operands, same accumulation order over K per element -> the same bits for
    every replica count; with injected faults, the outputs and counters the protection promises"""
    A, B = operands(oracle, M, N, K, seed=21)
    single, _ = run(rt, 3, A, B)
    for nc in (1, 2):
        C, st = run(rt, nc, A, B)
        assert C.tobytes() == single.tobytes(), (nc, np.abs(C - single).max())
        assert st.errors_corrected == st.dwc_detected == st.injected == 0
    check_faults_against_clean(rt, oracle, A, B, single, seed=3, p=0.01)
    ref = tf32(A).astype(np.float64) @ tf32(B).astype(np.float64)
    assert np.abs(single - ref).max() <= 2e-6 * K


@pytest.mark.parametrize("M", [384, 512])
def test_gemm_a_operand_collector_reuse_changes_nothing(rt, oracle, M):
    """DWC / TMR: the replicas of a k-step keep A in the tensor core's collector (tcgen05.mma collector::a::fill / use / lastuse) instead
    of re-reading it from shared memory -- same products, same accumulation order: the bits of the unprotected kernel, which issues
    plain MMAs, with and without faults.  M = 384 runs DWC and TMR on single CTAs, M = 512 runs DWC on CTA pairs."""
    N, K = 768, 352
    A, B = operands(oracle, M, N, K, seed=31)
    plain, _ = run(rt, 1, A, B)
    for nc in (2, 3):
        C, st = run(rt, nc, A, B)
        assert C.tobytes() == plain.tobytes() and st.errors_corrected == st.dwc_detected == 0
    check_faults_against_clean(rt, oracle, A, B, plain, seed=8, p=0.01)
    ref = tf32(A).astype(np.float64) @ tf32(B).astype(np.float64)
    assert np.abs(plain - ref).max() <= 2e-6 * K


def test_gemm_faults_are_voted_out_and_counted(rt, oracle):
    import coast_b200 as cb
    M, N, K = 256, 384, 128
    A, B = operands(oracle, M, N, K, seed=9)
    clean, _ = run(rt, 1, A, B)
    plan = cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=41, p=0.05)
    C3, st3 = run(rt, 3, A, B, plan=plan)
    assert C3.tobytes() == clean.tobytes()
    _, so = oracle.run(oracle.K_GEMM_TF32, 3, A, M * N, M=M, N=N, K=K, aux=B, flags=3,
                       plan=oracle.make_plan(oracle.PLAN_BERNOULLI, seed=41, p=0.05))
    assert st3.injected == so["injected"] > 3000
    assert st3.errors_corrected == so["errors_corrected"] == st3.injected and st3.first_fault_unit == so["first_fault_unit"]
    C2, st2 = run(rt, 2, A, B, plan=plan)
    _, so2 = oracle.run(oracle.K_GEMM_TF32, 2, A, M * N, M=M, N=N, K=K, aux=B,
                        plan=oracle.make_plan(oracle.PLAN_BERNOULLI, seed=41, p=0.05))
    assert st2.dwc_detected == so2["dwc_detected"] == st2.injected
    # DWC stores r0: elements whose fault hit replica 0 differ from clean in exactly one bit
    diff = (C2.view(np.uint32) ^ clean.view(np.uint32)).ravel()
    nz = diff[diff != 0]
    assert len(nz) > 0 and all(bin(int(x)).count("1") == 1 for x in nz[:200])


def test_gemm_table_plan(rt, oracle):
    import torch
    import coast_b200 as cb
    M, N, K = 128, 128, 64
    A, B = operands(oracle, M, N, K, seed=2)
    clean, _ = run(rt, 1, A, B)
    tab = np.zeros(M * N, dtype=np.uint32)
    picks = [(0, 0, 31), (5, 1, 0), (127 * 128 + 127, 2, 17), (64 * 128 + 3, 0, 22)]
    for u, r, b in picks:
        tab[u] = oracle.fault_entry(r, 0, b)
    tab[77] = oracle.fault_entry(0, 1, 3)          # site 1 does not exist -> ignored
    plan = cb.FaultPlan(mode=cb.PLAN_TABLE, table=torch.from_numpy(tab.view(np.int32)).cuda())
    C, st = run(rt, 3, A, B, plan=plan)
    assert C.tobytes() == clean.tobytes() and st.injected == 4 and st.errors_corrected == 4 and st.first_fault_unit == 0


def test_gemm_full_size_config4(rt, oracle):
    """4096 x 4096 x 4096: TMR output == unprotected output (bit-exact), spot rows against the fp64 reference."""
    import torch
    import coast_b200 as cb
    n = 4096
    dA = torch.empty(n * n, dtype=torch.float32, device="cuda")
    dB = torch.empty(n * n, dtype=torch.float32, device="cuda")
    rt.fill_philox(dA, seed=4)
    rt.fill_philox(dB, seed=44)
    # Philox words -> uniform(-1,1) floats, on device
    dA = (dA.view(torch.int32).to(torch.float64) / 2 ** 31).to(torch.float32).contiguous()
    dB = (dB.view(torch.int32).to(torch.float64) / 2 ** 31).to(torch.float32).contiguous()
    c1, _ = rt.run(cb.K_GEMM_TF32, 1, dA, n * n, M=n, N=n, K=n, aux=dB, out=torch.empty(n * n, dtype=torch.float32, device="cuda"))
    c3, st = rt.run(cb.K_GEMM_TF32, 3, dA, n * n, M=n, N=n, K=n, aux=dB, flags=3, out=torch.empty(n * n, dtype=torch.float32, device="cuda"),
                    plan=cb.FaultPlan(mode=cb.PLAN_BERNOULLI, seed=4, p=2 ** -12))
    assert torch.equal(c1.view(torch.int32), c3.view(torch.int32))
    assert st.errors_corrected == st.injected > 3000 and st.syncs == n * n
    A = dA.view(n, n)
    B = dB.view(n, n)
    rows = [0, 1, 2047, 4095]
    At = (A[rows].view(torch.int32) & -8192).view(torch.float32).to(torch.float64)
    Bt = (B.view(torch.int32) & -8192).view(torch.float32).to(torch.float64)
    ref = (At @ Bt).cpu().numpy()
    got = c3.view(n, n)[rows].cpu().numpy()
    assert np.abs(got - ref).max() <= 2e-6 * n
