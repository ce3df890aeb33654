"""tcgen05 GEMM tiles (engine 1) against an fp64 matmul: single bf16 product and the two-term split.

The launchers are persistent: the NT grid is at most one CTA per SM and a CTA walks the row tiles m_first,
+m_stride, ... through NBUF = 4 TMEM accumulators; a TN CTA reduces its split of P in nk k-blocks through 2-4
shared-memory stages.  The small cases run one tile per CTA; the cases listed in NT_PERSISTENT / TN_PERSISTENT run
several (the benchmark runs 7 row tiles per NT CTA and 14 k-blocks per TN CTA), so the accumulator and stage rings
wrap and the epilogue's look-ahead loads land on later tiles.  Each of those asserts that it reaches its regime on the
device it runs on (the sizes assume the 148 SMs of a B200)."""
import ctypes as C

import pytest
import torch

import util_neus as U

pytestmark = pytest.mark.gpu

NBUF = 4                      # TMEM accumulators of the NT kernel (4 for BN = 64 and 128)
R5 = 5 * 148 * 128            # five full waves of 128-row tiles on 148 SMs
# (M, N, K) of the NT cases whose first CTA walks more than NBUF row tiles, so the accumulator ring wraps
NT_PERSISTENT = [
    (R5 + 37, 64, 64),          # BN = 64, 148 CTAs on one column tile: 6 tiles on CTA 0, ragged last tile
    (65536, 256, 256),          # the benchmark's fine-pass shape (512 rays x 128 samples, 256 wide): 7 tiles
    (65537, 256, 256),          # ... plus one row: a last tile of one row
    (40000, 300, 256),          # 3 column tiles (ragged), 147 CTAs
    (50000, 256, 320),          # K > 256: B streamed with A, no resident panel
    (100000, 128, 40),          # nk = 1
]
NT_SINGLE_PERSISTENT = [(65536, 256, 256)]
# (P, N1, N2) of the TN cases whose k-block loop is longer than the stage ring
TN_PERSISTENT = {(65536, 256, 64), (65536, 256, 128), (65536, 256, 256), (70001, 257, 39), (65536, 40, 128)}


def _tn_regime(P, N1, N2, nprod):
    """(k-blocks of the first split, shared-memory stages, rows of the last split) under launch_gemm_tc_tn's grid."""
    BN = 64 if N2 <= 64 else (128 if N2 <= 128 else 256)
    nop = 2 if nprod == 3 else 1
    stages = min(4, (200 * 1024) // (nop * (128 * 64 * 2 + BN * 64 * 2)))
    ctas = -(-N1 // 128) * -(-N2 // BN)
    splits = -(-U.sm_count() // ctas)
    rows = -(-(-(-P // splits)) // 64) * 64
    splits = -(-P // rows)
    return rows // 64, stages, P - (splits - 1) * rows


def _run(M, N, K, nprod, seed=0):
    from avatarclip_b200 import _lib
    L = _lib.lib()
    L.avc_tc_gemm_nt_test.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                      C.c_void_p, C.c_size_t, C.c_void_p]
    L.avc_tc_gemm_nt_test.restype = C.c_int
    g = torch.Generator().manual_seed(seed)
    A = torch.randn(M, K, generator=g).cuda()
    B = (torch.randn(N, K, generator=g) * 0.1).cuda()
    Cm = torch.full((M, N), float("nan"), device="cuda")
    ws = torch.empty(4 * (M + N) * ((K + 7) // 8 * 8) + 8192, dtype=torch.uint8, device="cuda")
    _lib.check(L.avc_tc_gemm_nt_test(A.data_ptr(), B.data_ptr(), M, N, K, nprod, Cm.data_ptr(), ws.data_ptr(),
                                     ws.numel(), _lib.stream_ptr()), "avc_tc_gemm_nt_test")
    torch.cuda.synchronize()
    ref = (A.double() @ B.double().t())
    err = (Cm.double() - ref).abs().max().item() / ref.abs().max().item()
    return err


@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (256, 256, 256), (1000, 217, 256), (300, 39, 256), (4096, 256, 40),
                                   (513, 128, 320)] + NT_PERSISTENT)
def test_tc_gemm_split3(M, N, K):
    if (M, N, K) in NT_PERSISTENT:
        assert U.nt_tiles_per_cta(M, N) > NBUF, U.nt_tiles_per_cta(M, N)
    err = _run(M, N, K, 3)
    print(M, N, K, "split-3 rel-to-max err", err)
    U.log_parity("tc_gemm_nt", {"M": M, "N": N, "K": K, "nprod": 3, "rel_to_max": err})
    assert err < 3e-5


@pytest.mark.parametrize("M,N,K", [(256, 256, 256), (1000, 217, 256)] + NT_SINGLE_PERSISTENT)
def test_tc_gemm_single(M, N, K):
    if (M, N, K) in NT_SINGLE_PERSISTENT:
        assert U.nt_tiles_per_cta(M, N) > NBUF, U.nt_tiles_per_cta(M, N)
    err = _run(M, N, K, 1)
    print(M, N, K, "single-bf16 rel-to-max err", err)
    U.log_parity("tc_gemm_nt", {"M": M, "N": N, "K": K, "nprod": 1, "rel_to_max": err})
    assert err < 2e-2


def _run_tn(P, N1, N2, nprod, seed=0):
    from avatarclip_b200 import _lib
    L = _lib.lib()
    L.avc_tc_gemm_tn_test.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.avc_tc_gemm_tn_test.restype = C.c_int
    g = torch.Generator().manual_seed(seed)
    A = torch.randn(P, N1, generator=g).cuda()
    B = (torch.randn(P, N2, generator=g) * 0.1).cuda()
    base = torch.randn(N1, N2, generator=g).cuda()
    Cm = base.clone()
    r8 = lambda n: (n + 7) // 8 * 8
    ws = torch.empty(4 * P * (r8(N1) + r8(N2)) + 8192, dtype=torch.uint8, device="cuda")
    cs = torch.ones(N1, device="cuda")
    _lib.check(L.avc_tc_gemm_tn_test(A.data_ptr(), B.data_ptr(), P, N1, N2, nprod, Cm.data_ptr(), cs.data_ptr(),
                                     ws.data_ptr(), ws.numel(), _lib.stream_ptr()), "avc_tc_gemm_tn_test")
    torch.cuda.synchronize()
    ref = base.double() + A.double().t() @ B.double()
    cref = 1.0 + A.double().sum(0)
    cerr = (cs.double() - cref).abs().max().item() / cref.abs().max().item()
    assert cerr < (3e-5 if nprod == 3 else 2e-2), ("fused column sum", cerr)
    return (Cm.double() - ref).abs().max().item() / ref.abs().max().item()


@pytest.mark.parametrize("P,N1,N2", [(64, 128, 64), (640, 256, 256), (5000, 217, 256), (3000, 257, 39), (9000, 40, 128)]
                         + sorted(TN_PERSISTENT))
def test_tc_gemm_tn_split3(P, N1, N2):
    if (P, N1, N2) in TN_PERSISTENT:
        nk, stages, last = _tn_regime(P, N1, N2, 3)
        assert nk > stages, (nk, stages)                   # every stage is refilled at least once
        if P % 64:
            assert 0 < last < nk * 64 and last % 64, last   # the last split is short and ends inside a k-block
    err = _run_tn(P, N1, N2, 3)
    print(P, N1, N2, "TN split-3 rel-to-max err", err)
    U.log_parity("tc_gemm_tn", {"P": P, "N1": N1, "N2": N2, "nprod": 3, "rel_to_max": err})
    assert err < 3e-5


@pytest.mark.parametrize("P,N1,N2", [(65536, 256, 256)])
def test_tc_gemm_tn_single(P, N1, N2):
    nk, stages, _ = _tn_regime(P, N1, N2, 1)
    assert nk > stages, (nk, stages)
    err = _run_tn(P, N1, N2, 1)
    print(P, N1, N2, "TN single-bf16 rel-to-max err", err)
    U.log_parity("tc_gemm_tn", {"P": P, "N1": N1, "N2": N2, "nprod": 1, "rel_to_max": err})
    assert err < 2e-2
