"""GEMM kernels against torch fp64 matmul, through the C-ABI test hook gmvae_debug_gemm."""
import pytest
import torch

from tests.helpers import CONFIGS, make_engine
from tests.test_step_gpu import _record

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    e = make_engine(CONFIGS["tiny_vae"], "bf16")
    yield e
    e.close()


def _ref(A, B, ta, tb):
    A64, B64 = A.double(), B.double()
    return (A64.t() if ta else A64) @ (B64.t() if tb else B64)


@pytest.mark.parametrize("M,N,K,ta,tb,split", [
    (37, 50, 19, False, False, 1), (100, 512, 784, False, False, 1), (100, 10, 512, False, True, 1),
    (784, 512, 100, True, False, 1), (10, 128, 4096, True, False, 16), (65, 67, 1000, True, True, 3),
])
def test_simt_gemm(eng, M, N, K, ta, tb, split):
    g = torch.Generator().manual_seed(M * 7 + N)
    A = torch.randn((K, M) if ta else (M, K), generator=g)
    B = torch.randn((N, K) if tb else (K, N), generator=g)
    C = eng.debug_gemm(0, A, B, ta, tb, split).cpu().double()
    R = _ref(A, B, ta, tb)
    assert ((C - R).norm() / R.norm()).item() < 2e-6


def _bf16(t):
    return t.to(torch.bfloat16).to(torch.float32)


# K-major x K-major: forward / dgrad shapes.  A [M,K], B stored [N,K].
@pytest.mark.parametrize("M,N,K", [
    (128, 128, 64), (128, 64, 128), (100, 512, 784), (256, 784, 512), (300, 128, 512), (100, 64, 512),
    (129, 1024, 64), (16384, 512, 512), (100, 112, 72), (1000, 256, 1024), (16384, 784, 512), (4000, 10, 512),
    (4000, 512, 10), (3000, 24, 40), (20000, 128, 10),
])
def test_tc_gemm_kmajor(eng, M, N, K):
    g = torch.Generator().manual_seed(M + N + K)
    A = _bf16(torch.randn(M, K, generator=g)); B = _bf16(torch.randn(N, K, generator=g))
    C = eng.debug_gemm(1, A, B, False, True).cpu().double()
    R = _ref(A, B, False, True)
    assert ((C - R).norm() / R.norm()).item() < 1e-5     # bf16 inputs are exact; only fp32 accumulation differs


# MN-major x MN-major: weight-gradient shapes.  A stored [K,M], B stored [K,N]; K = batch.
@pytest.mark.parametrize("M,N,K,split", [
    (128, 128, 64, 1), (128, 64, 128, 1), (512, 512, 100, 1), (784, 512, 100, 2), (512, 784, 256, 3),
    (64, 512, 1000, 4), (512, 128, 16384, 37), (200, 136, 333, 2), (512, 512, 16384, 18), (784, 512, 16384, 10),
    (10, 512, 5000, 8), (512, 10, 5000, 8),
])
def test_tc_gemm_mnmajor(eng, M, N, K, split):
    g = torch.Generator().manual_seed(M + N + K)
    A = _bf16(torch.randn(K, M, generator=g)); B = _bf16(torch.randn(K, N, generator=g))
    C = eng.debug_gemm(1, A, B, True, False, split).cpu().double()
    R = _ref(A, B, True, False)
    assert ((C - R).norm() / R.norm()).item() < 1e-5


# K-major x MN-major: the forward GEMM of a layer outside the chained kernel, A [M,K] (activations), B stored [K,N] (the
# weight as stored), dispatched to the tile widths 64 / 128 / 256 that encode, decode and condition get.  M, N and K take the
# values below in a pairwise sample (every pair of values of two of them appears once: K = FWD_K[(i + j) % 7] for
# FWD_M[i], FWD_N[j]); N spans all three tile widths, their partial tiles and the model's real widths; K is unpadded or ends
# in a ragged k-block.
FWD_M = [1, 127, 128, 129, 4097, 16384, 32768]
FWD_N = [10, 16, 17, 33, 64, 65, 128, 129, 256, 257, 520, 784, 1024]
FWD_K = [7, 33, 64, 65, 97, 784, 1024]
FWD_CASES = [(m, n, FWD_K[(i + j) % len(FWD_K)]) for i, m in enumerate(FWD_M) for j, n in enumerate(FWD_N)]
# Tile counts around the persistent grid (min(tiles, SMs) CTAs): N = 256 is one 256-wide n-tile, so M = 128 t - 5 rows make t
# tiles, the last m-tile partial; t = SMs - 1, SMs, SMs + 1, 2 SMs and 4 SMs, read from the device.
FWD_SM_MULTIPLES = [("sms-1", 1, -1), ("sms", 1, 0), ("sms+1", 1, 1), ("2sms", 2, 0), ("4sms", 4, 0)]
# Element-wise bar |C - R| <= FWD_TOL * (|A| @ |B|): the inputs are bf16-exact, so the only error is fp32 accumulation (and
# the fp32 store).  Measured on one B200 (power limit 1000 W), worst over every case below: 4.1e-7 at (16384, 256, 1024).
FWD_TOL = 1e-6


def _fwd_check(eng, M, N, K, tag):
    g = torch.Generator().manual_seed(M * 31 + N * 7 + K)
    A = _bf16(torch.randn(M, K, generator=g)); B = _bf16(torch.randn(K, N, generator=g))
    C = eng.debug_gemm(1, A, B, False, False).double()
    A64, B64 = A.to(eng.device, torch.float64), B.to(eng.device, torch.float64)
    R = A64 @ B64
    S = A64.abs() @ B64.abs()
    fig = ((C - R).abs() / S.clamp_min(1e-300)).max().item()
    _record("tc_gemm_forward", {"tag": tag, "M": M, "N": N, "K": K, "err_over_abs_product": fig})
    bad = (C - R).abs() > FWD_TOL * S
    assert not bool(bad.any()), (M, N, K, int(bad.sum()), bad.nonzero()[:4].tolist(), fig)


@pytest.mark.parametrize("M,N,K", FWD_CASES)
def test_tc_gemm_forward(eng, M, N, K):
    _fwd_check(eng, M, N, K, "pairwise")


@pytest.mark.parametrize("tag,mult,off", FWD_SM_MULTIPLES, ids=[t[0] for t in FWD_SM_MULTIPLES])
def test_tc_gemm_forward_tiles_vs_sms(eng, tag, mult, off):
    sms = torch.cuda.get_device_properties(eng.device).multi_processor_count
    t = mult * sms + off
    _fwd_check(eng, 128 * t - 5, 256, 97, f"tiles={tag} ({t} tiles, {sms} SMs)")


def test_debug_gemm_refuses_mn_major_a_with_k_major_b(eng):
    A = torch.zeros(16, 8); B = torch.zeros(16, 8)
    with pytest.raises(RuntimeError, match="debug hook covers"):
        eng.debug_gemm(1, A, B, True, True)
