"""tcgen05 GEMM (hrp_gemm_strided) against a float64 torch reference, for every operand orientation the MLP
forward / backward uses, M, N or K of 1, long and ragged K, and operands 4, 8 or 12 bytes off a 16-byte boundary.

Tolerances are per element, from P = |A| |B| (the sum of the magnitudes of the K products of C[i, j]):
* 3xTF32 (mode 3) against A B in fp64: (2^-18 + 2^-22 sqrt(K)) P.  The split of each operand into two TF32 halves
  leaves at most ~2^-18.4 of a product; the fp32 accumulator's roundings grow like sqrt(K) per unit of P;
* single-pass TF32 (mode 1) against trunc(A) trunc(B) in fp64, trunc being what the tensor core does to an fp32 operand
  (tools/tf32_probe.py): 2^-22 sqrt(K) P.  The products are exact, so only the fp32 accumulation is left.
"""
import numpy as np
import pytest
import torch

from tf32_twin import trunc

pytestmark = pytest.mark.gpu


def _gemm(A, sam, sak, B, sbn, sbk, M, N, K, mode, bias=None, relu=0):
    from highway_rope_ppo_b200 import _lib

    lib = _lib.load()
    C = torch.full((M, N), float("nan"), device="cuda:0")
    _lib.check(lib.hrp_gemm_strided(M, N, K, A.data_ptr(), sam, sak, B.data_ptr(), sbn, sbk, C.data_ptr(), N,
                                    _lib.ptr(bias), relu, mode, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return C


CASES = [  # (M, N, K, a_k_contig, b_k_contig)
    (4096, 256, 60, True, True),     # layer 1 forward: X[B,60] W1[256,60]^T
    (4096, 256, 256, True, True),    # hidden forward
    (4096, 256, 256, True, False),   # dX = dY W: B(n,k) = W[k, n]
    (256, 256, 4096, False, False),  # dW = dY^T X: both batch-major
    (256, 60, 4096, False, False),   # dW1
    (4096, 512, 256, True, True),    # [actor | critic] hidden layer: 128-wide N tiles
    (4096, 256, 512, True, False),   # d(h2): K = 2H against W[k, n]
    (512, 256, 4096, False, False),  # [dWa1 ; dWc1]
    (64, 256, 60, True, True),       # the reference's minibatch sizes (main.py:53): one partial M tile
    (32, 128, 128, True, False),
    (200, 96, 72, True, True),       # ragged M / N / K with 16-byte aligned pitches
    (72, 200, 136, False, False),
    (136, 72, 200, False, True),
    (100, 70, 45, True, True),       # ragged edges everywhere, unaligned pitches
    (129, 257, 33, False, True),
    (32, 32, 8, True, True),
    (1, 256, 60, True, True),        # M = 1, N = 1, K = 1
    (4096, 1, 256, True, False),
    (64, 128, 1, True, True),
    (1, 1, 1, False, False),
    (300, 200, 7, True, True),       # K = 7, 33: one partial K block
    (129, 96, 33, True, False),
    (256, 128, 4100, False, False),  # long ragged K, both operands batch-major
    (96, 128, 45, False, False),     # both MN-contiguous with ragged K (ST_MNK4)
    (64, 64, 7, False, False),
]


def _bound(A, B, K, mode):
    """Per-element tolerance of the module docstring; A [M, K], B [N, K] as multiplied."""
    P = A.double().abs() @ B.double().abs().t()
    return ((2.0 ** -18 if mode == 3 else 0.0) + 2.0 ** -22 * np.sqrt(K)) * P + 1e-30


def _want(A, B, mode):
    if mode == 1:
        A, B = trunc(A.contiguous()), trunc(B.contiguous())
    return A.double() @ B.double().t()


@pytest.mark.parametrize("M,N,K,akc,bkc", CASES)
@pytest.mark.parametrize("mode", [3, 1])
def test_tc_gemm_matches_float64(M, N, K, akc, bkc, mode):
    g = torch.Generator(device="cuda:0").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn((M, K) if akc else (K, M), generator=g, device="cuda:0")
    B = torch.randn((N, K) if bkc else (K, N), generator=g, device="cuda:0")
    Am = A if akc else A.t()
    Bm = B if bkc else B.t()
    sam, sak = (K, 1) if akc else (1, M)
    sbn, sbk = (K, 1) if bkc else (1, N)
    got = _gemm(A, sam, sak, B, sbn, sbk, M, N, K, mode)
    assert torch.isfinite(got).all()
    ratio = ((got.double() - _want(Am, Bm, mode)).abs() / _bound(Am, Bm, K, mode)).max().item()
    assert ratio <= 1.0, ratio


OFFSET_CASES = [  # (M, N, K, a_k_contig, b_k_contig)
    (200, 96, 72, True, True),
    (72, 200, 136, False, False),
    (136, 72, 200, False, True),
    (256, 256, 64, True, False),
]


@pytest.mark.parametrize("off_a,off_b", [(1, 0), (2, 2), (3, 1), (0, 3), (1, 3)])
@pytest.mark.parametrize("M,N,K,akc,bkc", OFFSET_CASES)
@pytest.mark.parametrize("mode", [3, 1])
def test_tc_gemm_unaligned_operands_match_float64(M, N, K, akc, bkc, off_a, off_b, mode):
    """A and B starting 1, 2 or 3 floats past a 16-byte boundary (pitches that are multiples of 4): the scalar, 8-byte
    and 16-byte operand staging and, in mode 1, the cp.async path, against the same per-element bounds."""
    g = torch.Generator(device="cuda:0").manual_seed(M + N + K + 10 * off_a + off_b)
    bufa = torch.randn(M * K + 4, generator=g, device="cuda:0")
    bufb = torch.randn(N * K + 4, generator=g, device="cuda:0")
    A = bufa[off_a:off_a + M * K].view((M, K) if akc else (K, M))
    B = bufb[off_b:off_b + N * K].view((N, K) if bkc else (K, N))
    assert (A.data_ptr() - bufa.data_ptr()) == 4 * off_a and bufa.data_ptr() % 16 == 0
    Am = A if akc else A.t()
    Bm = B if bkc else B.t()
    sam, sak = (K, 1) if akc else (1, M)
    sbn, sbk = (K, 1) if bkc else (1, N)
    got = _gemm(A, sam, sak, B, sbn, sbk, M, N, K, mode)
    assert torch.isfinite(got).all()
    ratio = ((got.double() - _want(Am, Bm, mode)).abs() / _bound(Am, Bm, K, mode)).max().item()
    assert ratio <= 1.0, ratio


def test_tc_gemm_bias_relu_epilogue():
    M, N, K = 300, 256, 60
    g = torch.Generator(device="cuda:0").manual_seed(1)
    A, B = torch.randn((M, K), generator=g, device="cuda:0"), torch.randn((N, K), generator=g, device="cuda:0")
    bias = torch.randn(N, generator=g, device="cuda:0")
    got = _gemm(A, K, 1, B, K, 1, M, N, K, 3, bias=bias, relu=1)
    want = torch.relu(A.double() @ B.double().t() + bias.double())
    assert (got.double() - want).abs().max().item() <= 1e-5 * want.abs().max().item()


def test_math_modes_agree_on_the_policy_forward():
    """hrp_ppo_forward in fp32 SIMT mode vs tensor-core modes on the same weights."""
    from highway_rope_ppo_b200 import _lib
    from highway_rope_ppo_b200.ppo.agent import PPOAgent

    lib = _lib.load()
    torch.manual_seed(0)
    agent = PPOAgent(60, 2, hidden_dim=256, batch_size=512, device="cuda:0")
    x = torch.randn(512, 60, device="cuda:0") * 0.5
    outs = {}
    try:
        for mode in (0, 3, 1):
            _lib.check(lib.hrp_ppo_set_math(mode))
            mean, _, value = agent.actor_critic.forward(x)
            outs[mode] = (mean.clone(), value.clone())
    finally:
        lib.hrp_ppo_set_math(3)
    assert (outs[3][0] - outs[0][0]).abs().max().item() < 2e-6 and (outs[3][1] - outs[0][1]).abs().max().item() < 2e-6
    assert (outs[1][0] - outs[0][0]).abs().max().item() < 5e-3 and (outs[1][1] - outs[0][1]).abs().max().item() < 5e-3
