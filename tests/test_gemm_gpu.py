"""tcgen05 GEMM (hrp_gemm_strided) against a float64 torch reference, for every operand orientation the MLP
forward / backward uses.  Tolerances: 3xTF32 mode 1e-5 of max|C| (fp32-grade: the TMEM accumulator is fp32); single-pass TF32 mode 2e-3 of
sqrt(K) * max|A| * max|B| (10-bit mantissa operands)."""
import numpy as np
import pytest
import torch

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
]


@pytest.mark.parametrize("M,N,K,akc,bkc", CASES)
@pytest.mark.parametrize("mode", [3, 1])
def test_tc_gemm_matches_float64(M, N, K, akc, bkc, mode):
    g = torch.Generator(device="cuda:0").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn((M, K) if akc else (K, M), generator=g, device="cuda:0")
    B = torch.randn((N, K) if bkc else (K, N), generator=g, device="cuda:0")
    Am = A if akc else A.t()
    Bm = B if bkc else B.t()
    want = (Am.double() @ Bm.double().t())
    sam, sak = (K, 1) if akc else (1, M)
    sbn, sbk = (K, 1) if bkc else (1, N)
    got = _gemm(A, sam, sak, B, sbn, sbk, M, N, K, mode)
    assert torch.isfinite(got).all()
    err = (got.double() - want).abs().max().item()
    if mode == 3:
        # the TMEM accumulator adds K products in fp32 without intermediate rounding to nearest: allow growth with K
        assert err <= 1e-5 * max(1.0, K / 512) * want.abs().max().item() + 1e-6, err
    else:
        assert err <= 2e-3 * np.sqrt(K) * 4.0 * 4.0 / 4, err


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
