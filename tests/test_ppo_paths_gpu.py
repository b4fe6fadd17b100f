"""The PPO kernels against the fp64 oracles on every code path their shapes select, in math modes 3, 1 and 0.

``hrp_ppo.cu`` / ``hrp_mlp_tc.cu`` choose among code paths from the shapes and the flat-buffer offsets: tensor cores or
the SIMT ``sgemm_kernel`` (M >= 32 and N >= 32), one segmented ``[a1 | c1]`` GEMM or two head GEMMs (H % 64), the N tile
width, the operand staging (S % 4, H % 4, the weights' alignment in the flat buffer, which ``log_std`` shifts by A
floats), the vectorised or scalar epilogue, the fused or unfused act heads, and the split caps of the backward
(B > 4096, B > 8192).  Every ``CASES`` / ``CAT_CASES`` entry names the path it is there to reach.

Per case: ``forward`` (mean or logits, value); ``act`` deterministic, with given noise, and sampled (the returned
log-prob is the oracle's for the returned sample); ``hrp_ppo_loss_grad_ex`` with the clipped value loss (every metric and
the whole gradient), on the rows directly and gathered through ``idx`` out of a larger rollout, which must give the same
bits; one ``hrp_clip_adam_step`` against ``ppo_ref.clip_adam``.  The oracles (``oracle/ppo_ref.py``,
``oracle/ppo_categorical_ref.py``, ``tests/ppo_options_oracle.py``) run in float64 on the GPU.

Inputs stay off the kinks, so that a mismatch means arithmetic and not a branch taken differently:
* states: a row with a hidden pre-activation within 1e-4 of 0 is redrawn (``_relu_margin``).  Where math mode 1 runs
  the forward on tensor cores (B >= 32 and H >= 32) the TF32 twin's pre-activations must keep that margin too: there the
  kernel's ReLU masks are the twin's, not the oracle's;
* the pre-tanh actions of the loss and of the noise path have |z| <= 2.5, where log(1 - tanh(z)^2 + 1e-6) is well
  conditioned;
* a row whose probability ratio (oracle's or twin's) lies within 1e-2 of 1 +- eps_clip gets its old log-prob moved by
  0.03, and the old values / returns keep every case of the clipped value loss 0.2 c away from its kinks
  (``_old_values``).

Tolerances, one rule per quantity (s = sqrt(max(1, S / 256)): the rules grow with the length of the first layer's
reduction, which only the K = 1280 and K = 4608 rows reach):
* modes 3 and 0: mean / logits / value / pre-tanh 2e-5 s; log-prob 5e-5 s per action dimension (one for a categorical
  policy); loss 2e-5 s max(1, |loss|), actor / entropy / approx_kl 2e-5 s, critic 2e-5 s max(1, critic), clip fraction
  0.5 / B; gradient 1e-4 s max|grad| + 2e-6 s; after one clip + Adam step, parameters 5e-6 where the clipped gradient
  exceeds 1e-5 and 3.1e-4 (the step's lr bound) everywhere, moments 1e-5 relative + 1e-6 of their max;
* mode 1: the bound of modes 3 and 0 plus K_TF32 = 2 times max|twin - oracle| of the same quantity, where the twin
  (``tests/tf32_twin.py``) is the oracle with every operand of the four hidden Linear layers truncated to TF32 in the
  forward and the backward.  The kernel truncates the same operands (or, on its SIMT GEMMs, none), so its distance to
  the oracle is at most the twin's, elementwise, up to fp32 rounding;
* a sampled log-prob is compared at the kernel's own z: its rule plus |z - mean| / std^2 times the mean's bound, per
  action dimension (the kernel's mean enters it).
The worst err / bound ratio per quantity and mode is printed at the end of the module.
"""
import math
from dataclasses import dataclass

import numpy as np
import pytest
import torch

import tf32_twin
from oracle import ppo_categorical_ref as cref
from oracle import ppo_ref
from ppo_options_oracle import loss_and_grad, loss_and_grad_cat
from test_ppo_options_gpu import _agent, _ex, _lib, _old_values, _relu_margin

pytestmark = pytest.mark.gpu

MODES = [3, 1, 0]
K_TF32 = 2.0
MARGIN = 1e-4
CLIP_V = 1.0


@dataclass(frozen=True)
class Case:
    row: int
    S: int
    A: int
    H: int
    B: int
    path: str


CASES = [
    Case(1, 60, 2, 256, 4096, "baseline: segmented [a1|c1] GEMM, act heads fused in 128-wide tiles, mode-1 cp.async "
                              "staging (w1 8-byte aligned)"),
    Case(2, 64, 4, 256, 64, "w1 16-byte aligned (ST_K4 x ST_K4), 32-wide narrow trunk tiles (mode 3), fused act in "
                            "64-wide tiles"),
    Case(3, 60, 1, 256, 64, "w1 at an odd float offset: scalar K staging"),
    Case(4, 25, 3, 128, 8193, "S < 32: dW1 on SIMT split-K; B > 8192: split cap and colsum cap; last loss CTA holds "
                              "one row"),
    Case(5, 61, 4, 320, 4096, "odd S; H % 128 != 0 forces 64-wide tiles on the segmented GEMM"),
    Case(6, 60, 2, 96, 4096, "H % 64 != 0: two head GEMMs into ac, unfused heads_act_kernel"),
    Case(7, 60, 3, 102, 1000, "H % 4 != 0: scalar epilogue and masks, transpose with H % 32 != 0, ragged M tile"),
    Case(8, 60, 2, 16, 4096, "H < 32: every hidden GEMM on SIMT in every mode"),
    Case(9, 7, 4, 64, 33, "tiny K, M one past 32"),
    Case(10, 60, 3, 256, 31, "B < 32: SIMT throughout, unfused act"),
    Case(11, 60, 2, 256, 65536, "64k-env minibatch: 32 splits of ~2048 rows, 64 colsum chunks, 4096 loss CTAs"),
    Case(12, 4608, 1, 64, 128, "widest observation VecNormalize accepts, K = 4608"),
    Case(13, 1280, 2, 256, 256, "S > 1024"),
    Case(14, 60, 4, 2496, 16, "(A + 1) H 4 bytes > 48 KB of shared memory in the unfused heads_act_kernel"),
]
# the categorical head has no log_std: its weights sit A floats earlier, so its staging differs
CAT_CASES = [Case(c.row, c.S, n, c.H, c.B, c.path + f" (categorical, n = {n})")
             for c, n in zip([c for c in CASES if c.row in (4, 5, 6, 7, 11)], [2, 3, 5, 8, 2])]

RATIOS = {}


@pytest.fixture(scope="module", autouse=True)
def _ratio_table():
    yield
    print("\nworst err / bound per quantity and math mode:")
    for (q, mode), r in sorted(RATIOS.items()):
        print(f"  {q:24s} mode {mode}: {r:.3g}")


def _check(case, mode, q, got, want, bound):
    """|got - want| <= bound elementwise (bound: scalar or tensor); records the worst ratio."""
    got = torch.as_tensor(got, dtype=torch.float64).cpu()
    want = torch.as_tensor(want, dtype=torch.float64).cpu()
    bound = torch.as_tensor(bound, dtype=torch.float64).cpu()
    assert torch.isfinite(got).all(), (case.row, q, "non-finite kernel output")
    ratio = float(((got - want).abs() / bound).max()) if got.numel() else 0.0
    RATIOS[(q, mode)] = max(RATIOS.get((q, mode), 0.0), ratio)
    assert ratio <= 1.0, f"row {case.row} ({case.path}), mode {mode}, {q}: err / bound = {ratio:.3g}"


def _dmax(a, b):
    return float((torch.as_tensor(a, dtype=torch.float64) - torch.as_tensor(b, dtype=torch.float64)).abs().max())


def _states(flat, case, discrete, g):
    """B fp32-representable states with every hidden pre-activation at least MARGIN from 0 (oracle, and twin where
    mode 1 runs the forward on tensor cores), drawn on the host from g, checked on the GPU in fp64."""
    S, A, H, B = case.S, case.A, case.H, case.B
    tc = B >= 32 and H >= 32
    rows, have = [], 0
    for _ in range(400):
        cand = (torch.randn(max(B, 4096), S, generator=g) * 0.5).float().double().cuda()
        ok = _relu_margin(flat, cand, S, A, H, discrete) > MARGIN
        if tc:
            with tf32_twin.tf32(H):
                ok &= _relu_margin(flat, cand, S, A, H, discrete) > MARGIN
        rows.append(cand[ok])
        have += int(ok.sum())
        if have >= B:
            return torch.cat(rows)[:B]
    raise AssertionError(f"row {case.row}: too few states off the ReLU kinks")


class _Prepared:
    pass


_CACHE = {}


def _prepare(case, discrete):
    """Agent, inputs and the oracle's and the twin's results of one case (built once, shared by its three modes)."""
    key = (case.row, discrete)
    if key in _CACHE:
        return _CACHE[key]
    _CACHE.clear()
    S, A, H, B = case.S, case.A, case.H, case.B
    torch.manual_seed(1000 + case.row)
    p = _Prepared()
    p.agent = _agent(S, A, H, B, discrete)
    flat = p.flat = p.agent.actor_critic.flat.double()
    g = p.g = torch.Generator().manual_seed(case.row)
    x = p.x = _states(flat, case, discrete, g)
    ref = cref if discrete else ppo_ref
    with torch.no_grad():
        if discrete:
            p.o_fwd = ref.forward(flat, x, S, A, H)
            with tf32_twin.tf32(H):
                p.t_fwd = ref.forward(flat, x, S, A, H)
            p.noise = torch.rand(B, generator=g, dtype=torch.float64).clamp(1e-6, 1 - 1e-6).float()
        else:
            mean, log_std, value = ref.forward(flat, x, S, A, H)
            with tf32_twin.tf32(H):
                t_mean, _, t_value = ref.forward(flat, x, S, A, H)
            p.o_fwd, p.t_fwd = (mean, value), (t_mean, t_value)
            std = log_std.exp()
            zc = (mean + std * torch.randn(B, A, generator=g, dtype=torch.float64).cuda()).clamp(-2.5, 2.5)
            p.noise = ((zc - mean) / std).float()
            n64 = p.noise.double().cuda()
            p.o_noise = (mean + std * n64, ref.evaluate(flat, x, mean + std * n64, S, A, H)[0])
            with tf32_twin.tf32(H):
                p.t_noise = (t_mean + std * n64, ref.evaluate(flat, x, t_mean + std * n64, S, A, H)[0])
    # one minibatch of the loss
    if discrete:
        act = torch.randint(0, A, (B,), generator=g).cuda()
        pre = act.float().view(B, 1)
        with torch.no_grad():
            logp = cref.evaluate(flat, x, act, S, A, H)[0]
            with tf32_twin.tf32(H):
                t_logp = cref.evaluate(flat, x, act, S, A, H)[0]
    else:
        act = (p.o_fwd[0] + torch.randn(B, A, generator=g, dtype=torch.float64).cuda()).clamp(-2.5, 2.5).float().double()
        pre = act.float()
        with torch.no_grad():
            logp = ppo_ref.evaluate(flat, x, act, S, A, H)[0]
            with tf32_twin.tf32(H):
                t_logp = ppo_ref.evaluate(flat, x, act, S, A, H)[0]
    old = logp + 0.2 * torch.randn(B, generator=g, dtype=torch.float64).cuda()
    near = torch.zeros(B, dtype=torch.bool, device="cuda")
    for lp in (logp, t_logp):
        ratio = torch.exp(lp - old)
        near |= ((ratio - 0.8).abs() < 1e-2) | ((ratio - 1.2).abs() < 1e-2)
    old = torch.where(near, old - 0.03, old).float().double()
    adv = torch.randn(B, generator=g, dtype=torch.float64).float().double().cuda()
    vo, R, _ = _old_values(p.o_fwd[1].view(-1).cpu(), CLIP_V, g)
    vo, R = vo.cuda(), R.cuda()
    fn = loss_and_grad_cat if discrete else loss_and_grad
    p.o_loss = fn(flat, x, act, old, adv, R, S, A, H, old_value=vo, clip_value=CLIP_V)
    with tf32_twin.tf32(H):
        p.t_loss = fn(flat, x, act, old, adv, R, S, A, H, old_value=vo, clip_value=CLIP_V)
    p.dev = {"states": x.float(), "pre_tanh": pre.contiguous(), "log_prob": old.float(), "adv": adv.float(),
             "ret": R.float()}
    p.vo = vo.float()
    _CACHE[key] = p
    return p


def _with_mode(lib, _l, mode):
    prev = lib.hrp_ppo_get_math()
    _l.check(lib.hrp_ppo_set_math(mode))
    return prev


def _tf(mode, d):
    """The mode-1 term of a bound: K_TF32 times the twin's distance to the oracle."""
    return K_TF32 * d if mode == 1 else 0.0


def _loss_and_adam(case, mode, p, lib, _l, s):
    """hrp_ppo_loss_grad_ex on the rows and through idx (bit-identical), metrics and gradient against the oracle, then
    one clip + Adam step against ppo_ref.clip_adam."""
    B = case.B
    agent, ac = p.agent, p.agent.actor_critic
    o, t = p.o_loss, p.t_loss
    _l.check(_ex(lib, agent, p.dev, None, B, p.vo, CLIP_V), "hrp_ppo_loss_grad_ex")
    grad, m = agent.grad.clone(), agent._metrics.clone()
    # the same minibatch gathered out of a 2B-row rollout
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(case.row + 7))
    src = (2 * perm).cuda()
    big = {k: torch.zeros((2 * B,) + v.shape[1:], dtype=v.dtype, device="cuda") for k, v in p.dev.items()}
    big_vo = torch.zeros(2 * B, device="cuda")
    for k in p.dev:
        big[k][src] = p.dev[k]
    big_vo[src] = p.vo
    _l.check(_ex(lib, agent, big, src, B, big_vo, CLIP_V), "hrp_ppo_loss_grad_ex")
    assert torch.equal(agent.grad, grad) and torch.equal(agent._metrics, m), (case.row, mode, "idx path differs")
    _l.check(_ex(lib, agent, p.dev, None, B, p.vo, CLIP_V), "hrp_ppo_loss_grad_ex")
    assert torch.equal(agent.grad, grad), (case.row, mode, "a second run differs")
    m = m.cpu().numpy().astype(np.float64)
    _check(case, mode, "loss", m[0], o["loss"], 2e-5 * s * max(1.0, abs(o["loss"])) + _tf(mode, abs(t["loss"] - o["loss"])))
    for i, k in ((1, "actor"), (3, "entropy"), (5, "approx_kl")):
        _check(case, mode, k, m[i], o[k], 2e-5 * s + _tf(mode, abs(t[k] - o[k])))
    _check(case, mode, "critic", m[2], o["critic"],
           2e-5 * s * max(1.0, o["critic"]) + _tf(mode, abs(t["critic"] - o["critic"])))
    _check(case, mode, "clip_fraction", m[4], o["clip_fraction"],
           0.5 / B + _tf(mode, abs(t["clip_fraction"] - o["clip_fraction"])))
    assert m[6] == 1.0
    want = o["grad"]
    _check(case, mode, "grad", grad, want,
           (1e-4 * float(want.abs().max()) + 2e-6) * s + _tf(mode, _dmax(t["grad"], want)))
    # one clip + Adam step from zero moments on the kernel's gradient
    n = ac.num_params
    prm, ea, eas = ac.flat.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    step, scratch = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(128, device="cuda")
    _l.check(lib.hrp_clip_adam_step(prm.data_ptr(), grad.data_ptr(), ea.data_ptr(), eas.data_ptr(), step.data_ptr(), n,
                                    3e-4, 0.9, 0.999, 1e-8, 0.5, scratch.data_ptr(), torch.cuda.current_stream().cuda_stream),
             "hrp_clip_adam_step")
    g64 = grad.double()
    zero = torch.zeros_like(g64)
    p1, m1, v1, total = ppo_ref.clip_adam(p.flat, g64, zero, zero, 1)
    assert int(step.item()) == 1
    _check(case, mode, "adam exp_avg", ea, m1, 1e-5 * m1.abs() + 1e-6 * float(m1.abs().max()) + 1e-30)
    _check(case, mode, "adam exp_avg_sq", eas, v1, 1e-5 * v1.abs() + 1e-6 * float(v1.abs().max()) + 1e-30)
    solid = g64.abs() * min(1.0, 0.5 / total) > 1e-5
    assert int(solid.sum()) > 0
    _check(case, mode, "adam params", prm[solid], p1[solid], 5e-6)
    _check(case, mode, "adam params (all)", prm, p1, 3.1e-4)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", CASES, ids=[f"row{c.row}-S{c.S}-A{c.A}-H{c.H}-B{c.B}" for c in CASES])
def test_gaussian_paths_match_fp64(case, mode):
    _l, lib = _lib()
    p = _prepare(case, False)
    S, A, H, B = case.S, case.A, case.H, case.B
    s = math.sqrt(max(1.0, S / 256))
    ac = p.agent.actor_critic
    prev = _with_mode(lib, _l, mode)
    try:
        x32 = p.dev["states"]
        (o_mean, o_val), (t_mean, t_val) = p.o_fwd, p.t_fwd
        b_mean = 2e-5 * s + _tf(mode, _dmax(t_mean, o_mean))
        b_val = 2e-5 * s + _tf(mode, _dmax(t_val, o_val))
        mean, std, value = ac.forward(x32)
        _check(case, mode, "mean", mean, o_mean, b_mean)
        _check(case, mode, "value", value, o_val, b_val)
        mean2, _, value2 = ac.forward(x32)
        assert torch.equal(mean, mean2) and torch.equal(value, value2), (case.row, mode, "a second run differs")

        det = ac.act(x32, deterministic=True)
        _check(case, mode, "act pre_tanh", det["pre_tanh"], o_mean, b_mean)
        _check(case, mode, "act value", det["value"], o_val.view(-1), b_val)
        _check(case, mode, "act action", det["action"], torch.tanh(det["pre_tanh"].double()), 1e-6)

        out = ac.act(x32, noise=p.noise.cuda().contiguous())
        (o_z, o_lp), (t_z, t_lp) = p.o_noise, p.t_noise
        _check(case, mode, "act pre_tanh", out["pre_tanh"], o_z, 2e-5 * s + _tf(mode, _dmax(t_z, o_z)))
        _check(case, mode, "act log_prob", out["log_prob"], o_lp, 5e-5 * s * A + _tf(mode, _dmax(t_lp, o_lp)))
        _check(case, mode, "act value", out["value"], o_val.view(-1), b_val)
        _check(case, mode, "act action", out["action"], torch.tanh(out["pre_tanh"].double()), 1e-6)

        smp = ac.act(x32)
        z = smp["pre_tanh"].double()
        sd = p.agent.actor_critic.log_std.double().exp()
        nrm = (z - o_mean) / sd
        assert torch.isfinite(nrm).all() and float(nrm.abs().max()) < 6.5
        if B >= 1000:
            assert abs(float(nrm.mean())) < 0.1 and 0.9 < float(nrm.std()) < 1.1
        _check(case, mode, "act action", smp["action"], torch.tanh(z), 1e-6)
        _check(case, mode, "act value", smp["value"], o_val.view(-1), b_val)
        keep = z.abs().max(1).values <= 2.5
        assert int(keep.sum()) >= max(1, B // 2)
        with torch.no_grad():
            lp_o = ppo_ref.evaluate(p.flat, p.x[keep], z[keep], S, A, H)[0]
            d_lp = 0.0
            if mode == 1:
                with tf32_twin.tf32(H):
                    d_lp = _dmax(ppo_ref.evaluate(p.flat, p.x[keep], z[keep], S, A, H)[0], lp_o)
        slope = ((z[keep] - o_mean[keep]).abs() / sd ** 2).sum(1)
        _check(case, mode, "sampled log_prob", smp["log_prob"][keep], lp_o, 5e-5 * s * A + _tf(mode, d_lp) + slope * b_mean)

        _loss_and_adam(case, mode, p, lib, _l, s)
    finally:
        lib.hrp_ppo_set_math(prev)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", CAT_CASES, ids=[f"row{c.row}-S{c.S}-n{c.A}-H{c.H}-B{c.B}" for c in CAT_CASES])
def test_categorical_paths_match_fp64(case, mode):
    _l, lib = _lib()
    p = _prepare(case, True)
    S, n, H, B = case.S, case.A, case.H, case.B
    s = math.sqrt(max(1.0, S / 256))
    ac = p.agent.actor_critic
    prev = _with_mode(lib, _l, mode)
    try:
        x32 = p.dev["states"]
        (o_lg, o_val), (t_lg, t_val) = p.o_fwd, p.t_fwd
        b_lg = 2e-5 * s + _tf(mode, _dmax(t_lg, o_lg))
        b_val = 2e-5 * s + _tf(mode, _dmax(t_val, o_val))
        logits, none, value = ac.forward(x32)
        assert none is None
        _check(case, mode, "logits", logits, o_lg, b_lg)
        _check(case, mode, "value", value, o_val, b_val)
        o_logp = torch.log_softmax(o_lg, -1)
        rows = torch.arange(B, device="cuda")

        det = ac.act(x32, deterministic=True)
        ids = det["action"][:, 0].long()
        top = torch.sort(o_lg, 1).values
        clear = top[:, -1] - top[:, -2] > 2 * b_lg
        assert torch.equal(ids[clear], o_lg.argmax(1)[clear]) and bool((det["action"][:, 1] == 0).all())
        _check(case, mode, "act value", det["value"], o_val.view(-1), b_val)

        out = ac.act(x32, noise=p.noise.cuda())
        ids = out["action"][:, 0].long()
        want, margin = cref.sample(torch.softmax(o_lg, -1).cpu().numpy(), p.noise.double().numpy())
        sure = torch.from_numpy(margin > 1e-5 + 4 * b_lg).cuda()
        assert torch.equal(ids[sure], torch.from_numpy(want).cuda()[sure])
        assert torch.equal(out["pre_tanh"][:, 0].long(), ids)
        # log_softmax moves by at most twice the largest logit error
        _check(case, mode, "act log_prob", out["log_prob"], o_logp[rows, ids], 5e-5 * s + 2 * b_lg)

        smp = ac.act(x32)
        ids = smp["action"][:, 0].long()
        assert bool(((ids >= 0) & (ids < n)).all())
        _check(case, mode, "sampled log_prob", smp["log_prob"], o_logp[rows, ids], 5e-5 * s + 2 * b_lg)
        _check(case, mode, "act value", smp["value"], o_val.view(-1), b_val)

        _loss_and_adam(case, mode, p, lib, _l, s)
    finally:
        lib.hrp_ppo_set_math(prev)


# -- clip + Adam over several steps --------------------------------------------------------------------------------------
ADAM_N = [1, 511, 512, 513, 61439, 61440, 61441] + [sum(int(np.prod(s)) for _, s in ppo_ref.shapes(c.S, c.A, c.H))
                                                    for c in CASES if c.row in (11, 14)]


@pytest.mark.parametrize("lr_on_device", [False, True], ids=["lr-by-value", "lr-on-device"])
@pytest.mark.parametrize("n", ADAM_N)
def test_clip_adam_ten_steps_match_fp64(n, lr_on_device):
    """hrp_clip_adam_step(_ex) against ppo_ref.clip_adam in fp64 over 10 steps that alternate clipped (norm 2) and
    unclipped (norm 0.2) gradients at varying learning rates: 120 CTAs of 512 threads cover 61440 elements, so n = 61441
    and the parameter counts of rows 11 and 14 go round the grid-stride loop.  Both take the kernel's own fp32 state and
    the same gradients.  Moments to 1e-5 relative + 1e-6 of their max, parameters to 2e-6 where every clipped gradient
    exceeded 1e-6 = 100 eps (Adam divides by sqrt(v) + eps), the step counter exactly."""
    _l, lib = _lib()
    g = torch.Generator(device="cuda").manual_seed(n)
    st = torch.cuda.current_stream().cuda_stream
    p0 = torch.randn(n, generator=g, device="cuda") * 0.1
    prm, ea, eas = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    step, scratch = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(128, device="cuda")
    lrs = [3e-4, 1e-4, 2.5e-3, 7e-5, 1e-3, 3e-4, 5e-4, 2e-4, 1e-4, 4e-4]
    lr_dev = torch.zeros(1, dtype=torch.float64, device="cuda")
    p64, m64, v64 = p0.double(), torch.zeros(n, dtype=torch.float64, device="cuda"), \
        torch.zeros(n, dtype=torch.float64, device="cuda")
    solid = torch.ones(n, dtype=torch.bool, device="cuda")
    clipped = 0
    for it, lr in enumerate(lrs):
        norm = 2.0 if it % 2 == 0 else 0.2
        grad = torch.randn(n, generator=g, device="cuda")
        grad *= norm / float(grad.double().norm())
        if lr_on_device:
            lr_dev.fill_(lr)
            rc = lib.hrp_clip_adam_step_ex(prm.data_ptr(), grad.data_ptr(), ea.data_ptr(), eas.data_ptr(),
                                           step.data_ptr(), n, 0.5, lr_dev.data_ptr(), 0.9, 0.999, 1e-8, 0.5,
                                           scratch.data_ptr(), st)
        else:
            rc = lib.hrp_clip_adam_step(prm.data_ptr(), grad.data_ptr(), ea.data_ptr(), eas.data_ptr(), step.data_ptr(),
                                        n, lr, 0.9, 0.999, 1e-8, 0.5, scratch.data_ptr(), st)
        _l.check(rc, "hrp_clip_adam_step")
        p64, m64, v64, total = ppo_ref.clip_adam(p64, grad.double(), m64, v64, it + 1, lr=lr)
        clipped += total > 0.5
        solid &= grad.double().abs() * min(1.0, 0.5 / total) > 1e-6
        assert int(step.item()) == it + 1
        for name, got, want in (("exp_avg", ea, m64), ("exp_avg_sq", eas, v64)):
            err = (got.double() - want).abs()
            bound = 1e-5 * want.abs() + 1e-6 * float(want.abs().max()) + 1e-30
            assert bool((err <= bound).all()), (n, it, name, float((err / bound).max()))
        assert bool(torch.isfinite(prm).all())
        if bool(solid.any()):
            err = float((prm.double() - p64).abs()[solid].max())
            assert err <= 2e-6, (n, it, err)
    assert clipped == len(lrs) // 2
    assert int(solid.sum()) > n // 2


# -- hrp_ppo_act_multi ------------------------------------------------------------------------------------------------
MULTI_DIMS = [(1, 1), (33, 31), (1000, 999), (1024, 1024)]


def _policy(S, A, H, g):
    """A flat parameter buffer with nn.Linear's initial ranges and a log_std in [-0.5, 0.5]."""
    parts = []
    for name, shp in ppo_ref.shapes(S, A, H):
        if name == "log_std":
            parts.append(torch.rand(shp, generator=g, dtype=torch.float64) - 0.5)
        else:
            fan_in = S if name.startswith("shared.0") else H
            parts.append((torch.rand(shp, generator=g, dtype=torch.float64) * 2 - 1) / math.sqrt(fan_in))
    return torch.cat([q.reshape(-1) for q in parts]).float()


def test_act_multi_matches_fp64_over_three_chunks():
    """One hrp_ppo_act_multi call with 70 items (three launches of at most 32) of every A in 1..4 and (S, H) from 1 x 1
    to 1024 x 1024, deterministic and sampled items mixed: deterministic means and values against ppo_ref.forward in
    fp64 (2e-5 sqrt(max(1, S / 256)), the matrix-vector products reduce in fp32), sampled log-probs against
    ppo_ref.evaluate at the returned pre-tanh action with the rule of the batched act above."""
    _l, lib = _lib()
    g = torch.Generator().manual_seed(5)
    pols = {}
    for A in range(1, 5):
        for S, H in MULTI_DIMS:
            pols[(S, A, H)] = _policy(S, A, H, g).cuda()
    keys = list(pols)
    count = 70
    items = (_l.HrpActItem * count)()
    states, outs, meta = [], [], []
    for i in range(count):
        S, A, H = keys[i % len(keys)]
        x = (torch.randn(S, generator=g) * 0.5).cuda()
        out = torch.full((2 * A + 2,), float("nan"), device="cuda")
        det = i % 3 == 0
        it = items[i]
        it.params_dev, it.state_dev, it.out_dev = pols[(S, A, H)].data_ptr(), x.data_ptr(), out.data_ptr()
        it.seed, it.draw, it.row = 77 + i, 3, i
        it.state_dim, it.action_dim, it.hidden_dim, it.deterministic = S, A, H, int(det)
        states.append(x)
        outs.append(out)
        meta.append((S, A, H, det))
    _l.check(lib.hrp_ppo_act_multi(items, count, torch.cuda.current_stream().cuda_stream), "hrp_ppo_act_multi")
    torch.cuda.synchronize()
    checked = 0
    for i, (S, A, H, det) in enumerate(meta):
        s = math.sqrt(max(1.0, S / 256))
        flat = pols[(S, A, H)].double()
        x = states[i].double().view(1, S)
        mean, log_std, value = ppo_ref.forward(flat, x, S, A, H)
        got = outs[i].double()
        assert torch.isfinite(got).all(), (i, S, A, H)
        z = got[A:2 * A]
        np.testing.assert_allclose(got[:A].cpu(), torch.tanh(z).cpu(), atol=1e-6)
        assert abs(float(got[2 * A + 1] - value.view(()))) <= 2e-5 * s, (i, S, A, H)
        if det:
            assert float((z - mean.view(-1)).abs().max()) <= 2e-5 * s, (i, S, A, H)
            assert float(got[2 * A]) == 0.0
        else:
            sd = log_std.exp()
            nrm = (z - mean.view(-1)) / sd
            assert float(nrm.abs().max()) < 6.5, (i, S, A, H)
            if float(z.abs().max()) <= 2.5:   # where log(1 - tanh(z)^2 + 1e-6) is well conditioned
                lp = ppo_ref.evaluate(flat, x, z.view(1, A), S, A, H)[0]
                slope = float(((z - mean.view(-1)).abs() / sd ** 2).sum())
                tol = 5e-5 * s * A + slope * 2e-5 * s
                assert abs(float(got[2 * A] - lp.view(()))) <= tol, (i, S, A, H, float(got[2 * A]), float(lp))
                checked += 1
    assert checked >= 20


# -- policies wider than the single-state kernel ---------------------------------------------------------------------------
def test_single_state_act_of_a_wide_policy_falls_back_to_the_batched_kernels():
    """S = 1280, H = 1100 is beyond hrp_ppo_act_multi (HRP_ACT_MAX_DIM = 1024): get_action takes the batched kernels and
    equals the batched deterministic act bit for bit and the fp64 oracle within the forward's rule; sampling works;
    act_item refuses the policy with a ValueError naming the limit (the multiplexer then fails only that experiment)."""
    from highway_rope_ppo_b200 import _lib as L

    S, A, H = 1280, 2, 1100
    torch.manual_seed(3)
    agent = _agent(S, A, H, 8, False)
    ac = agent.actor_critic
    x = (torch.randn(S, generator=torch.Generator().manual_seed(4)) * 0.5).cuda()
    action, pre, lp, value = ac.get_action(x, deterministic=True)
    assert lp is None
    want = ac.act(x.view(1, S), deterministic=True)
    assert np.array_equal(pre, want["pre_tanh"].cpu().numpy().reshape(-1))
    assert np.array_equal(action, want["action"].cpu().numpy().reshape(-1))
    assert value == want["value"].cpu().numpy().reshape(())
    flat = ac.flat.double()
    mean, _, v64 = ppo_ref.forward(flat, x.double().view(1, S), S, A, H)
    s = math.sqrt(S / 256)
    assert float((torch.from_numpy(pre).double() - mean.cpu().view(-1)).abs().max()) <= 2e-5 * s
    assert abs(float(value) - float(v64)) <= 2e-5 * s
    action, pre, lp, value = ac.get_action(x)
    assert lp is not None and np.isfinite(lp) and np.all(np.isfinite(pre))
    np.testing.assert_allclose(action, np.tanh(pre), atol=1e-6)
    out = agent.select_action(x.cpu().numpy())
    assert out is not None
    with pytest.raises(ValueError, match=str(L.ACT_MAX_DIM)):
        ac.act_item(x, torch.empty(2 * A + 2, device="cuda"), True)
