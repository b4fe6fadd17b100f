"""The data-parallel PPO update against the fp64 update of the whole batch it stands for, on one GPU.

A. Shard sums of the kernels, one process.  One global minibatch of B_g rows is split into W equal shards, and
``hrp_ppo_loss_grad_kl`` runs on each with ``loss_scale = 1 / (B_l W)`` (``ppo/distributed.py``), the clipped value loss,
a KL output and a zero stop word.  The W gradients, metric vectors and KL shares are added in rank order in fp32, the
order of the peer-memory exchange (``csrc/hrp_comm.cu``), and compared with the fp64 oracle of the whole minibatch under
the rules of ``tests/test_ppo_paths_gpu.py`` (whose inputs, off the ReLU / ratio / value-clip kinks, are reused);
``metrics[6]`` must be 1 within W 2^-24.  The shapes put the shards on another kernel path than the whole minibatch would
take: across the B > 8192 and B > 4096 split caps, the scalar epilogue (H % 4 != 0, where the three-term rank-order sum
is not commutative), tensor cores at 32 rows and SIMT at 16.  ``hrp_adv_stats`` per shard, the three doubles summed,
then ``hrp_adv_normalize`` against a two-pass fp64 normalization of the global buffer.

B. W gloo ranks, all on ``cuda:0``, against the global fp64 update.  Under a non-NCCL group the agent turns off the
peer-memory exchange and the captured collectives, so W gloo processes on one device run the Python of the NCCL path:
eager all-reduces of the advantage moments, the gradient (P + 1 floats with target_kl), the explained-variance moments
and the metrics, then ``hrp_clip_adam_step[_ex|_kl]``.  A module fixture spawns each W in {2, 4} once; every rank runs
every case and saves what it holds, and the parent runs the oracles.  The oracle of one update: GAE per env, one
unbiased normalization over all envs, global minibatch k = the union over ranks of each rank's slice k of the (shared)
local permutation mapped to global sample ids, the mean loss over its B W samples, ``ppo_ref.clip_adam``.  Parameters to
1e-4 of the oracle's largest parameter motion and metrics to 2e-3 relative (the rules of the existing full-update
tests), the explained variance to 1e-6 of its fp64 value, and every rank bit-identical.  VecNormalize: after three
rollouts every rank's statistics are bit-identical, and after a reset and one fixed-action step they are those of
``tests/vecnormalize_oracle.py`` over the envs of all ranks, within 1e-12 relative.  The training loop
(``train_vectorized``, its episode statistics and its evaluation) on W env shards against the same job in one process.

At 215k parameters (the S = 60, H = 256 update) Adam turns gradients within the kernels' fp32 error into full steps of
either sign, so that update and the same update run unsharded are held to one rule: every parameter within the largest
motion, and 0.1 of it where the gradient is >= 1e-3 of the largest at every step.  The first update of the training
loop (16.6k parameters) is held to 1e-4 of the motion there and 1e-3 over all parameters.
"""
import math
import os
import socket
import time
from datetime import timedelta

import numpy as np
import pytest
import torch

import target_kl_oracle
from oracle import gae_bootstrap as gb
from oracle import ppo_categorical_ref as cref
from oracle import ppo_ref
from ppo_options_oracle import loss_and_grad, loss_and_grad_cat
from test_ppo_options_gpu import _agent, _fill_rollout, _lib
from test_ppo_paths_gpu import CLIP_V, RATIOS, Case, _check, _prepare

pytestmark = pytest.mark.gpu

U32, U64 = 2.0 ** -24, 2.0 ** -53


@pytest.fixture(scope="module", autouse=True)
def _ratio_table():
    yield
    print("\nworst err / bound per quantity and math mode (shard sums):")
    for (q, mode), r in sorted(RATIOS.items()):
        if q.startswith("shard "):
            print(f"  {q:24s} mode {mode}: {r:.3g}")
    for W, t in sorted(SPAWN_SECONDS.items()):
        print(f"  {W} gloo ranks on one device: every case in {t:.1f} s")


# -- A. shard sums of the loss kernels -----------------------------------------------------------------------------------
def _shards(row, S, A, H, B, discrete, worlds, path):
    return [(Case(row, S, A, H, B, path), discrete, W) for W in worlds]


SHARDS = (_shards(201, 60, 2, 256, 16384, False, (2, 4, 8), "shards of 8192 / 4096 / 2048 rows: below the B > 8192 and "
                                                          "B > 4096 split caps")
          + _shards(202, 60, 3, 102, 3000, False, (3,), "H % 4 != 0: scalar epilogue, three-term rank-order sum")
          + _shards(203, 60, 4, 256, 64, False, (2, 4), "32-row shards on tensor cores, 16-row shards on SIMT")
          + _shards(204, 60, 5, 256, 8192, True, (2, 4), "categorical n = 5, shards of 4096 / 2048 rows")
          + _shards(205, 60, 8, 102, 96, True, (3,), "categorical n = 8, H % 4 != 0, 32-row shards"))


@pytest.mark.parametrize("mode", [3, 0])
@pytest.mark.parametrize("case,discrete,W", SHARDS,
                         ids=[f"{'cat' if d else 'gauss'}-A{c.A}-H{c.H}-B{c.B}-W{W}" for c, d, W in SHARDS])
def test_shard_sums_match_the_global_minibatch(case, discrete, W, mode):
    """Each shard's metrics[5] increment is its KL share bit for bit; the rank-order fp32 sums of the W shards match the
    fp64 oracle of the whole minibatch with the bounds of test_ppo_paths_gpu.py (S = 60: s = 1)."""
    from highway_rope_ppo_b200.ppo import distributed

    _l, lib = _lib()
    p = _prepare(case, discrete)
    B, Bl = case.B, case.B // W
    agent, ac = p.agent, p.agent.actor_critic
    st = torch.cuda.current_stream().cuda_stream
    kl = torch.zeros(1, device="cuda")
    stop = torch.zeros(1, dtype=torch.int32, device="cuda")
    prev = lib.hrp_ppo_get_math()
    _l.check(lib.hrp_ppo_set_math(mode))
    try:
        grad = metrics = kl_sum = None
        for r in range(W):
            rows = slice(r * Bl, (r + 1) * Bl)
            d = {k: v[rows] for k, v in p.dev.items()}
            agent._metrics.zero_()
            kl.fill_(-1.0)
            _l.check(lib.hrp_ppo_loss_grad_kl(
                ac._h, ac.flat.data_ptr(), d["states"].data_ptr(), d["pre_tanh"].data_ptr(), d["log_prob"].data_ptr(),
                d["adv"].data_ptr(), d["ret"].data_ptr(), None, Bl, 0.2, 0.5, 0.005, distributed.loss_scale(Bl, W),
                p.vo[rows].data_ptr(), CLIP_V, kl.data_ptr(), stop.data_ptr(), agent.grad.data_ptr(),
                agent._metrics.data_ptr(), st), "hrp_ppo_loss_grad_kl")
            assert kl.item() == agent._metrics[5].item(), (r, "the KL share is not metrics[5]'s increment")
            # rank order: ((g0 + g1) + g2) + ..., in fp32
            grad = agent.grad.clone() if grad is None else grad + agent.grad
            metrics = agent._metrics.clone() if metrics is None else metrics + agent._metrics
            kl_sum = kl.clone() if kl_sum is None else kl_sum + kl
        assert int(stop.item()) == 0
    finally:
        lib.hrp_ppo_set_math(prev)
    o = p.o_loss
    m = metrics.cpu().numpy().astype(np.float64)
    _check(case, mode, "shard loss", m[0], o["loss"], 2e-5 * max(1.0, abs(o["loss"])))
    for i, k in ((1, "actor"), (3, "entropy"), (5, "approx_kl")):
        _check(case, mode, f"shard {k}", m[i], o[k], 2e-5)
    _check(case, mode, "shard critic", m[2], o["critic"], 2e-5 * max(1.0, o["critic"]))
    _check(case, mode, "shard clip_fraction", m[4], o["clip_fraction"], 0.5 / B)
    _check(case, mode, "shard count", m[6], 1.0, W * U32)
    _check(case, mode, "shard kl (P + 1)", kl_sum, o["approx_kl"], 2e-5)
    want = o["grad"]
    _check(case, mode, "shard grad", grad, want, 1e-4 * float(want.abs().max()) + 2e-6)


# -- A. advantage normalization across shards ----------------------------------------------------------------------------
def _adv_bound(a, n_local, W):
    """Per-element bound of hrp_adv_stats (per shard) + fp64 sum over shards + hrp_adv_normalize against the exact
    (a - mean) / (std + 1e-8), with mean and unbiased std of the global buffer a (fp64, n = W n_local).

    Sums: every term passes through at most k = ceil(n_l / (nb 256)) (a thread's grid-stride loop, nb = min(256,
    ceil(n_l / 256)) blocks) + 5 (warp shuffles) + 8 (warps) + nb (blocks) + W (shards) fp64 additions, so
    |S^ - S| <= k u64 sum|a| and |Q^ - Q| <= k u64 Q (a^2 of a float is exact in fp64).  Then, u64 = 2^-53, u32 = 2^-24:
      mean:  e_mu = |S^ - S| / n + u64 |mu|;  rounded to float: e_m = e_mu + u32 (|mu| + e_mu)
      var:   (Q^ - n mean^2) / (n - 1):  e_var = (|Q^ - Q| + n (2|mu| + e_mu) e_mu + 3 u64 (Q + n (|mu| + e_mu)^2))
             / (n - 1) + u64 var, the cancellation in Q^ - n mean^2 being what grows with |mu| / sd
      sd:    e_sd = e_var / sd + u64 sd (|sqrt x - sqrt y| <= |x - y| / sqrt y), rounded to float: + u32 (sd + e_sd),
             and the fp32 add of 1e-8: e_den = e_sdf + u32 (D + e_sdf) with D = sd + 1e-8
      a - m: one fp32 subtract: e_num = e_m + u32 (|a - mu| + e_m)
      out:   (|d| + e_num) / (D - e_den) - |d| / D <= (e_num + |d| e_den / D) / (D - e_den), plus the divide's
             u32 (|d| + e_num) / (D - e_den),  d = a - mu
    with a margin of 1 % for the first-order terms dropped and 1e-300 for an exact zero."""
    a = a.double()
    n = a.numel()
    nb = min(256, -(-n_local // 256))
    k = -(-n_local // (nb * 256)) + 5 + 8 + nb + W
    mu, sd = float(a.mean()), float(a.std())
    Q, S1 = float((a * a).sum()), float(a.abs().sum())
    var = sd * sd
    e_mu = k * U64 * S1 / n + U64 * abs(mu)
    e_m = e_mu + U32 * (abs(mu) + e_mu)
    e_var = (k * U64 * Q + n * (2 * abs(mu) + e_mu) * e_mu + 3 * U64 * (Q + n * (abs(mu) + e_mu) ** 2)) / (n - 1) \
        + U64 * var
    e_sd = e_var / sd + U64 * sd
    e_sdf = e_sd + U32 * (sd + e_sd)
    D = sd + 1e-8
    e_den = e_sdf + U32 * (D + e_sdf)
    d = (a - mu).abs()
    e_num = e_m + U32 * (d + e_m)
    return 1.01 * ((e_num + d * e_den / D) / (D - e_den) + U32 * (d + e_num) / (D - e_den)) + 1e-300


ADV = [(n, 3) for n in (1, 255, 256, 257, 65536, 65537)] + [(2 ** 24 + 3, 1)]


@pytest.mark.parametrize("ratio", [0.0, 10.0, 1e3], ids=["mu0", "mu10sd", "mu1e3sd"])
@pytest.mark.parametrize("n_local,W", ADV, ids=[f"n{n}-W{W}" for n, W in ADV])
def test_sharded_adv_normalization_matches_fp64(n_local, W, ratio):
    """hrp_adv_stats on each of W shards of n_local elements, the (sum, sum of squares, n) triples summed in rank
    order in fp64, hrp_adv_normalize on each shard with the sums, against (a - mean) / (std + 1e-8) of the whole buffer
    in two-pass fp64, elementwise within _adv_bound.  65537 is past 256 blocks x 256 threads, so the grid-stride loop
    of hrp_adv_stats runs; the last row is one unsharded buffer of 2^24 + 3 elements."""
    _l, lib = _lib()
    st = torch.cuda.current_stream().cuda_stream
    sd = 2.5
    g = torch.Generator(device="cuda").manual_seed(n_local * 7 + W)
    a = (torch.randn(n_local * W, generator=g, device="cuda", dtype=torch.float64) * sd + ratio * sd).float()
    total = torch.zeros(3 + 512, dtype=torch.float64, device="cuda")
    for r in range(W):
        stats = torch.zeros(3 + 512, dtype=torch.float64, device="cuda")
        _l.check(lib.hrp_adv_stats(a[r * n_local:].data_ptr(), n_local, stats.data_ptr(), st), "hrp_adv_stats")
        assert float(stats[2]) == n_local
        total[:3] += stats[:3]
    out = a.clone()
    for r in range(W):
        _l.check(lib.hrp_adv_normalize(out[r * n_local:].data_ptr(), n_local, total.data_ptr(), st), "hrp_adv_normalize")
    a64 = a.double()
    want = (a64 - a64.mean()) / (a64.std() + 1e-8)
    bound = _adv_bound(a, n_local, W)
    err = (out.double() - want).abs()
    ratio_ = float((err / bound).max())
    RATIOS[("shard adv normalize", 0)] = max(RATIOS.get(("shard adv normalize", 0), 0.0), ratio_)
    assert torch.isfinite(out).all() and ratio_ <= 1.0, (n_local, W, ratio, ratio_)


def test_adv_normalization_of_one_element_is_nan_like_torch_std():
    """n = 1: the unbiased variance is 0 / 0, and torch.std (the reference's normalization, agent.py:204) gives NaN."""
    _l, lib = _lib()
    st = torch.cuda.current_stream().cuda_stream
    a = torch.tensor([1.5], device="cuda")
    stats = torch.zeros(3 + 512, dtype=torch.float64, device="cuda")
    _l.check(lib.hrp_adv_stats(a.data_ptr(), 1, stats.data_ptr(), st), "hrp_adv_stats")
    _l.check(lib.hrp_adv_normalize(a.data_ptr(), 1, stats.data_ptr(), st), "hrp_adv_normalize")
    assert math.isnan(float(ppo_ref.normalize_adv(np.array([1.5], np.float32))[0]))
    assert math.isnan(float(a[0]))


# -- B. W gloo ranks on cuda:0 -------------------------------------------------------------------------------------------
SMALL = (12, 16, 10, 20)    # (S, H, T, E_g)
VARIANTS = {
    "ragged": dict(shape=SMALL, bs=30, epochs=3),      # 100 or 50 local samples: the last minibatch holds 10 or 20
    "wide": dict(shape=(60, 256, 8, 1024), bs=1024, epochs=2),
    "clip_value_set_lr": dict(shape=SMALL, bs=30, epochs=3, clip_value=0.2, lrs=(2e-4, 5e-5)),
    # lr 3e-3 (set_lr): the KL reaches ~1e-4 within the update, far above its fp32 error
    "target_kl": dict(shape=SMALL, bs=30, epochs=3, own_logp=True, lrs=(3e-3,)),
    "bootstrap_truncated": dict(shape=SMALL, bs=30, epochs=3, boot=True),
}
POLICIES = {"gaussian": (False, 2), "categorical": (True, 5)}
SPAWN_SECONDS = {}
VN_E, VN_T, VN_SEED = 256, 8, 3
# case R: train_vectorized on E envs in all (E / W per rank), K evaluation episodes per rank, highway-v0 of 5 s so that
# every env ends an episode within the first rollout.  K >= 32: the act path takes tensor cores on the shards' evaluation
# batches as on the single process's (below 32 rows it runs on SIMT, whose last bits differ)
LOOP = dict(E=512, H=64, T=8, iterations=2, K=32, bs=512, epochs=2, seed=7)
ROLLOUT_KEYS = ("states", "action", "pre_tanh", "log_prob", "value", "reward", "terminated", "truncated", "done")


def _make_agent(pol, v, target_kl=None):
    discrete, A = POLICIES[pol]
    S, H = v["shape"][:2]
    torch.manual_seed(5)      # the same initial parameters in every process
    return _agent(S, A, H, v["bs"], discrete, epochs=v["epochs"], clip_value=v.get("clip_value"), target_kl=target_kl)


def _global_data(agent, v, u):
    """A synthetic [T, E_g] rollout drawn from the agent's current parameters (tests/test_ppo_options_gpu.py's
    _fill_rollout), plus last values and, for bootstrap_truncated, termination / truncation flags and final values
    that are NaN wherever they must not be read.  Leaves the E_g-column rollout in agent.memory."""
    S, H, T, E = v["shape"]
    ac = agent.actor_critic
    X, act, old, value, reward, done = _fill_rollout(agent, T, E, 100 * u + 7)
    if v.get("own_logp"):   # the policy's own log-probs: the KL grows from ~0 during the update
        flat0 = ac.flat.cpu().double()
        with torch.no_grad():
            lp = (cref if agent.discrete else ppo_ref).evaluate(flat0, X, act, S, ac.action_dim, H)[0]
        old = lp.numpy().astype(np.float32)
        agent.memory.rollout["log_prob"].copy_(torch.from_numpy(old.reshape(T, E)).cuda())
    rng = np.random.default_rng(500 + u)
    d = dict(X=X, act=act, old=old, value=value, reward=reward, done=done,
             last=rng.standard_normal(E).astype(np.float32))
    if v.get("boot"):
        term = rng.random((T, E)) < 0.05
        trunc = (rng.random((T, E)) < 0.1) & ~term
        d.update(term=term, trunc=trunc, done=term | trunc,
                 final_value=np.where(trunc, rng.standard_normal((T, E)), np.nan).astype(np.float32))
    return d


def _load_shard(agent, d, v, W, rank):
    """Replace agent.memory's rollout by this rank's env columns of the global one."""
    T, E = v["shape"][2:]
    El = E // W
    cols = slice(rank * El, (rank + 1) * El)
    full = agent.memory.rollout
    agent.memory.rollout = None
    S = full["states"].shape[2]
    r = agent.memory.begin_rollout(T, El, S, full["action"].shape[2], full["pre_tanh"].shape[2],
                                   bootstrap_truncated=bool(v.get("boot")))
    for k in ("states", "action", "pre_tanh", "log_prob", "value", "reward"):
        r[k].copy_(full[k][:, cols])
    cu = lambda x: torch.from_numpy(np.ascontiguousarray(x[:, cols])).cuda()
    r["done"].copy_(cu(d["done"].astype(np.uint8)))
    if v.get("boot"):
        r["terminated"].copy_(cu(d["term"].astype(np.uint8)))
        r["truncated"].copy_(cu(d["trunc"].astype(np.uint8)))
        r["final_value"].copy_(cu(d["final_value"]))
    return torch.from_numpy(d["last"][cols].copy()).cuda()


def _minibatches(v, W, u):
    """Global sample ids (t E_g + e) of every minibatch of the update, all epochs: minibatch k is the union over ranks
    of each rank's slice k of the local permutation, which every rank draws after np.random.seed(11 + u)."""
    T, E = v["shape"][2:]
    El = E // W
    n = T * El
    np.random.seed(11 + u)
    perm = np.arange(n, dtype=np.int64)
    np.random.shuffle(perm)
    out = []
    for _ in range(v["epochs"]):
        for start in range(0, n, v["bs"]):
            t, e = np.divmod(perm[start:start + v["bs"]], El)
            out.append(np.concatenate([t * E + r * El + e for r in range(W)]))
    return out


def _oracle(pol, v, W, d, u, state, lr, target_kl):
    """One global fp64 update from Adam state (flat, m, v, step); returns target_kl_oracle.update's dict plus the
    explained variance of the update's values."""
    discrete, A = POLICIES[pol]
    S, H, T, E = v["shape"]
    N = T * E
    if v.get("boot"):
        adv, _ = gb.gae(d["reward"], d["value"], d["term"], d["trunc"], d["final_value"], d["last"])
    else:
        adv = np.zeros((T, E), dtype=np.float32)
        for e in range(E):
            adv[:, e], _ = ppo_ref.gae(d["reward"][:, e], d["value"][:, e], d["done"][:, e], d["last"][e])
    cu = lambda x: torch.as_tensor(np.asarray(x)).double().cuda()
    value = cu(d["value"].reshape(N))
    ret = cu((adv + d["value"]).reshape(N))        # fp32 returns, as the kernel stores them
    a = cu(adv.reshape(N))
    advn = (a - a.mean()) / (a.std() + 1e-8)
    X, act, old = cu(d["X"]), torch.as_tensor(d["act"]).cuda(), cu(d["old"])
    if not discrete:
        act = act.double()
    fn = loss_and_grad_cat if discrete else loss_and_grad
    mbs = [torch.from_numpy(i).cuda() for i in _minibatches(v, W, u)]
    c = v.get("clip_value")

    def loss_fn(flat, k):
        i = mbs[k]
        kw = {} if c is None else dict(old_value=value[i], clip_value=c)
        return fn(flat, X[i], act[i], old[i], advn[i], ret[i], S, A, H, **kw)

    res = target_kl_oracle.update(*state, len(mbs), loss_fn, target_kl, lr=lr)
    res["count"] = len(mbs)
    res["ev"] = float(1.0 - (ret - value).var() / ret.var())
    return res


def _kl_limit(pol, W):
    """target_kl such that the update stops part-way: 1.5 target_kl halfway between the KL of the minibatch k >= 1 that
    clears all earlier ones by the widest gap and the largest of those (unstopped oracle run, first update)."""
    v = VARIANTS["target_kl"]
    agent = _make_agent(pol, v)
    d = _global_data(agent, v, 0)
    flat = agent.actor_critic.flat.double()
    agent.close()
    state = (flat, torch.zeros_like(flat), torch.zeros_like(flat), 0)
    kls = [r["approx_kl"] for r in _oracle(pol, v, W, d, 0, state, v["lrs"][0], None)["records"]]
    gaps = [(kls[k] - max(kls[:k]), k) for k in range(1, len(kls))]
    gap, k = max(gaps)
    assert gap > 1e-6, kls
    return (kls[k] + max(kls[:k])) / 2 / 1.5


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _snapshot(agent, met):
    opt = agent.optimizer
    return dict(flat=agent.actor_critic.flat.cpu(), m=opt.exp_avg.cpu(), v=opt.exp_avg_sq.cpu(),
                step=int(opt.step_dev.item()), metrics=dict(met))


def _vecnormalize_case(rank, W, dev):
    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.envs.vec_normalize import VecNormalize
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training.routine import collect_rollout

    E, T, seed = VN_E, VN_T, VN_SEED
    cfg = dict(HIGHWAY_CONFIG, duration=5)
    w = VecNormalize(HighwayVecEnv(cfg, E, device=dev, env_id_base=rank * E, seed=seed))
    torch.manual_seed(0)
    agent = PPOAgent(w.N * w.F_out, 2, lr=3e-4, hidden_dim=64, batch_size=512, epochs=1, device=dev)
    obs = w.reset(seed=seed).clone()
    for _ in range(3):
        r = collect_rollout(w, agent, T, obs, bootstrap_truncated=True)
        obs = r["states"][T].clone()
    out = dict(captured=getattr(agent, "_rollout_graph", None) is not None, obs_buf=w.obs_rms.buf.cpu(),
               ret_buf=w.ret_rms.buf.cpu())
    plain = HighwayVecEnv(cfg, E, device=dev, env_id_base=rank * E, seed=seed + 1)
    w2 = VecNormalize(HighwayVecEnv(cfg, E, device=dev, env_id_base=rank * E, seed=seed + 1))
    raw0 = plain.reset(seed=seed + 1).clone()    # reset and step return the handle's own buffers
    w2.reset(seed=seed + 1)
    a = torch.linspace(-1, 1, 2 * E * W, device=dev).view(W * E, 2)[rank * E:(rank + 1) * E].contiguous()
    po, pr, pte, ptr = (x.clone() for x in plain.step(a))
    w2.step(a)
    out.update(obs_shape=tuple(plain.obs_shape), raw=[x.cpu().numpy() for x in (raw0, po, pr, pte, ptr)],
               obs_mean=w2.obs_rms.mean.cpu().numpy(), obs_var=w2.obs_rms.var.cpu().numpy(),
               obs_count=float(w2.obs_rms.count), ret_mean=float(w2.ret_rms.mean), ret_var=float(w2.ret_rms.var),
               ret_count=float(w2.ret_rms.count), returns=w2.returns.cpu().numpy())
    for e in (w, w2, plain):
        e.close()
    return out


def _run_loop(pol, E, base, K):
    """train_vectorized(LOOP["iterations"], eval_episodes=K) on E envs from global env id ``base``.  Returns its history,
    the per-episode returns of the evaluation before the first iteration, and the first rollout, the bootstrap values,
    the parameters before and after, and the metrics of the first update (snapshotted around agent.update)."""
    import copy

    from highway_rope_ppo_b200.config.base_config import HIGHWAY_CONFIG
    from highway_rope_ppo_b200.envs.highway_vec import HighwayVecEnv
    from highway_rope_ppo_b200.ppo.agent import PPOAgent
    from highway_rope_ppo_b200.training import routine

    discrete, A = POLICIES[pol]
    cfg = copy.deepcopy(HIGHWAY_CONFIG)
    cfg["duration"] = 5
    if discrete:
        cfg["action"] = {"type": "DiscreteMetaAction"}
    env = HighwayVecEnv(cfg, E, device="cuda:0", env_id_base=base, seed=LOOP["seed"])
    torch.manual_seed(5)
    agent = PPOAgent(env.N * env.F_out, A, lr=3e-4, hidden_dim=LOOP["H"], batch_size=LOOP["bs"], epochs=LOOP["epochs"],
                     device="cuda:0", discrete=discrete)
    snap, evals = {}, []
    update, evaluate = agent.update, routine.evaluate_vectorized

    def first_update(last_value=0.0):
        if snap:
            return update(last_value=last_value)
        r = agent.memory.rollout
        snap.update({k: r[k].cpu() for k in ROLLOUT_KEYS}, last=last_value.cpu(), flat0=agent.actor_critic.flat.cpu())
        met = update(last_value=last_value)
        snap.update(_snapshot(agent, met))
        return met

    def recorded(*a, **kw):
        out = evaluate(*a, **kw)
        evals.append(out["returns"].copy())
        return out

    agent.update = first_update
    routine.evaluate_vectorized = recorded
    try:
        np.random.seed(11)
        hist = routine.train_vectorized(env, agent, LOOP["iterations"], LOOP["T"], seed=LOOP["seed"], eval_episodes=K)
    finally:
        routine.evaluate_vectorized = evaluate
        agent.close()
        env.close()
    return dict(hist=hist, evals=evals, snap=snap)


def _worker(rank, W, port, out_dir, limits):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=W, timeout=timedelta(seconds=120))
    dev = torch.device("cuda", 0)
    # VecNormalize all-gathers its moments as a CUDA tensor, which gloo does (so collect_rollout must not capture it)
    probe = torch.full((2,), float(rank), dtype=torch.float64, device=dev)
    got = torch.zeros(2 * W, dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(got, probe)
    res = {"gloo_cuda_gather": torch.equal(got.cpu(), torch.arange(W, dtype=torch.float64).repeat_interleave(2)),
           "cases": {}, "loop": {}}
    for pol in POLICIES:
        for name, v in VARIANTS.items():
            agent = _make_agent(pol, v, limits[pol] if name == "target_kl" else None)
            ups = []
            for u, lr in enumerate(v.get("lrs", (None,))):
                d = _global_data(agent, v, u)
                last = _load_shard(agent, d, v, W, rank)
                if lr is not None:
                    agent.set_lr(lr)
                np.random.seed(11 + u)
                met = agent.update(last_value=last)
                ups.append(dict(data=d, **_snapshot(agent, met)))
            res["cases"][(pol, name)] = ups
            agent.close()
    res["vecnormalize"] = _vecnormalize_case(rank, W, dev)
    El = LOOP["E"] // W
    for pol in POLICIES:
        res["loop"][pol] = _run_loop(pol, El, rank * El, LOOP["K"])
    torch.cuda.synchronize()
    torch.save(res, os.path.join(out_dir, f"r{rank}.pt"))
    dist.destroy_process_group()


@pytest.fixture(scope="module", params=[2, 4], ids=["W2", "W4"])
def ranks(request, tmp_path_factory):
    """Runs every case of part B on W gloo ranks on cuda:0 (torch.multiprocessing.spawn, joined: no rank outlives the
    fixture; the group's 120 s timeout turns a lost rank into an error) and returns (W, [what each rank saved])."""
    import torch.multiprocessing as mp

    _lib()   # the library must already be built: the ranks only load it
    W = request.param
    out = tmp_path_factory.mktemp(f"ranks{W}")
    limits = {pol: _kl_limit(pol, W) for pol in POLICIES}
    t0 = time.perf_counter()
    mp.spawn(_worker, args=(W, _free_port(), str(out), limits), nprocs=W, join=True)
    SPAWN_SECONDS[W] = time.perf_counter() - t0
    return W, limits, [torch.load(out / f"r{r}.pt", weights_only=False) for r in range(W)]


@pytest.mark.timeout(900)
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("pol", list(POLICIES))
def test_sharded_update_matches_the_global_fp64_update(ranks, pol, variant):
    W, limits, res = ranks
    v = VARIANTS[variant]
    ups = [r["cases"][(pol, variant)] for r in res]
    for other in ups[1:]:
        for a, b in zip(ups[0], other):
            for k in ("flat", "m", "v"):
                assert torch.equal(a[k], b[k]), (W, k, "ranks differ")
            assert a["step"] == b["step"] and a["metrics"] == b["metrics"], (W, "ranks differ")
    agent = _make_agent(pol, v)
    flat0 = agent.actor_critic.flat.double()
    agent.close()
    target_kl = limits[pol] if variant == "target_kl" else None
    lrs = v.get("lrs", (3e-4,))
    motion, solid = _check_updates(pol, v, W, flat0, ups[0], lrs, target_kl)
    if variant != "wide":
        assert motion["all"] <= 1e-4, (variant, pol, W, motion)
        return
    # Adam moves a parameter by ~lr whatever the size of its gradient, so at 215k parameters some whose gradient is within
    # the fp32 error of the kernels step the other way.  The same update run unsharded (one process, the same samples,
    # minibatches of the same size) against its oracle deviates alike (0.03 to 0.29 of the motion over all parameters
    # measured on a B200, the sharded ones 0.16 to 0.46): which parameter flips is a matter of rounding.  Both are held
    # to the same rule: no parameter off by more than the largest motion, and 0.1 of it where every step's gradient is
    # >= 1e-3 of the largest (0.012 to 0.034 unsharded, 0.023 to 0.055 sharded).
    one = _unsharded_deviation(pol, v, W)
    assert int(solid.sum()) >= solid.numel() // 100
    for dev in (one, motion):
        assert dev["all"] <= 1.0 and dev["solid"] <= 0.1, (W, motion, one)


def _check_updates(pol, v, W, flat0, ups, lrs, target_kl):
    """The updates ``ups`` (what one rank saved) against the chained global oracle from flat0: metrics to 2e-3 relative,
    explained variance to 1e-6, step counter and target_kl decisions exactly.  Returns the final parameters' max error
    over the oracle's largest parameter motion, over all parameters and over those whose oracle gradient was >= 1e-3
    of its largest at every step, and that mask."""
    state = (flat0, torch.zeros_like(flat0), torch.zeros_like(flat0), 0)
    solid = torch.ones(flat0.numel(), dtype=torch.bool)
    for u, (up, lr) in enumerate(zip(ups, lrs)):
        o = _oracle(pol, v, W, up["data"], u, state, lr, target_kl)
        state = (o["flat"], o["m"], o["v"], o["step"])
        met = up["metrics"]
        for k, src in (("loss", "loss"), ("policy_loss", "actor"), ("value_loss", "critic"), ("entropy", "entropy"),
                       ("approx_kl", "approx_kl"), ("clip_fraction", "clip_fraction")):
            want = float(np.mean([q[src] for q in o["records"]]))
            assert abs(met[k] - want) <= 2e-3 * max(1.0, abs(want)), (W, u, k, met[k], want)
        assert abs(met["explained_variance"] - o["ev"]) <= 1e-6, (W, u, met["explained_variance"], o["ev"])
        assert up["step"] == o["step"], (W, u, up["step"], o["step"])
        if target_kl is not None:
            assert (met["optimizer_steps"], met["stopped_early"]) == (o["steps"], o["stopped"]), (W, met, o["steps"])
            assert o["stopped"] and 0 < o["steps"] < o["count"]
        solid &= torch.stack([(r["grad"].abs() >= 1e-3 * r["grad"].abs().max()) for r in o["records"]]).all(0).cpu()
    want = state[0].cpu()
    moved = float((want - flat0.cpu()).abs().max())
    err = (ups[-1]["flat"].double() - want).abs()
    out = {"all": float(err.max()) / moved, "solid": float(err[solid].max()) / moved}
    print(f"{pol} W={W}: max parameter motion {moved:.3e}, max error / motion {out['all']:.3g} over all parameters, "
          f"{out['solid']:.3g} over the {int(solid.sum())} of {solid.numel()} with solid gradients")
    return out, solid


def _unsharded_deviation(pol, v, W):
    """The W-rank update of variant v in this process as one rank with W times the minibatch size (the same samples,
    minibatch size and step count), against its oracle: what _check_updates returns, without the mask."""
    v1 = dict(v, bs=v["bs"] * W)
    agent = _make_agent(pol, v1)
    flat0 = agent.actor_critic.flat.double()
    d = _global_data(agent, v1, 0)
    last = _load_shard(agent, d, v1, 1, 0)
    np.random.seed(11)
    met = agent.update(last_value=last)
    up = dict(data=d, **_snapshot(agent, met))
    agent.close()
    return _check_updates(pol, v1, 1, flat0, [up], (3e-4,), None)[0]


@pytest.mark.timeout(900)
def test_sharded_vecnormalize_statistics_match_one_process(ranks):
    """Eager rollouts (collect_rollout does not capture under gloo), statistics bit-identical on every rank after three
    of them, and after a reset and one fixed-action step equal to the numpy restatement over all envs of all ranks."""
    from vecnormalize_oracle import VecNormOracle

    W, _, res = ranks
    vn = [r["vecnormalize"] for r in res]
    assert not any(x["captured"] for x in vn)
    for x in vn[1:]:
        assert torch.equal(x["obs_buf"], vn[0]["obs_buf"]) and torch.equal(x["ret_buf"], vn[0]["ret_buf"])
    raw = [np.concatenate([x["raw"][i] for x in vn]) for i in range(5)]
    o = VecNormOracle(W * VN_E, vn[0]["obs_shape"])
    o.reset(raw[0])
    o.step(raw[1], raw[2], raw[3], raw[4])
    rel = lambda got, want: np.all(np.abs(np.asarray(got) - want) <= 1e-12 * np.abs(want) + 1e-15)
    for x in vn:
        assert rel(x["obs_mean"], o.obs_rms.mean) and rel(x["obs_var"], o.obs_rms.var)
        assert rel(x["obs_count"], o.obs_rms.count)
        assert rel(x["ret_mean"], o.ret_rms.mean) and rel(x["ret_var"], o.ret_rms.var)
        assert rel(x["ret_count"], o.ret_rms.count)
    assert np.array_equal(np.concatenate([x["returns"] for x in vn]), o.returns)
    assert all(r["gloo_cuda_gather"] for r in res)


_ONE_PROCESS = {}


@pytest.mark.timeout(900)
@pytest.mark.parametrize("pol", list(POLICIES))
def test_sharded_training_loop_matches_one_process(ranks, pol):
    """Case R: train_vectorized on W highway-v0 shards (env_id_base = rank E / W) against the same job in one process
    of E envs.  The first rollout, concatenated over ranks, is the single process's bit for bit (every field); the
    training episodes of the first iteration (all of them end in it) have the same count and their return and length
    sums agree within 1e-12 relative (they are added in another order); the evaluation before it plays the same episodes
    with bit-identical returns; the first sharded update equals the global fp64 oracle of case U.  Later iterations
    differ from the single process: its minibatches are not the union of the ranks'."""
    W, _, res = ranks
    loops = [r["loop"][pol] for r in res]
    key = (pol, W)
    if key not in _ONE_PROCESS:
        _ONE_PROCESS[key] = _run_loop(pol, LOOP["E"], 0, LOOP["K"] * W)
    one = _ONE_PROCESS[key]
    for k in ROLLOUT_KEYS:
        assert torch.equal(torch.cat([x["snap"][k] for x in loops], 1), one["snap"][k]), (W, k)
    for x in loops:
        assert x["hist"][0]["episodes"] == one["hist"][0]["episodes"] >= LOOP["E"], (W, x["hist"][0]["episodes"])
        for k in ("episode_return_mean", "episode_return_std", "episode_length_mean", "terminated_fraction",
                  "eval_return_mean", "eval_return_std", "eval_length_mean", "eval_terminated_fraction"):
            a, b = x["hist"][0][k], one["hist"][0][k]
            assert abs(a - b) <= 1e-12 * abs(b) + 1e-15, (W, k, a, b)
        # later iterations: all-reduced figures, the same on every rank
        assert all(x["hist"][-1][k] == loops[0]["hist"][-1][k] for k in x["hist"][-1] if k != "samples_per_s"), W
    assert np.array_equal(np.concatenate([x["evals"][0] for x in loops]), one["evals"][0])
    # the first update: every rank's state is the same, and it is the oracle's
    for x in loops[1:]:
        for k in ("flat", "m", "v"):
            assert torch.equal(x["snap"][k], loops[0]["snap"][k]), (W, k)
    snap = loops[0]["snap"]
    T, S = LOOP["T"], one["snap"]["states"].shape[2]
    cat = lambda k: torch.cat([x["snap"][k] for x in loops], 1)
    N = T * LOOP["E"]
    pre = cat("pre_tanh").reshape(N, -1)
    d = dict(X=cat("states")[:T].reshape(N, S).double(), act=pre[:, 0].long() if POLICIES[pol][0] else pre.double(),
             old=cat("log_prob").reshape(N).numpy(), value=cat("value").numpy(), reward=cat("reward").numpy(),
             done=cat("done").numpy().astype(bool), last=torch.cat([x["snap"]["last"] for x in loops]).numpy())
    v = dict(shape=(S, LOOP["H"], T, LOOP["E"]), bs=LOOP["bs"], epochs=LOOP["epochs"])
    motion, _ = _check_updates(pol, v, W, snap["flat0"].double().cuda(), [dict(data=d, **snap)], (3e-4,), None)
    # 16.6k parameters: as in the wide update of case U, a few with rounding-level gradients take Adam steps of the
    # other sign (2e-4 to 4e-4 of the motion measured on a B200); the others hold the 1e-4 rule (1e-5 measured)
    assert motion["all"] <= 1e-3 and motion["solid"] <= 1e-4, (pol, W, motion)
