"""The tensor-core PPO minibatch against float64 autograd of the oracle, at every tile geometry the host set-up can choose.

One minibatch is T1 (train_fwd_bwd_tc_kernel: forward, losses, backward, feature-major slabs of leading dimension ld, one scalar slot per
CTA), T2 (wgrad_tc_kernel: the slabs reduced in 64-column chunks) and a tail (reduce_tc_kernel, or the fused finish_tc_kernel) that sums
the scalar slots of the T1 CTAs and the matrix slots of the T2 CTAs.  T1 runs 64-row half tiles when a minibatch has too few 128-row tiles
to fill the SMs, so the columns T1 covers (whole tiles of its own height) need not reach ld; T2 and the tail must read only what T1 wrote.
The workspace and the scratch come from torch.empty, so every case here runs on buffers filled with NaN first, or with the finite
left-overs of a larger minibatch: a read of anything T1 did not write shows up in the result.  The float64 oracle sits ~1e-5 from the fp32
kernels, so the bars are those of the TF32-vs-fp32 comparison in test_gpu_ppo.py."""
import ctypes
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from omniisaacgymenvs_loop_b200.rl.policy import PolicyMLP  # noqa: E402
from oracle import loopz_oracle as Z  # noqa: E402
from oracle import ppo_oracle as P  # noqa: E402
from tests.util import assert_close  # noqa: E402

DEV = "cuda:0"
H, TM, WK = 128, 128, 64          # hidden width, UMMA tile rows, T2 chunk columns (csrc/ppo_mlp_tc_impl.inc)
TAIL, SENTINEL = 256, -4242.5     # caller buffers are views into longer ones: rows >= M must come back bit-unchanged
BLOCKS = ("sigma", "w1", "b1", "w2", "b2", "wv", "bv", "wmu", "bmu")
STATS = ("a_loss", "c_loss", "entropy", "b_loss", "kl", "loss")
E_CLIP, KINK = 0.2, 0.02          # the policy's clip range; how far every sample of a minibatch stays from a kink of the clipped losses


def geometry(M, sms, tile_rows=None):
    """train_tile_rows + train_setup of csrc/ppo_mlp_tc_impl.inc: the slab leading dimension, T1's tile height, tile count and grid, the
    T2 chunk count and the slab columns T1 writes.  `tile_rows` forces the tile height (the loopz learner always runs whole tiles)."""
    ld = -(-M // TM) * TM
    ts = tile_rows or (TM // 2 if 2 * (ld // TM) <= sms else TM)
    tiles = -(-M // ts)
    return dict(ld=ld, ts=ts, tiles=tiles, g1=min(tiles, sms), nchunks=tiles * ts // WK, covered=tiles * ts)


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def minibatch_size(label, n_sms):
    """The sizes by what they exercise; `lim` is the largest minibatch that still runs on half tiles (9472 on 148 SMs)."""
    lim = n_sms // 2 * TM
    return {"one": 1, "half_tile": 64, "odd_129": 129, "odd_4800": 4800, "lim-127": lim - 127, "lim-64": lim - 64, "lim": lim,
            "lim+1": lim + 1, "ctl_65": 65, "ctl_200": 200, "ragged": 8192 * 3 + 5, "128x200": 128 * 200}[label]


def check_regime(label, M, n_sms):
    """The size is in the regime its label claims (so that the test still covers it on a GPU with another SM count)."""
    g = geometry(M, n_sms)
    if label in ("one", "half_tile", "odd_129", "odd_4800", "lim-127", "lim-64"):
        # an odd number of half tiles: T1 writes ld - 64 of the ld slab columns
        assert g["ts"] == TM // 2 and g["tiles"] % 2 == 1 and g["covered"] == g["ld"] - WK, (label, g)
    elif label in ("ctl_65", "ctl_200", "lim"):
        assert g["ts"] == TM // 2 and g["covered"] == g["ld"], (label, g)
    elif label == "lim+1":
        assert g["ts"] == TM and g["covered"] == g["ld"], (label, g)
    else:                                   # whole tiles, several per T1 CTA, more T2 chunks than T2 CTAs
        assert g["ts"] == TM and g["tiles"] > n_sms and g["nchunks"] > 128, (label, g)


# ---- inputs and the float64 reference ------------------------------------------------------------------------------------------
class Rms64:
    """The fp32 normaliser moments the kernels read, in float64 (oracle RunningMeanStd.normalize / denormalize without its fp32 casts)."""

    def __init__(self, rms):
        self.mean, self.var, self.eps = rms.mean32.cpu().double(), rms.var32.cpu().double(), rms.eps

    def normalize(self, x):
        return torch.clamp((x - self.mean) / torch.sqrt(self.var + self.eps), -5.0, 5.0)

    def denormalize(self, x):
        return torch.sqrt(self.var + self.eps) * torch.clamp(x, -5.0, 5.0) + self.mean


def make_policy(D, seed):
    pol = PolicyMLP(D, DEV, seed=seed, lr=3e-4, e_clip=E_CLIP, tensor_cores=True)
    assert pol.tensor_cores
    g = torch.Generator().manual_seed(seed)
    pol.params.add_((0.02 * torch.randn(pol.P, generator=g)).to(DEV))      # non-zero biases and log-std
    pol.obs_rms.update((torch.randn((500, D), generator=g) * 2 + 0.3).to(DEV))
    pol.val_rms.load(torch.tensor([0.3]), torch.tensor([2.0]), torch.tensor(50.0))
    return pol


def make_batch(pol, M, seed):
    """A rollout-like minibatch: actions sampled from the policy (float64 forward) plus drift, old log-probs the current ones plus noise,
    old values the current ones plus a little drift, old mu / sigma the current ones.  A sample whose probability ratio or value delta sits
    within rounding distance of a clip boundary flips a whole per-sample term between two TF32 evaluations, which at 10k rows is as large
    as the bars: every log-ratio stays KINK away from log(1 +- e_clip) (a few percent of the samples are clipped), every value delta KINK
    inside +- e_clip.  float32, as the kernels see it; the reference reads the same values."""
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(s, generator=g, dtype=torch.float64)
    obs = (rn(M, pol.D) * 2).float().double()
    mu, value, logstd = P.mlp_forward(pol.params.cpu().double(), Rms64(pol.obs_rms).normalize(obs), pol.D)
    sigma = torch.exp(logstd)
    actions = (mu + sigma * rn(M, 2) + 0.2 * rn(M, 2)).float().double()
    log_ratio = 0.1 * rn(M)
    for c in (math.log(1.0 - E_CLIP), math.log(1.0 + E_CLIP)):
        log_ratio = torch.where((log_ratio - c).abs() < KINK, torch.where(log_ratio >= c, c + KINK, c - KINK), log_ratio)
    b = dict(obs=obs, actions=actions, old_logp_actions=P.neglogp(actions, mu, sigma, logstd) + log_ratio, advantages=rn(M),
             old_values=value + (0.05 * rn(M, 1)).clamp(KINK - E_CLIP, E_CLIP - KINK), returns=rn(M, 1) * 0.5,
             mu=mu + 0.02 * rn(M, 2), sigma=sigma)
    return {k: v.float().contiguous() for k, v in b.items()}


def reference(pol, b):
    """oracle minibatch_loss + autograd in float64: (gradient, statistics, new mu, new sigma)."""
    prm = pol.params.cpu().double().requires_grad_(True)
    loss, st = P.minibatch_loss(prm, {k: v.double() for k, v in b.items()}, pol.D, Rms64(pol.obs_rms), e_clip=E_CLIP)
    loss.backward()
    stats = {k: float(st[k].detach()) for k in STATS if k != "loss"}
    stats["loss"] = float(loss.detach())
    return prm.grad, stats, st["mu"], st["sigma"]


def poison(pol, M):
    """A workspace of exactly the size this minibatch asks for, and the scratch, filled with NaN."""
    need = int(pol.lib.ppo_train_tc_workspace_floats(ctypes.c_int64(M)))
    pol._ws = torch.full((need,), float("nan"), device=DEV)
    pol.scratch.fill_(float("nan"))


def run(pol, b, fn):
    """Calls minibatch_grad / minibatch_step with mu / sigma as the first M rows of longer buffers; returns those buffers."""
    M = b["obs"].shape[0]
    d = {k: v.to(DEV) for k, v in b.items()}
    mu = torch.full((M + TAIL, 2), SENTINEL, device=DEV)
    sg = torch.full((M + TAIL, 2), SENTINEL, device=DEV)
    mu[:M], sg[:M] = d["mu"], d["sigma"]
    fn(d["obs"], d["actions"], d["old_logp_actions"], d["advantages"], d["old_values"].reshape(-1), d["returns"].reshape(-1), mu[:M], sg[:M])
    torch.cuda.synchronize()
    return mu, sg


# ---- checks ------------------------------------------------------------------------------------------------------------------------
def check_gradient(got, want, D, what):
    got = got.cpu().double()
    L = P.param_layout(D)
    bad = [n for n in BLOCKS if not torch.isfinite(got[L[n][0]:L[n][1]]).all()]
    assert not bad, f"{what}: non-finite gradient in {bad}"
    for name in BLOCKS:
        a, b = got[L[name][0]:L[name][1]], want[L[name][0]:L[name][1]]
        scale = float(b.abs().max())
        err = float((a - b).abs().max())
        # TF32 operands + tanh.approx: 2 % of the block's scale, + 5e-5 for the scalar blocks (means of sign-alternating per-sample terms)
        assert err <= 2e-2 * scale + 5e-5, (what, name, err, scale)
        if b.numel() > 2:
            cos = float(torch.nn.functional.cosine_similarity(a, b, dim=0))
            assert cos > 0.999, (what, name, cos)


def check_stats(got, want, what):
    for k in STATS:
        assert math.isfinite(got[k]) and abs(got[k] - want[k]) <= 5e-3 * abs(want[k]) + 2e-4, (what, k, got[k], want[k])


def check_write_back(mu, sg, mu64, sg64, M, what):
    assert_close(mu[:M], mu64, 5e-3, 5e-3, f"{what}: written-back mu")
    assert_close(sg[:M], sg64, 1e-6, 1e-7, f"{what}: written-back sigma")
    assert bool((mu[M:] == SENTINEL).all()) and bool((sg[M:] == SENTINEL).all()), f"{what}: rows >= M of mu / sigma were written"


def check_slabs(pol, M, n_sms, what):
    """The T1 output T2 reads, in the layout of train_setup ((4 H + DP + 16) rows x ld): finite in every column T2 reads, and the padding
    columns of the last tile (samples >= M) of X^T, dz1^T, dz2^T and dz3^T exactly 0, so that they add nothing to the weight gradients."""
    g = geometry(M, n_sms)
    ld, cols = g["ld"], g["nchunks"] * WK
    assert cols <= g["covered"], (what, g)
    DP = 16 if pol.D < 16 else 48
    ws = pol._ws[: (4 * H + DP + 16) * ld].view(4 * H + DP + 16, ld)
    slabs = dict(h1t=ws[0:H], h2t=ws[H:2 * H], dz2t=ws[2 * H:3 * H], dz1t=ws[3 * H:4 * H], xt=ws[4 * H:4 * H + DP],
                 dz3t=ws[4 * H + DP:4 * H + DP + 3])
    for name, s in slabs.items():
        assert bool(torch.isfinite(s[:, :cols]).all()), f"{what}: {name} has non-finite values in the columns T2 reads ({cols} of ld {ld})"
    for name in ("xt", "dz1t", "dz2t", "dz3t"):
        pad = slabs[name][:, M:cols]
        assert bool((pad == 0).all()), f"{what}: {name} columns {M}..{cols} (samples >= M) are not zero"


# ---- the cases -----------------------------------------------------------------------------------------------------------------------
SIZES = ("one", "half_tile", "odd_129", "odd_4800", "lim-127", "lim-64", "lim", "lim+1", "ctl_65", "ctl_200", "ragged", "128x200")
# K = 16 (D = 13) and K = 48 with X / W1 aliased over W2^T (D = 33) at every size; the K-padding edges (bias column last of the first
# 16-wide block at D = 15, first of the second block at D = 16, last of the 48-wide tile at D = 47; D = 1) at one affected size and a control
CASES = [(D, s) for D in (13, 33) for s in SIZES] + [(D, s) for D in (1, 15, 16, 47) for s in ("odd_129", "ctl_200")]


@pytest.mark.parametrize("D,size", CASES)
def test_minibatch_grad_vs_float64(D, size):
    n_sms = sms()
    M = minibatch_size(size, n_sms)
    check_regime(size, M, n_sms)
    pol = make_policy(D, seed=D)
    b = make_batch(pol, M, seed=M)
    want, wstats, mu64, sg64 = reference(pol, b)
    poison(pol, M)
    mu, sg = run(pol, b, pol.minibatch_grad)
    what = f"minibatch_grad D={D} M={M}"
    check_gradient(pol.grads[:pol.P], want, D, what)
    check_stats(pol.stats(), wstats, what)
    check_write_back(mu, sg, mu64, sg64, M, what)
    check_slabs(pol, M, n_sms, what)


@pytest.mark.parametrize("D,size", CASES)
def test_minibatch_step_vs_float64(D, size):
    """The fused step: T1, T2 and one cooperative kernel that reduces the partial gradients into `grads`, clips, applies Adam and the
    adaptive learning rate.  Adam is checked in float64 on the kernel's own gradient, which isolates it from the TF32 noise."""
    n_sms = sms()
    M = minibatch_size(size, n_sms)
    check_regime(size, M, n_sms)
    pol = make_policy(D, seed=D)
    b = make_batch(pol, M, seed=M)
    want, wstats, mu64, sg64 = reference(pol, b)
    p0, lr0 = pol.params.cpu().double(), float(pol.lr)
    poison(pol, M)
    mu, sg = run(pol, b, pol.minibatch_step)
    what = f"minibatch_step D={D} M={M}"
    s = pol.stats()
    assert math.isfinite(s["loss"]), f"{what}: loss {s['loss']} (the tail also reports NaN for a skipped step)"
    g = pol.grads[:pol.P].cpu().double()
    check_gradient(g, want, D, what)
    check_stats(s, wstats, what)
    check_write_back(mu, sg, mu64, sg64, M, what)
    norm64 = float(want.norm())
    assert abs(s["grad_norm"] - norm64) <= 5e-3 * norm64, (what, s["grad_norm"], norm64)
    assert abs(s["grad_norm"] - float(g.norm())) <= 1e-5 * float(g.norm()), (what, s["grad_norm"], float(g.norm()))
    assert s["lr"] == lr0 and int(pol.step) == 1
    new, _, _, _ = P.adam_step(p0, g, torch.zeros_like(g), torch.zeros_like(g), 1, s["lr"])
    got = pol.params.cpu().double()
    assert not torch.equal(got, p0), f"{what}: the parameters did not move"
    assert_close(got, new, 1e-6, 1e-9, f"{what}: params after clip + Adam")
    assert float(pol.lr) == pytest.approx(P.adaptive_lr(s["lr"], s["kl"]), rel=1e-6), (what, float(pol.lr), s["kl"])


@pytest.mark.parametrize("D,size", [(13, "odd_129"), (13, "odd_4800"), (33, "odd_4800")])
def test_minibatch_grad_after_a_larger_minibatch(D, size):
    """No NaN: the stale but finite slabs and slots of an 8192 + 50 row minibatch are what a long training run leaves in the workspace
    and the scratch when a smaller minibatch follows."""
    n_sms = sms()
    M = minibatch_size(size, n_sms)
    check_regime(size, M, n_sms)
    pol = make_policy(D, seed=D)
    big = 8192 + 50
    pol._ws = ws = torch.zeros(int(pol.lib.ppo_train_tc_workspace_floats(ctypes.c_int64(big))), device=DEV)
    pol.scratch.zero_()
    run(pol, make_batch(pol, big, seed=big), pol.minibatch_grad)
    b = make_batch(pol, M, seed=M)
    want, wstats, mu64, sg64 = reference(pol, b)
    mu, sg = run(pol, b, pol.minibatch_grad)
    assert pol._ws is ws                    # the smaller minibatch ran on the same workspace
    what = f"minibatch_grad D={D} M={M} after M={big}"
    check_gradient(pol.grads[:pol.P], want, D, what)
    check_stats(pol.stats(), wstats, what)
    check_write_back(mu, sg, mu64, sg64, M, what)


@pytest.mark.parametrize("D", [1, 15, 16, 47])
def test_forward_at_padding_edges_vs_float64(D):
    """forward_tc_kernel (act / values) at the K-padding edges against oracle policy_inference in float64, with the Philox noise of the
    oracle mirror; the bars of test_gpu_ppo.test_tensor_core_forward_vs_fp32.  Output buffers are views with a sentinel tail."""
    pol = make_policy(D, seed=100 + D)
    prm = pol.params.cpu().double()
    shapes = dict(actions=(2,), neglogpacs=(), values=(1,), mus=(2,), sigmas=(2,))
    for M in (1, 127, 129, 16384 + 77):
        obs = torch.randn((M, D), generator=torch.Generator().manual_seed(M)) * 3
        counter = pol.sample_counter - pol._counter_offset_host
        bufs = {k: torch.full((M + TAIL, *s), SENTINEL, device=DEV) for k, s in shapes.items()}
        out = pol.act(obs.to(DEV), out={k: v[:M] for k, v in bufs.items()})
        eps = P.normal_eps(pol.seed, np.arange(M), counter).double()
        ref = P.policy_inference(prm, obs.double(), D, Rms64(pol.obs_rms), Rms64(pol.val_rms), eps=eps)
        what = f"forward D={D} M={M}"
        assert_close(out["mus"], ref["mus"], 5e-3, 5e-3, f"{what}: mus")
        assert_close(out["values"], ref["values"], 5e-3, 1e-2, f"{what}: values")
        assert_close(out["sigmas"], ref["sigmas"], 1e-6, 1e-7, f"{what}: sigmas")
        assert_close(out["actions"] - out["mus"], ref["actions"] - ref["mus"], 1e-5, 1e-5, f"{what}: sampling noise")
        assert_close(out["neglogpacs"], ref["neglogpacs"], 1e-5, 1e-5, f"{what}: neglogp")
        vals = torch.full((M + TAIL, 1), SENTINEL, device=DEV)
        pol.values(obs.to(DEV), out=vals[:M])
        assert_close(vals[:M], ref["values"], 5e-3, 1e-2, f"{what}: get_values")
        for k, v in list(bufs.items()) + [("values()", vals)]:
            assert bool((v[M:] == SENTINEL).all()), f"{what}: rows >= M of {k} were written"


@pytest.mark.parametrize("n,Tn", [(40, 4), (375, 4)])
def test_loopz_tensor_core_gradient_on_poisoned_workspace(n, Tn):
    """The loopz learner's tensor-core trunk shares train_setup but always runs whole 128-row tiles, so T1 covers every slab column T2
    reads even at ragged minibatches (160 rows would be a half-tile size with an uncovered chunk on the classic path).  Against the
    float64 oracle with the yardstick of test_gpu_loopz.test_tensor_core_gradient_vs_fp32_kernels: every weight matrix within 3x (+5 %)
    of what truncating only the weights to TF32 moves it, measured here in float64 as well."""
    from omniisaacgymenvs_loop_b200.algo.ppo import PPO, module as Mo
    B, D = n * Tn, 33
    g = geometry(B, sms(), tile_rows=TM)
    assert B % TM != 0 and g["nchunks"] * WK == g["covered"] == g["ld"], g
    arch = dict(speed_dim=3, mass_dim=8, mass_latent_dim=8, mass_encoder_shape=[64, 16])
    actor = Mo.Actor(Mo.MLPEncode_wrap([128, 128], "LeakyReLU", D, 2, "Tanh", False, **arch),
                     Mo.SquashedGaussianDiagonalCovariance(2, 0.3, action_scale=1.0), DEV, seed=0)
    critic = Mo.Critic(Mo.MLPEncode_wrap([128, 128], "LeakyReLU", D, 1, **arch), DEV)
    ppo = PPO(actor=actor, critic=critic, num_envs=n, num_transitions_per_env=Tn, device=DEV, mini_batch_sampling="in_order",
              use_cuda_graph=False, tensor_cores=True, num_learning_epochs=1, num_mini_batches=1, learning_rate=0.0, max_grad_norm=1e9)
    assert ppo.tensor_cores
    cfg = Z.LoopzCfg()
    gen = torch.Generator().manual_seed(B)
    rn = lambda *s: torch.randn(s, generator=gen, dtype=torch.float64)
    flat = (ppo.params.cpu().double() + 0.03 * rn(ppo.P)).float()
    ppo.params.copy_(flat)
    # a rollout-like minibatch: old log-probs / values are the networks' own float64 outputs plus a little drift (ratios and value deltas
    # inside the clip ranges)
    obs = rn(B, D).float().double()
    act = torch.tanh(rn(B, 2) * 1.2).float().double()
    pa, std, pc = Z.split(flat.double(), cfg)
    lp0, _ = Z.evaluate(Z.mlp_encode(pa, obs, cfg, True), std, act, cfg)
    v0 = Z.mlp_encode(pc, obs, cfg, False)
    values = (v0 + 0.03 * rn(B, 1)).float().double()
    cols = dict(actor_obs=obs, critic_obs=obs, actions=act, values=values, advantages=rn(B, 1).float().double(),
                returns=(values + 0.5 * rn(B, 1)).float().double(), actions_log_prob=(lp0.unsqueeze(1) + 0.03 * rn(B, 1)).float().double())
    for k, v in cols.items():
        getattr(ppo.storage, k).copy_(v.view(getattr(ppo.storage, k).shape))
    rows = [cols[k] for k in ("actor_obs", "critic_obs", "actions", "values", "advantages", "returns", "actions_log_prob")]
    want, loss, surr, vloss = Z.minibatch_grad(flat.double(), cfg, *rows)
    ft = flat.clone().view(torch.int32)
    ft &= ~0x1fff                                             # weights only, 10-bit mantissa
    trunc, *_ = Z.minibatch_grad(ft.view(torch.float32).double(), cfg, *rows)
    ppo.lib.ppo_loopz_tc_workspace_floats.restype = ctypes.c_int64
    nws = int(ppo.lib.ppo_loopz_tc_workspace_floats(ctypes.byref(ppo._store.net), ctypes.c_int64(B)))
    ppo._tc_ws = (B, torch.full((nws,), float("nan"), device=DEV))
    ppo.scratch.fill_(float("nan"))
    ppo._minibatch(0, B)
    got = ppo.grads[:ppo.P].cpu().double()
    assert torch.isfinite(got).all()
    cos = float(torch.dot(want, got) / (want.norm() * got.norm()))
    assert cos > 0.998, cos
    sizes = [int(np.prod(s)) for out in (2, 1) for s in Z.net_shapes(cfg, out)]
    sizes = sizes[:12] + [2] + sizes[12:]
    off = 0
    for i, sz in enumerate(sizes):
        if sz >= 1024:
            ea, eb, ec = want[off:off + sz], got[off:off + sz], trunc[off:off + sz]
            err_tc, err_tr = float((ea - eb).norm() / ea.norm()), float((ea - ec).norm() / ea.norm())
            assert err_tc <= 3.0 * err_tr + 0.05, (i, err_tc, err_tr)
        off += sz
    s = ppo.minibatch_statistics()
    for k, w in (("loss", loss), ("surrogate", surr), ("value_loss", vloss)):
        assert s[k] == pytest.approx(w, rel=5e-3, abs=5e-3), (k, s[k], w)
