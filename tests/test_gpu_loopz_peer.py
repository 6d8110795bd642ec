"""The loopz learner on several ranks (csrc/ppo_loopz.cu: grad_exchange_kernel, moment_exchange_kernel) on ONE GPU.  The ranks live in
this process (rl.peer.InProcessLoopzExchange: plain device windows, the same kernels and packet protocol) and run one after another:
before a rank's exchange runs, its peers' packets are placed into its window exactly as their kernels would have stored them, so no
kernel ever waits for a peer.  The concurrent run over NVLink, with an all-gathered checksum across ranks: scripts/check_loopz_peer.py."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

from omniisaacgymenvs_loop_b200 import _lib  # noqa: E402
from omniisaacgymenvs_loop_b200.algo.ppo.ppo import N_STAT  # noqa: E402
from omniisaacgymenvs_loop_b200.rl.peer import InProcessLoopzExchange  # noqa: E402
from tests.test_gpu_loopz import build  # noqa: E402

DEV = "cuda:0"
N_EX = _lib.ENUMS["PPO_LOOPZ_STAT_LOG_PROB"] + 1          # statistic sums that travel behind the gradient


def _place(win, world, ecap, seq, src_rank, dst_rank, words):
    """Packets {word, seq} of `src_rank` for entries 0.. into slot [seq & 1][src_rank] of `dst_rank`'s window (int32 view)."""
    base = (((seq & 1) * world + src_rank) * ecap) * 2
    w = win[dst_rank]
    w[base:base + 2 * words.numel():2] = words
    w[base + 1:base + 2 * words.numel():2] = seq


def _exchange(k, net, grads):
    rc = _lib.lib().ppo_loopz_grad_exchange_f32(ctypes.byref(k.comm), ctypes.byref(net), _lib.ptr(grads), _lib.ptr(k.seq), _lib.ptr(k.err),
                                                _lib.stream())
    _lib.check(rc, "ppo_loopz_grad_exchange_f32")


@pytest.mark.parametrize("world", [2, 4])
def test_grad_exchange_packet_protocol(world):
    """Rank 0's exchange with the peers' packets already in its window: rank-order sum (bit-exact against the host), 1/world on the gradient
    only, its own packets stamped into every peer's window, the parity alternating and the sequence counter advancing."""
    _, _, ppo = build(n=64, horizon=8)
    net, P = ppo._store.net, ppo.P
    n = P + N_EX
    ex = InProcessLoopzExchange(net, DEV, world)
    k = ex.ranks[0]
    ecap = int(k.comm.cap) // (2 * world)
    assert ecap >= P + N_STAT
    win = [w.view(torch.int32) for w in ex.windows]
    g = torch.Generator().manual_seed(world)
    for it in range(5):
        seq = it + 1
        vals = [torch.randn(P + N_STAT, generator=g) * (r + 1) for r in range(world)]
        for r in range(1, world):
            _place(win, world, ecap, seq, r, 0, vals[r][:n].to(DEV).view(torch.int32))
        grads = vals[0].to(DEV)
        _exchange(k, net, grads)
        torch.cuda.synchronize()
        assert int(k.err.item()) == 0 and k.seq.tolist() == [seq, 0], k.seq.tolist()
        want = vals[0][:n].clone()
        for r in range(1, world):
            want = want + vals[r][:n]                         # fp32, rank order
        want[:P] *= 1.0 / world                               # the mean gradient; the statistics stay sums
        assert torch.equal(grads[:n].cpu(), want), "rank-order sum"
        assert torch.equal(grads[n:].cpu(), vals[0][n:]), "Adam's outputs are not exchanged"
        for r in range(1, world):                             # rank 0's packets in slot [parity][0] of every peer
            base = ((seq & 1) * world * ecap) * 2
            assert torch.equal(win[r][base:base + 2 * n:2].cpu(), vals[0][:n].view(torch.int32)), "packet payload"
            assert bool((win[r][base + 1:base + 2 * n:2] == seq).all()), "sequence stamp"
            other = (((seq + 1) & 1) * world * ecap) * 2
            assert bool((win[r][other + 1:other + 2 * n:2] == (seq - 1 if seq > 1 else 0)).all()), "the other parity is untouched"


def test_missing_peer_flag_is_sticky_and_skips_the_step():
    """With the error flag already set (a peer went missing earlier) the exchange does not wait, Adam skips the step and check_peers()
    raises."""
    _, _, ref = build(n=64, horizon=8)
    ex = InProcessLoopzExchange(ref._store.net, DEV, 2)
    _, _, ppo = build(n=64, horizon=8, rank=0, world_size=2, peer=ex.ranks[0])
    ppo.check_peers()
    ex.ranks[0].err.fill_(1)
    before = ppo.params.clone()
    ppo._minibatch(0, 64)
    torch.cuda.synchronize()
    assert torch.equal(ppo.params, before) and ppo.adam_step.tolist() == [0, 0] and ex.ranks[0].seq.tolist() == [1, 0]
    with pytest.raises(RuntimeError):
        ppo.check_peers()


def _fill(ppo, g, n, Tn, D=33):
    st = ppo.storage
    obs = torch.randn((Tn, n, D), generator=g)
    st.actor_obs.copy_(obs); st.critic_obs.copy_(obs)
    st.actions.copy_(torch.tanh(torch.randn((Tn, n, 2), generator=g) * 1.2))
    st.rewards.copy_(torch.randn((Tn, n, 1), generator=g))
    st.dones.copy_((torch.rand((Tn, n, 1), generator=g) < 0.05).to(torch.uint8))
    flat_obs = st.actor_obs.view(-1, D)
    (lp0, _), _ = ppo.actor.evaluate(flat_obs, st.actions.view(-1, 2))   # rollout-like: ratios near 1, values near the critic's
    st.actions_log_prob.copy_((lp0 + 0.03 * torch.randn(lp0.shape, generator=g).to(DEV)).view(Tn, n, 1))
    v0 = ppo.critic.predict(flat_obs)
    st.values.copy_((v0 + 0.1 * torch.randn(v0.shape, generator=g).to(DEV)).view(Tn, n, 1))
    st.step = Tn


@pytest.mark.parametrize("tensor_cores", [False, True])
def test_two_ranks_equal_one_rank_over_all_envs(tensor_cores):
    """Two in-process ranks of n envs each against one learner over the 2n envs: the sampled actions (global Philox rows), the advantages
    (moments exchanged), then one full update (4 epochs x 4 in-order minibatches, gradient exchanged every minibatch).  The ranks end
    bit-identical; the one-rank learner differs only by the order of its sums."""
    W, n, Tn = 2, 512, 8
    kw = dict(horizon=Tn, tensor_cores=tensor_cores, seed=7)
    _, _, big = build(n=W * n, **kw)
    net = big._store.net
    ex = InProcessLoopzExchange(net, DEV, W)
    ranks = [build(n=n, rank=r, world_size=W, peer=ex.ranks[r], **kw)[2] for r in range(W)]
    for p in ranks:
        p.params.copy_(big.params)
    # sampling: rank r draws the rows of the global envs [r n, (r + 1) n)
    obs0 = torch.randn((W * n, 33), device=DEV)
    a_big = big.observe(obs0).clone()
    for r, p in enumerate(ranks):
        assert torch.equal(p.observe(obs0[r * n:(r + 1) * n].contiguous()), a_big[r * n:(r + 1) * n]), "global Philox rows"
    g = torch.Generator().manual_seed(3)
    _fill(big, g, W * n, Tn)
    for r, p in enumerate(ranks):
        for name in ("actor_obs", "critic_obs", "actions", "rewards", "dones", "actions_log_prob", "values"):
            getattr(p.storage, name).copy_(getattr(big.storage, name)[:, r * n:(r + 1) * n])
        p.storage.step = Tn
    lv = torch.randn(W * n, generator=g).to(DEV)
    win = [w.view(torch.int32) for w in ex.windows]
    ecap = int(ex.ranks[0].comm.cap) // (2 * W)

    def next_seq():
        s = [p.peer.seq.tolist() for p in ranks]
        assert all(x == s[0] for x in s) and s[0][1] == 0
        return s[0][0] + 1

    # ---- advantages: each rank's local moments (a world-1 exchange leaves them in the scratch), placed, then each rank's real call
    solo = InProcessLoopzExchange(net, DEV, 1).ranks[0]
    moments = []
    for r, p in enumerate(ranks):
        p.storage.compute_returns(lv[r * n:(r + 1) * n], big.gamma, big.lam, peer=solo)
        moments.append(p.storage._scratch[:2].clone())
    seq = next_seq()
    for r in range(W):
        for q in range(W):
            if q != r:
                _place(win, W, ecap, seq, r, q, moments[r].view(torch.int32))
    for r, p in enumerate(ranks):
        p.storage.compute_returns(lv[r * n:(r + 1) * n], big.gamma, big.lam, peer=p.peer)
    big.storage.compute_returns(lv, big.gamma, big.lam)
    torch.cuda.synchronize()
    adv = torch.cat([p.storage.advantages for p in ranks], 1)
    assert torch.equal(torch.cat([p.storage.returns for p in ranks], 1), big.storage.returns)
    # the moments are fp64 sums in another order: the mean / std agree to ~1e-16, the fp32 advantages to their last bit
    assert float((adv - big.storage.advantages).abs().max()) <= 1e-6 * float(big.storage.advantages.abs().max())
    for r, p in enumerate(ranks):                         # both ranks standardised with the same bits
        assert p.storage._scratch[:2].tolist() == ranks[0].storage._scratch[:2].tolist()
    for r, p in enumerate(ranks):                         # the update below starts from the one-rank advantages
        p.storage.advantages.copy_(big.storage.advantages[:, r * n:(r + 1) * n])

    # ---- one update, minibatch by minibatch
    mb, mb_big = n * Tn // 4, W * n * Tn // 4
    big._accum.zero_()
    for p in ranks:
        p._accum.zero_()
    first = None
    for ep in range(4):
        for b in range(4):
            local = []
            for p in ranks:
                p._local_grad(b * mb, (b + 1) * mb)
                local.append(p.grads[:p.P + N_EX].clone())
            seq = next_seq()
            for r in range(W):
                for q in range(W):
                    if q != r:
                        _place(win, W, ecap, seq, r, q, local[r].view(torch.int32))
            for p in ranks:
                p._minibatch(b * mb, (b + 1) * mb)
            big._minibatch(b * mb_big, (b + 1) * mb_big)
            if ep == 0 and b == 0:
                first = float((ranks[0].params - big.params).abs().max())
    torch.cuda.synchronize()
    for p in ranks:
        p.check_peers()
    a, b = ranks
    for name in ("params", "exp_avg", "exp_avg_sq", "adam_step", "_accum"):
        assert torch.equal(getattr(a, name), getattr(b, name)), f"ranks differ in {name}"
    assert a.adam_step.tolist() == big.adam_step.tolist()
    # summation order is all that differs from the one-rank learner: the gradient sums of the two half minibatches are added across
    # ranks, not inside one reduction, which moves the gradient in its last bits and the parameters by a few ulp of their scale
    scale = float(big.params.abs().max())
    err = float((a.params - big.params).abs().max())
    assert first <= 1e-6 * scale, (first, scale)
    if not tensor_cores:
        assert err <= 1e-6 * scale, (err, scale)
    else:
        # on the tensor cores the weights are TF32 operands: once a parameter differs in its last bit, a TF32 rounding boundary between the
        # two values changes that operand by 2^-11 relative, the gradients then agree to ~1e-4 of their scale, and a gradient entry near
        # zero can change sign, so Adam's normalised step moves it by up to lr the other way.  Measured on a B200: 0.99 lr after 16 steps.
        assert err <= 2 * float(big.lr), (err, float(big.lr))


def test_world_one_is_the_single_rank_learner():
    """PPO(rank=0, world_size=1) builds no exchange, launches exactly the kernels of a PPO built without the new arguments, and updates
    to the same bits (eager and captured update)."""
    for graph in (False, True):
        _, _, a = build(n=256, horizon=8, graph=graph)
        _, _, b = build(n=256, horizon=8, graph=graph, rank=0, world_size=1)
        assert b.peer is None and b._store.row_offset == 0
        b.params.copy_(a.params)
        g = torch.Generator().manual_seed(5)
        _fill(a, g, 256, 8)
        for name in ("actor_obs", "critic_obs", "actions", "rewards", "dones", "actions_log_prob", "values"):
            getattr(b.storage, name).copy_(getattr(a.storage, name))
        b.storage.step = 8
        obs = torch.randn((256, 33), device=DEV)
        launches = []
        for p in (a, b):
            p.update(actor_obs=obs, value_obs=obs, log_this_iteration=False, update=0)
            torch.cuda.synchronize()
            c0 = _lib.launch_count()
            p.storage.step = 8
            p.update(actor_obs=obs, value_obs=obs, log_this_iteration=False, update=1)
            torch.cuda.synchronize()
            launches.append(_lib.launch_count() - c0)
        assert launches[0] == launches[1], launches
        for name in ("params", "exp_avg", "exp_avg_sq", "adam_step"):
            assert torch.equal(getattr(a, name), getattr(b, name)), name
        assert torch.equal(a.observe(obs), b.observe(obs))
