"""CPU suite, world_size 2 over gloo, on the loopz oracle: what the data-parallel loopz learner (PPO(rank, world_size), the exchanges of
csrc/ppo_loopz.cu) computes.  Each rank takes its shard of one seeded rollout over W x n envs, standardises its advantages with the
moments summed over the ranks, and steps Adam with the per-minibatch gradient sums added over the ranks and scaled by 1/(W M): after a
full update (4 epochs x 4 in-order minibatches) its parameters equal the oracle's one-rank update over all W x n envs.  Also the start-up
parameter broadcast and the episode-statistics reduction of scripts/train_loopz.py."""
import os
import socket
import types

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import loopz_oracle as Z

W, N, T, D = 2, 24, 8, 33


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rollout():
    """One seeded rollout over W x N envs ([T, W N, k] tensors), the parameters it was drawn with, the last values."""
    cfg = Z.LoopzCfg()
    g = torch.Generator().manual_seed(11)
    P = sum(int(torch.tensor(s).prod()) for out in (2, 1) for s in Z.net_shapes(cfg, out)) + 2
    flat = torch.randn(P, generator=g) * 0.1
    _, std, _ = Z.split(flat, cfg)
    std.fill_(0.3)
    pa, std, pc = Z.split(flat, cfg)
    obs = torch.randn((T, W * N, D), generator=g)
    rows = obs.reshape(-1, D)
    actions = torch.tanh(torch.randn((T * W * N, 2), generator=g) * 1.2)
    lp, _ = Z.evaluate(Z.mlp_encode(pa, rows, cfg, True), std, actions, cfg)
    values = Z.mlp_encode(pc, rows, cfg, False) + 0.1 * torch.randn((T * W * N, 1), generator=g)
    st = {"actor_obs": obs, "critic_obs": obs, "actions": actions.view(T, W * N, 2),
          "actions_log_prob": (lp + 0.03 * torch.randn(lp.shape, generator=g)).view(T, W * N, 1), "values": values.view(T, W * N, 1),
          "rewards": torch.randn((T, W * N, 1), generator=g), "dones": (torch.rand((T, W * N, 1), generator=g) < 0.05).to(torch.uint8)}
    return cfg, flat, st, torch.randn((W * N, 1), generator=g)


def _worker(rank, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(W))
    dist.init_process_group("gloo", rank=rank, world_size=W)
    torch.set_num_threads(1)
    try:
        cfg, flat0, st, lv = _rollout()
        # start-up: every rank takes rank 0's parameters
        flat = flat0.clone() if rank == 0 else torch.zeros_like(flat0)
        dist.broadcast(flat, 0)
        sh = {k: v[:, rank * N:(rank + 1) * N] for k, v in st.items()}
        # advantages: GAE on the shard, standardised with the fp64 moments summed over the ranks (total W T N, unbiased std)
        returns, _ = Z.compute_returns(sh["rewards"], sh["values"], sh["dones"], lv[rank * N:(rank + 1) * N], cfg.gamma, cfg.lam)
        a = returns - sh["values"]
        mom = torch.stack([a.double().sum(), (a.double() ** 2).sum()])
        dist.all_reduce(mom)
        total = W * T * N
        mean = mom[0] / total
        sd = torch.sqrt((mom[1] - mom[0] * mean) / (total - 1))
        sh["advantages"] = (a - mean.float()) / (sd.float() + 1e-8)
        sh["returns"] = returns
        # the update: per minibatch, local gradient SUMS added over the ranks, then 1/(W M) = the mean over the global minibatch
        cols = [sh[k].reshape(-1, sh[k].shape[-1]) for k in ("actor_obs", "critic_obs", "actions", "values", "advantages", "returns",
                                                              "actions_log_prob")]
        opt = Z.Adam(flat.numel(), cfg.learning_rate)
        M = T * N // 4
        for _ in range(4):
            for b in range(4):
                sel = slice(b * M, (b + 1) * M)
                grad, loss, _, _ = Z.minibatch_grad(flat, cfg, *[c[sel] for c in cols])
                span = torch.cat([grad * M, torch.tensor([loss * M])])
                dist.all_reduce(span)
                span /= W * M
                if torch.isfinite(span[-1]):
                    opt.step(flat, span[:-1], cfg.max_grad_norm)
        # the log line: finished-episode sums (return, length, count) of all ranks
        from scripts.train_loopz import LoopzRunner
        fin = torch.tensor([10.0 * (rank + 1), 100.0 * (rank + 1), 2.0 * (rank + 1)], dtype=torch.float64)
        runner = types.SimpleNamespace(fin=fin, ppo=types.SimpleNamespace(world=W))
        stats = LoopzRunner.pop_episode_stats(runner)
        q.put((rank, flat0 if rank == 0 else None, flat, opt.t, stats, float(fin.abs().sum())))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_two_rank_update_equals_one_rank_update_over_all_envs():
    port = _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, port, q)) for r in range(W)]
    for p in procs:
        p.start()
    out = sorted((q.get(timeout=300) for _ in range(W)), key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    cfg, flat0, st, lv = _rollout()
    assert torch.equal(out[0][1], flat0)
    # one rank over all W x N envs
    st["returns"], st["advantages"] = Z.compute_returns(st["rewards"], st["values"], st["dones"], lv, cfg.gamma, cfg.lam)
    flat = flat0.clone()
    opt = Z.Adam(flat.numel(), cfg.learning_rate)
    Z.train_step(flat, cfg, st, 4, 4, opt)
    for rank, _, got, steps, stats, fin_left in out:
        assert steps == opt.t == 16
        # summation order (over ranks vs inside one minibatch, fp64 moments vs torch.std) is all that differs
        assert float((got - flat).abs().max()) <= 2e-6, (rank, float((got - flat).abs().max()))
        assert stats == (5.0, 6) and fin_left == 0.0      # (10 + 20) / (2 + 4) over both ranks, the sums cleared
    assert torch.equal(out[0][2], out[1][2])              # the ranks agree bit for bit
