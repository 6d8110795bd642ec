"""The loopz PPO trainer on the C-ABI kernels: observe / step / update with the reference's signatures.

Mirrors `omniisaacgymenvs/algo/ppo/ppo.py:12-325`.  Per minibatch the reference runs two network forwards, the clipped
surrogate / clipped value losses, autograd, `clip_grad_norm_` and Adam (~150 eager launches and two `.item()` syncs); here
it is `ppo_loopz_minibatch_grad_f32` + `ppo_loopz_adam_step_f32` (4 launches, no host sync), and with `in_order` sampling
the whole `_train_step` is replayed from one CUDA graph.  Kept behaviours: advantages standardised over the full batch,
minibatches are contiguous time-major row blocks (`in_order`) or chunks of one permutation per epoch (`shuffle`), an
optimiser step is skipped when its loss is not finite, the mean losses are taken over the valid updates, the learning-rate
schedule only moves when `update_scheduler()` is called (the live script never calls it).
`flat_expert` (the imitation term of a different project's teacher) is not supported: the USV pipeline passes None.

Data-parallel over `world_size` ranks (one process per GPU, `num_envs` envs each, rank r owning global envs [r*num_envs, (r+1)*num_envs)):
the parameters are broadcast from rank 0 at construction, sampling draws the Philox streams of the global env ids, the advantage moments
and every minibatch gradient are summed over the ranks inside the update (rl.peer.PeerLoopzExchange, no host in the loop, capturable),
and Adam sees the mean over all ranks' samples.  With `in_order` sampling the union of the ranks' minibatch k is the one-rank minibatch k
over all envs, so a W-rank update equals the one-rank update over W x num_envs envs up to summation order, with bit-identical
parameters on every rank.  With `shuffle` each rank permutes its own rows (the same generator seed on every rank): parameters stay
identical across ranks, but the minibatches are not those of any one-rank run."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from ... import _lib
from .module import Actor, Critic, _Store, _act, _as_dev
from .storage import RolloutStorage

N_STAT = _lib.ENUMS["PPO_LOOPZ_STAT_COUNT"]
STAT = {k[len("PPO_LOOPZ_STAT_"):].lower(): v for k, v in _lib.ENUMS.items()
        if k.startswith("PPO_LOOPZ_STAT_") and k != "PPO_LOOPZ_STAT_COUNT"}


class PPO:
    def __init__(self, actor: Actor, critic: Critic, num_envs, num_transitions_per_env, num_learning_epochs, num_mini_batches,
                 clip_param=0.2, gamma=0.998, lam=0.95, value_loss_coef=0.5, entropy_coef=0.0, learning_rate=5e-4, max_grad_norm=0.5,
                 use_clipped_value_loss=True, log_dir="run", device="cuda:0", mini_batch_sampling="shuffle", log_intervals=10,
                 flat_expert=None, use_cuda_graph=True, tensor_cores=False, rank=0, world_size=1, group=None, peer=None):
        """`rank`, `world_size`, `group`: data-parallel training (torch.distributed must be initialised when world_size > 1; it is used
        at construction only).  `peer`: the exchange windows to use instead of building a rl.peer.PeerLoopzExchange over `group`
        (one rank of rl.peer.InProcessLoopzExchange); no parameter broadcast then."""
        if flat_expert is not None:
            raise NotImplementedError("flat_expert (imitation term) is not part of the USV pipeline (rlgames_train_loopz.py:93)")
        if mini_batch_sampling not in ("shuffle", "in_order"):
            raise NameError(mini_batch_sampling + " is not a valid sampling method. Use one of the followings: shuffle, order")
        self.lib = _lib.lib()
        self.actor, self.critic = actor, critic
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.UsvLibraryError("the loopz PPO runs on CUDA only (no CPU fallback)")
        # one flat parameter vector for both networks: [actor | std | critic] = the reference optimiser's parameter order (ppo.py:60)
        net = actor._store.net
        store = _Store(net, self.device)
        store.seed, store.counter = actor._store.seed, actor._store.counter - actor._store._offset_host
        store.flat[:store.PA + 2].copy_(actor._store.flat[:store.PA + 2])
        store.flat[store.PA + 2:].copy_(critic._store.flat[store.PA + 2:])
        actor._bind(store)
        critic._bind(store)
        self._store = store
        self.P = store.P
        self.rank, self.world = int(rank), int(world_size)
        if not 0 <= self.rank < self.world:
            raise ValueError(f"rank {rank} outside world_size {world_size}")
        store.row_offset = self.rank * int(num_envs)
        self.peer = None
        if self.world > 1:
            if peer is None:
                import torch.distributed as dist
                from ...rl.peer import PeerLoopzExchange
                dist.broadcast(store.flat, 0, group=group)                    # every rank starts from rank 0's parameters
                peer = PeerLoopzExchange(net, self.device, self.rank, self.world, group)
            if peer.world != self.world or peer.rank != self.rank:
                raise ValueError(f"exchange windows of rank {peer.rank} / {peer.world} for rank {self.rank} / {self.world}")
            self.peer = peer
        f32 = dict(dtype=torch.float32, device=self.device)
        self.params = store.flat
        self.exp_avg, self.exp_avg_sq = torch.zeros(self.P, **f32), torch.zeros(self.P, **f32)
        self.grads = torch.zeros(self.P + N_STAT, **f32)
        self.lib.ppo_loopz_train_scratch_floats.restype = ctypes.c_int64
        self.scratch = torch.empty(int(self.lib.ppo_loopz_train_scratch_floats(ctypes.byref(net))), **f32)
        self.base_lr = float(learning_rate)
        self.lr = torch.full((1,), float(learning_rate), **f32)
        self._sched_epoch = 0
        self.adam_step = torch.zeros(2, dtype=torch.int32, device=self.device)
        self._parity = 0
        self._accum = torch.zeros(3, **f32)

        self.storage = RolloutStorage(num_envs, num_transitions_per_env, [actor.obs_shape[0]], [critic.obs_shape[0]],
                                      actor.action_shape, self.device)
        self.mini_batch_sampling = mini_batch_sampling
        self.batch_sampler = (self.storage.mini_batch_generator_shuffle if mini_batch_sampling == "shuffle"
                              else self.storage.mini_batch_generator_inorder)
        self.rl_coeff = 1
        self.num_transitions_per_env, self.num_envs = int(num_transitions_per_env), int(num_envs)
        self.clip_param, self.num_learning_epochs, self.num_mini_batches = clip_param, int(num_learning_epochs), int(num_mini_batches)
        self.value_loss_coef, self.entropy_coef, self.gamma, self.lam = value_loss_coef, entropy_coef, gamma, lam
        self.max_grad_norm, self.use_clipped_value_loss = max_grad_norm, use_clipped_value_loss
        self.loss_params = _lib.STRUCTS["PpoLoopzLossParams"](clip_param, value_loss_coef, entropy_coef, int(use_clipped_value_loss))
        self.adam_params = _lib.STRUCTS["PpoLoopzAdamParams"](0.9, 0.999, 1e-8, max_grad_norm)
        self.log_dir = log_dir
        self.writer = None                      # the reference logs to TensorBoard; here log() prints and returns the scalars
        self.tot_timesteps, self.tot_time = 0, 0
        self.ep_infos = []
        self.log_intervals = log_intervals
        self.actions = self.actions_log_prob = self.actor_obs = None
        self.fuse_value, self._fused_obs = True, None
        self.flat_expert = None
        # tcgen05 path of the minibatch gradient (TF32 operands; in-order minibatches only); the fp32 SIMT kernels are the numerics reference
        self.tensor_cores = bool(tensor_cores) and mini_batch_sampling == "in_order"
        self._tc_ws = None
        self.use_cuda_graph = bool(use_cuda_graph) and mini_batch_sampling == "in_order"
        self._graph = None
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed(store.seed)
        self.last_stats = {}

    # ---- rollout ------------------------------------------------------------------------------------------------
    def update_rl_coeff(self, coeffs):
        self.rl_coeff = np.clip(coeffs, 0, 1)

    def observe(self, actor_obs):
        """actor.sample(obs); the observation, action and log-prob go straight into the current storage slot."""
        st = self.storage
        if st.step >= st.num_transitions_per_env:
            raise AssertionError("Rollout buffer overflow")
        as_numpy = isinstance(actor_obs, np.ndarray)
        obs_t = _as_dev(actor_obs, self.device)
        s = st.step
        st.actor_obs[s].copy_(obs_t)
        # the USV loop hands the SAME observation to step(value_obs=...) (rlgames_train_loopz.py:1038,1184): evaluate the critic on it in
        # the same launch (grid y = network); step() recognises the object and skips its own critic launch
        fuse = self.fuse_value and not as_numpy and st.critic_obs.shape[2:] == st.actor_obs.shape[2:]
        self._fused_obs = actor_obs if fuse else None
        _act(self._store, st.actor_obs[s], st.actor_obs[s] if fuse else None, None, st.actions[s], st.actions_log_prob[s].view(-1), None,
             st.values[s].view(-1) if fuse else None, self.num_envs, True)
        self.actor_obs = st.actor_obs[s]
        self.actions, self.actions_log_prob = st.actions[s], st.actions_log_prob[s].view(-1)
        return self.actions.cpu().numpy() if as_numpy else self.actions

    def step(self, value_obs, rews, dones, infos, prewritten: bool = False):
        """`prewritten`: storage.rewards[step] / storage.dones[step] were already filled on the device (the fused bookkeeping kernel of
        scripts/train_loopz.py writes them), rews / dones are ignored."""
        st = self.storage
        s = st.step
        if s >= st.num_transitions_per_env:
            raise AssertionError("Rollout buffer overflow")
        if value_obs is not None and value_obs is self._fused_obs:
            st.critic_obs[s].copy_(st.actor_obs[s])                # values[s] was written by observe()
        else:
            st.critic_obs[s].copy_(_as_dev(value_obs, self.device))
            _act(self._store, None, st.critic_obs[s], None, None, None, None, st.values[s].view(-1), self.num_envs, False)
        self._fused_obs = None
        if not prewritten:
            if isinstance(rews, np.ndarray):
                rews = torch.from_numpy(rews)
            if isinstance(dones, np.ndarray):
                dones = torch.from_numpy(dones)
            st.rewards[s].copy_(rews.to(self.device, torch.float32).view(-1, 1))
            st.dones[s].copy_(dones.to(self.device).view(-1, 1))
        st.step += 1
        for info in infos:
            ep_info = info.get("episode")
            if ep_info is not None:
                self.ep_infos.append(ep_info)

    # ---- learning -----------------------------------------------------------------------------------------------
    def update(self, actor_obs, value_obs, log_this_iteration, update):
        last_values = self.critic.predict(value_obs)
        self.storage.compute_returns(last_values, self.gamma, self.lam, peer=self.peer)
        mean_value_loss, mean_surrogate_loss, infos = self._train_step()
        self.storage.clear()
        if log_this_iteration and len(self.ep_infos) > 0:
            self.log({"mean_value_loss": mean_value_loss, "mean_surrogate_loss": mean_surrogate_loss, "ep_infos": self.ep_infos,
                      "it": update})
        self.ep_infos.clear()
        return mean_value_loss, mean_surrogate_loss

    def _minibatch(self, lo: int, hi: int, index=None):
        """One optimiser step on rows [lo, hi) of the flattened storage, or on the rows listed in `index`."""
        M = self._local_grad(lo, hi, index)
        if self.peer is not None:
            rc = self.lib.ppo_loopz_grad_exchange_f32(ctypes.byref(self.peer.comm), ctypes.byref(self._store.net), _lib.ptr(self.grads),
                                                      _lib.ptr(self.peer.seq), _lib.ptr(self.peer.err), _lib.stream())
            _lib.check(rc, "ppo_loopz_grad_exchange_f32")
        rc = self.lib.ppo_loopz_adam_step_f32(_lib.ptr(self.params), _lib.ptr(self.grads), _lib.ptr(self.exp_avg), _lib.ptr(self.exp_avg_sq),
                                              _lib.ptr(self.lr), _lib.ptr(self.adam_step), ctypes.c_int32(self._parity), _lib.ptr(self._accum),
                                              ctypes.c_int64(self.P), ctypes.c_int64(M * self.world), ctypes.byref(self.loss_params),
                                              ctypes.byref(self.adam_params), _lib.stream())
        _lib.check(rc, "ppo_loopz_adam_step_f32")
        self._parity ^= 1

    def _local_grad(self, lo: int, hi: int, index=None) -> int:
        """This rank's minibatch gradient and statistic sums into self.grads; returns the minibatch size."""
        st = self.storage
        ao, co, ac, va, ad, re, lp = st._flat()
        if index is None:
            args, M, idx = [ao[lo:hi], co[lo:hi], ac[lo:hi], lp[lo:hi], ad[lo:hi], va[lo:hi], re[lo:hi]], hi - lo, None
        else:
            args, M, idx = [ao, co, ac, lp, ad, va, re], int(index.numel()), index
        if self.tensor_cores and idx is None:
            if self._tc_ws is None or self._tc_ws[0] < M:
                self.lib.ppo_loopz_tc_workspace_floats.restype = ctypes.c_int64
                nws = int(self.lib.ppo_loopz_tc_workspace_floats(ctypes.byref(self._store.net), ctypes.c_int64(M)))
                if nws < 0:
                    raise NotImplementedError("tensor-core loopz path: obs_dim - mass_dim + 8 must be <= 47")
                self._tc_ws = (M, torch.zeros(nws, dtype=torch.float32, device=self.device))
            rc = self.lib.ppo_loopz_minibatch_grad_tc(_lib.ptr(self.params), ctypes.byref(self._store.net), *[_lib.ptr(a) for a in args],
                                                      ctypes.byref(self.loss_params), _lib.ptr(self.grads), _lib.ptr(self._tc_ws[1]),
                                                      ctypes.c_int64(M), _lib.stream())
            _lib.check(rc, "ppo_loopz_minibatch_grad_tc")
        else:
            rc = self.lib.ppo_loopz_minibatch_grad_f32(_lib.ptr(self.params), ctypes.byref(self._store.net), *[_lib.ptr(a) for a in args],
                                                       _lib.ptr(idx), ctypes.byref(self.loss_params), _lib.ptr(self.grads),
                                                       _lib.ptr(self.scratch), ctypes.c_int64(M), _lib.stream())
            _lib.check(rc, "ppo_loopz_minibatch_grad_f32")
        return M

    def _run_epochs(self):
        batch = self.num_envs * self.num_transitions_per_env
        mb = batch // self.num_mini_batches
        for _ in range(self.num_learning_epochs):
            if self.mini_batch_sampling == "in_order":
                for b in range(self.num_mini_batches):
                    self._minibatch(b * mb, (b + 1) * mb)
            else:
                for idx in self.storage.shuffled_indices(self.num_mini_batches, self._gen):
                    self._minibatch(0, 0, idx.contiguous())

    def _train_step(self):
        self._accum.zero_()
        n_steps = self.num_learning_epochs * self.num_mini_batches
        if self.use_cuda_graph and n_steps % 2 == 0:
            if self._graph is None:
                # warm the kernels (cudaFuncSetAttribute etc.) outside capture on a throw-away copy of the optimiser state
                keep = [t.clone() for t in (self.params, self.exp_avg, self.exp_avg_sq, self.adam_step, self._accum)]
                mb = self.num_envs * self.num_transitions_per_env // self.num_mini_batches
                self._minibatch(0, mb)          # the real minibatch size: every workspace is allocated before the capture
                self._minibatch(0, mb)
                for t, k in zip((self.params, self.exp_avg, self.exp_avg_sq, self.adam_step, self._accum), keep):
                    t.copy_(k)
                torch.cuda.synchronize(self.device)
                g = torch.cuda.CUDAGraph()
                side = torch.cuda.Stream(self.device)
                side.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(side):
                    with torch.cuda.graph(g, stream=side):
                        self._run_epochs()
                torch.cuda.current_stream(self.device).wait_stream(side)
                self._graph = g
            self._graph.replay()
        else:
            self._run_epochs()
        acc = self._accum.tolist()          # the one host read of the update (the reference reads two scalars per minibatch)
        n_valid = acc[2]
        mean_value_loss = acc[0] / n_valid if n_valid > 0 else 0.0
        mean_surrogate_loss = acc[1] / n_valid if n_valid > 0 else 0.0
        self.last_stats = {"num_valid_updates": int(n_valid), "mean_value_loss": mean_value_loss,
                           "mean_surrogate_loss": mean_surrogate_loss}
        return mean_value_loss, mean_surrogate_loss, self.last_stats

    def check_peers(self) -> None:
        """Raises when an exchange with the peer ranks timed out on this rank (one host read; from the failing exchange on, Adam skips
        every step, so ranks cannot silently diverge)."""
        if self.peer is not None:
            self.peer.check()

    def minibatch_statistics(self):
        """Statistics of the LAST minibatch step (means over the minibatch), one host read."""
        g = self.grads[self.P:].tolist()
        return {k: g[v] for k, v in STAT.items()}

    def update_scheduler(self):
        """LambdaLR(0.9998 ** epoch).step()  [ref ppo.py:62-63,323-324]."""
        self._sched_epoch += 1
        self.lr.fill_(self.base_lr * (0.9998 ** self._sched_epoch))

    # ---- checkpoints (the reference's .pt dictionary, rlgames_train_loopz.py:1291-1297) ----------------------------
    def _optimizer_tensors(self):
        """(shape, offset) of every tensor of the flat vector in the reference optimiser's parameter order
        [*actor.parameters(), *critic.parameters()] = actor architecture (12) | std | critic architecture (12)  [ref ppo.py:60]."""
        import math
        inner = lambda a: getattr(a, "architecture", a)          # MLPEncode_wrap -> MLPEncode
        shapes = ([s for _, s in inner(self.actor.architecture)._shapes] + [(self.actor.distribution.dim,)] +
                  [s for _, s in inner(self.critic.architecture)._shapes])
        out, off = [], 0
        for shp in shapes:
            out.append((shp, off))
            off += math.prod(shp)
        if off != self.P:
            raise RuntimeError(f"optimizer layout covers {off} of {self.P} parameters")
        return out

    def optimizer_state_dict(self):
        """torch.optim.Adam.state_dict() layout (what the reference saves as 'optimizer_state_dict', rlgames_train_loopz.py:1295, and feeds
        to ppo.optimizer.load_state_dict, :856): state[i] = {step, exp_avg, exp_avg_sq} per parameter tensor + one param group."""
        import math
        step = float(self.adam_step[self._parity].item())
        state = {}
        for i, (shp, off) in enumerate(self._optimizer_tensors()):
            n = math.prod(shp)
            state[i] = {"step": torch.tensor(step), "exp_avg": self.exp_avg[off:off + n].view(shp).clone(),
                        "exp_avg_sq": self.exp_avg_sq[off:off + n].view(shp).clone()}
        if step == 0:
            state = {}                           # a fresh torch optimiser has no per-parameter state yet
        group = {"lr": float(self.lr.item()), "betas": (0.9, 0.999), "eps": 1e-08, "weight_decay": 0, "amsgrad": False, "maximize": False,
                 "foreach": None, "capturable": False, "differentiable": False, "fused": None, "decoupled_weight_decay": False,
                 "initial_lr": self.base_lr, "params": list(range(len(self._optimizer_tensors())))}
        return {"state": state, "param_groups": [group]}

    def load_optimizer_state_dict(self, sd) -> None:
        import math
        tens = self._optimizer_tensors()
        state = sd.get("state", {})
        if state and len(state) != len(tens):
            raise ValueError(f"optimizer_state_dict holds {len(state)} parameter states, this learner has {len(tens)} tensors")
        step = 0
        for i, (shp, off) in enumerate(tens):
            st = state.get(i, state.get(str(i)))
            if st is None:
                continue
            n = math.prod(shp)
            if tuple(st["exp_avg"].shape) != tuple(shp):
                raise ValueError(f"optimizer state {i}: shape {tuple(st['exp_avg'].shape)} != {tuple(shp)}")
            self.exp_avg[off:off + n].copy_(st["exp_avg"].reshape(-1))
            self.exp_avg_sq[off:off + n].copy_(st["exp_avg_sq"].reshape(-1))
            step = int(float(st["step"]))
        if not state:
            self.exp_avg.zero_()
            self.exp_avg_sq.zero_()
        self.adam_step.fill_(step)
        groups = sd.get("param_groups") or [{}]
        if "lr" in groups[0]:
            self.lr.fill_(float(groups[0]["lr"]))

    def state_dict(self, update: int = 0):
        return {"actor_architecture_state_dict": self.actor.architecture.state_dict(),
                "actor_distribution_state_dict": self.actor.distribution.state_dict(),
                "critic_architecture_state_dict": self.critic.architecture.state_dict(),
                "optimizer_state_dict": self.optimizer_state_dict(),
                "update": int(update)}

    def load_state_dict(self, ckpt):
        self.actor.architecture.load_state_dict(ckpt["actor_architecture_state_dict"])
        if "actor_distribution_state_dict" in ckpt:
            self.actor.distribution.load_state_dict(ckpt["actor_distribution_state_dict"])
        if "critic_architecture_state_dict" in ckpt:
            self.critic.architecture.load_state_dict(ckpt["critic_architecture_state_dict"])
        if "optimizer_state_dict" in ckpt:
            self.load_optimizer_state_dict(ckpt["optimizer_state_dict"])
        elif "optimizer_state" in ckpt:                     # round-1 files of this repo (flat blobs)
            opt = ckpt["optimizer_state"]
            self.exp_avg.copy_(opt["exp_avg"])
            self.exp_avg_sq.copy_(opt["exp_avg_sq"])
            self.adam_step.fill_(int(opt["step"]))
            self.lr.fill_(float(opt["lr"]))
        else:
            import warnings
            warnings.warn("checkpoint carries no optimizer state: Adam restarts from zero moments")
        return int(ckpt.get("update", -1)) + 1 if "update" in ckpt else 0

    def log(self, variables, width=80, pad=28):
        self.tot_timesteps += self.num_transitions_per_env * self.num_envs
        out = {}
        first = variables["ep_infos"][0]
        for key in (list(first.keys()) if isinstance(first, dict) else []):
            vals = []
            for ep in variables["ep_infos"]:
                if isinstance(ep, dict) and key in ep:
                    v = ep[key]
                    v = float(v.float().mean().item()) if torch.is_tensor(v) else float(np.mean(v))
                    if np.isfinite(v):
                        vals.append(v)
            if vals:
                out["Episode/" + str(key)] = float(np.mean(vals))
        out["Loss/value_function"] = variables["mean_value_loss"]
        out["Loss/surrogate"] = variables["mean_surrogate_loss"]
        out["Policy/mean_noise_std"] = float(self.actor.distribution.std.mean().item())
        lines = ["#" * width] + [f"{k + ':':>{pad}} {v:.4f}" for k, v in out.items()]
        print("\n".join(lines))
        return out
