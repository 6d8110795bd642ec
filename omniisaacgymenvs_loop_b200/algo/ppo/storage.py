"""RolloutStorage of the loopz PPO: device-resident [T, N, ...] buffers, GAE + advantage standardisation in one C-ABI call.

Mirrors `omniisaacgymenvs/algo/ppo/storage.py:45-148` (attribute names, `add_transitions`, `compute_returns`, the two
minibatch generators).  `add_transitions` accepts numpy arrays (the reference's contract) or CUDA tensors (no host trip)."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from ... import _lib


def _dev(x, device, dtype=torch.float32) -> torch.Tensor:
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(x)
    return x.to(device=device, dtype=dtype)


class RolloutStorage:
    def __init__(self, num_envs, num_transitions_per_env, actor_obs_shape, critic_obs_shape, actions_shape, device):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.UsvLibraryError("RolloutStorage lives on a CUDA device (no CPU fallback)")
        T, N = int(num_transitions_per_env), int(num_envs)
        f32 = dict(dtype=torch.float32, device=self.device)
        self.actor_obs = torch.zeros(T, N, *actor_obs_shape, **f32)
        self.critic_obs = torch.zeros(T, N, *critic_obs_shape, **f32)
        self.rewards = torch.zeros(T, N, 1, **f32)
        self.actions = torch.zeros(T, N, *actions_shape, **f32)
        self.dones = torch.zeros(T, N, 1, dtype=torch.uint8, device=self.device)
        self.actions_log_prob = torch.zeros(T, N, 1, **f32)
        self.values = torch.zeros(T, N, 1, **f32)
        self.returns = torch.zeros(T, N, 1, **f32)
        self.advantages = torch.zeros(T, N, 1, **f32)
        self.num_transitions_per_env = T
        self.num_envs = N
        self.step = 0
        L = _lib.lib()
        L.ppo_loopz_returns_scratch_bytes.restype = ctypes.c_int64
        self._scratch = torch.empty(int(L.ppo_loopz_returns_scratch_bytes()) // 8, dtype=torch.float64, device=self.device)

    def add_transitions(self, actor_obs, critic_obs, actions, rewards, dones, values, actions_log_prob):
        if self.step >= self.num_transitions_per_env:
            raise AssertionError("Rollout buffer overflow")
        s = self.step
        # non-finite entries are zeroed by the kernels that read these buffers (the reference does it here, storage.py:70-78)
        self.critic_obs[s].copy_(_dev(critic_obs, self.device))
        self.actor_obs[s].copy_(_dev(actor_obs, self.device))
        self.actions[s].copy_(_dev(actions, self.device))
        self.rewards[s].copy_(_dev(rewards, self.device).view(-1, 1))
        self.dones[s].copy_(_dev(dones, self.device, torch.uint8).view(-1, 1))
        self.values[s].copy_(_dev(values, self.device).view(-1, 1))
        self.actions_log_prob[s].copy_(_dev(actions_log_prob, self.device).view(-1, 1))
        self.step += 1

    def clear(self):
        self.step = 0

    def compute_returns(self, last_values, gamma, lam, peer=None):
        """`peer` (a rl.peer.PeerLoopzExchange of world > 1): this storage is one rank's shard, the advantages are standardised over
        the batch of all ranks."""
        last_values = _dev(last_values, self.device).reshape(-1).contiguous()
        args = [_lib.ptr(self.rewards), _lib.ptr(self.values), _lib.ptr(self.dones), _lib.ptr(last_values), ctypes.c_float(gamma),
                ctypes.c_float(lam), _lib.ptr(self.returns), _lib.ptr(self.advantages), _lib.ptr(self._scratch),
                ctypes.c_int32(self.num_transitions_per_env), ctypes.c_int64(self.num_envs)]
        if peer is not None:
            rc = _lib.lib().ppo_loopz_returns_peer_f32(*args, ctypes.byref(peer.comm), _lib.ptr(peer.seq), _lib.ptr(peer.err), _lib.stream())
            _lib.check(rc, "ppo_loopz_returns_peer_f32")
            return
        rc = _lib.lib().ppo_loopz_returns_f32(*args, _lib.stream())
        _lib.check(rc, "ppo_loopz_returns_f32")

    def _flat(self):
        return (self.actor_obs.view(-1, *self.actor_obs.size()[2:]), self.critic_obs.view(-1, *self.critic_obs.size()[2:]),
                self.actions.view(-1, self.actions.size(-1)), self.values.view(-1, 1), self.advantages.view(-1, 1),
                self.returns.view(-1, 1), self.actions_log_prob.view(-1, 1))

    def shuffled_indices(self, num_mini_batches, generator=None):
        """One permutation of the batch cut into minibatches, remainder dropped (BatchSampler(SubsetRandomSampler), storage.py:130)."""
        batch_size = self.num_envs * self.num_transitions_per_env
        mb = batch_size // num_mini_batches
        perm = torch.randperm(batch_size, device=self.device, generator=generator)
        return [perm[i * mb:(i + 1) * mb] for i in range(batch_size // mb)] if mb > 0 else []

    def mini_batch_generator_shuffle(self, num_mini_batches):
        for indices in self.shuffled_indices(num_mini_batches):
            yield tuple(t[indices] for t in self._flat())

    def mini_batch_generator_inorder(self, num_mini_batches):
        batch_size = self.num_envs * self.num_transitions_per_env
        mb = batch_size // num_mini_batches
        for b in range(num_mini_batches):
            yield tuple(t[b * mb:(b + 1) * mb] for t in self._flat())


class ObsStorage:
    """Supervised (observation, expert target) buffer of the DAgger / SysID trainers  [ref: omniisaacgymenvs/algo/ppo/storage.py:4-42]:
    `[T, N, ...]` tensors on `device`, time-major flattening, in-order minibatches = contiguous row blocks (views, no copy),
    shuffled minibatches from one `torch.randperm` (the reference draws them with `BatchSampler(SubsetRandomSampler(...))`,
    `drop_last=True`).  `add_obs` takes numpy (the reference's contract) or tensors already on the device.  A plain tensor container:
    no kernel behind it, so any device is accepted."""

    def __init__(self, num_envs, num_transitions_per_env, obs_shape, action_shape, device):
        self.device = torch.device(device)
        self.obs = torch.zeros(num_transitions_per_env, num_envs, *obs_shape, dtype=torch.float32, device=self.device)
        self.expert = torch.zeros(num_transitions_per_env, num_envs, *action_shape, dtype=torch.float32, device=self.device)
        self.num_envs = int(num_envs)
        self.num_transitions_per_env = int(num_transitions_per_env)
        self.step = 0

    def add_obs(self, obs, expert_action):
        if self.step >= self.num_transitions_per_env:
            raise AssertionError("Rollout buffer overflow")
        self.obs[self.step].copy_(_dev(obs, self.device))
        self.expert[self.step].copy_(_dev(expert_action, self.device))
        self.step += 1

    def clear(self):
        self.step = 0

    def _flat(self):
        return self.obs.view(-1, *self.obs.size()[2:]), self.expert.view(-1, *self.expert.size()[2:])

    def mini_batch_generator_inorder(self, num_mini_batches):
        obs, expert = self._flat()
        mb = (self.num_envs * self.num_transitions_per_env) // num_mini_batches
        for b in range(num_mini_batches):
            yield obs[b * mb:(b + 1) * mb], expert[b * mb:(b + 1) * mb]

    def mini_batch_generator_shuffle(self, num_mini_batches, generator=None):
        obs, expert = self._flat()
        batch = self.num_envs * self.num_transitions_per_env
        mb = batch // num_mini_batches
        perm = torch.randperm(batch, generator=generator).to(self.device)
        for b in range(batch // mb):                                  # drop_last=True
            idx = perm[b * mb:(b + 1) * mb]
            yield obs[idx], expert[idx]
