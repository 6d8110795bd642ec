"""USV SysID distillation (the DAgger stack's USV path) on the C-ABI kernels of csrc/dagger_sysid.cu
[ref: omniisaacgymenvs/algo/ppo/dagger.py:13-196 -- USVSysIDAgent, USVSysIDTrainer].

  teacher latent   z* = mass_encoder(priv_tail)                (frozen; `MLPEncode.mass_encoder`, dagger_mlp_forward_f32)
  student latent   z^ = id_encoder(history_flat)               (`StateHistoryEncoder`, dagger_history_encoder_forward_f32)
  action           a  = frozen_action_head([obs_nonpriv, z^])  (frozen; `MLPEncode.action_mlp`)
  update           4 epochs x 4 in-order minibatches of  MSE(z^, z*) -> Adam(5e-4), StepLR(200, 0.1) once per update
                   (dagger_sysid_minibatch_step_f32: forward + backward + Adam in two launches per minibatch, no host sync inside an update)
  distillation     USVSysIDDistiller: the same update, collected on the fused student step into a frame store (dagger_sysid_collect_f32,
                   one launch per control step); the training and forward kernels rebuild each window from the store
  deployment       USVSysIDStudentPolicy: history ring + z^ + action head in one launch per control step (dagger_student_act_f32),
                   loaded from the file scripts/dagger_usv_sysid_loopz.py --save writes (student_checkpoint)

Same class / method surface as the reference; numpy in -> numpy out where the reference does that, CUDA tensors stay on the device."""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from ... import _lib
from .module import E1, E2, H, FlatMLP, MLPEncode, StateHistoryEncoder
from .storage import ObsStorage

FILL_MODES = ("zeros", "repeat")
# what a student checkpoint records beside the trainer's state and the teacher's PPO state (scripts/dagger_usv_sysid_loopz.py --save)
STUDENT_META = {"history_len": int, "priv_dim": int, "obs_nonpriv_dim": int, "latent_dim": int, "fill_history_on_reset": str, "seed": int}


class USVSysIDAgent:
    def __init__(self, *, teacher_mass_encoder, id_encoder: StateHistoryEncoder, frozen_action_head, history_len: int, obs_nonpriv_dim: int,
                 device: str) -> None:
        self.teacher_mass_encoder, self.id_encoder, self.frozen_action_head = teacher_mass_encoder, id_encoder, frozen_action_head
        self.history_len, self.obs_nonpriv_dim = int(history_len), int(obs_nonpriv_dim)
        self.history_dim = self.history_len * self.obs_nonpriv_dim
        self.device = torch.device(device)
        if id_encoder.tsteps != self.history_len or id_encoder.input_size != self.obs_nonpriv_dim:
            raise ValueError("id_encoder was built for another history shape")

    def set_itr(self, _itr) -> None:
        return

    def get_history_encoding(self, sysid_obs_torch: torch.Tensor) -> torch.Tensor:
        # sysid_obs = [history_flat | current non-privileged obs]: the kernel reads the history columns of the wide rows in place
        return self.id_encoder(sysid_obs_torch)

    def evaluate(self, sysid_obs_torch: torch.Tensor) -> torch.Tensor:
        zhat = self.get_history_encoding(sysid_obs_torch)
        cur = sysid_obs_torch[:, self.history_dim:self.history_dim + self.obs_nonpriv_dim]
        return self.frozen_action_head(torch.cat([cur.to(zhat.device, torch.float32), zhat], dim=1))

    def get_student_action(self, sysid_obs_torch: torch.Tensor) -> torch.Tensor:
        return self.evaluate(sysid_obs_torch)

    def teacher_latent(self, priv_tail_torch: torch.Tensor) -> torch.Tensor:
        return self.teacher_mass_encoder(priv_tail_torch)


class USVSysIDTrainer:
    """MSE(id_encoder(history), mass_encoder(priv tail)) with Adam + StepLR(200, 0.1), in-order minibatches of the time-major storage."""

    def __init__(self, *, actor: USVSysIDAgent, num_envs: int, num_transitions_per_env: int, history_dim: int, latent_dim: int,
                 num_learning_epochs: int = 4, num_mini_batches: int = 4, device: str, learning_rate: float = 5e-4) -> None:
        self.actor, self.device = actor, torch.device(device)
        self.history_dim, self.latent_dim = int(history_dim), int(latent_dim)
        enc = actor.id_encoder
        if self.history_dim != enc.tsteps * enc.input_size or self.latent_dim != enc.output_size:
            raise ValueError("history_dim / latent_dim do not match the id_encoder")
        self.storage = ObsStorage(int(num_envs), int(num_transitions_per_env), [self.history_dim], [self.latent_dim], self.device)
        self.num_transitions_per_env, self.num_envs = int(num_transitions_per_env), int(num_envs)
        self.num_learning_epochs, self.num_mini_batches = int(num_learning_epochs), int(num_mini_batches)
        self.itr = 0
        self.base_lr = float(learning_rate)
        f32 = dict(dtype=torch.float32, device=self.device)
        P = enc.flat.numel()
        self.exp_avg, self.exp_avg_sq = torch.zeros(P, **f32), torch.zeros(P, **f32)
        self.grads = torch.zeros(P + 1, **f32)
        L = _lib.lib()
        self.scratch = torch.empty(int(L.dagger_train_scratch_floats(ctypes.c_int32(enc.input_size), ctypes.c_int32(enc.tsteps),
                                                                     ctypes.c_int32(enc.output_size))), **f32)
        self.lr = torch.full((1,), self.base_lr, **f32)
        self.adam_step = torch.zeros(2, dtype=torch.int32, device=self.device)
        self._parity = 0
        self._mse = torch.zeros(1, **f32)

    # ---- rollout side ------------------------------------------------------------------------------------------------------
    def observe(self, sysid_obs):
        """Student action for the wrapper's sysid_obs; numpy in -> numpy out (the reference's contract), CUDA tensor in -> CUDA tensor out."""
        as_numpy = isinstance(sysid_obs, np.ndarray)
        obs = torch.from_numpy(sysid_obs).to(self.device) if as_numpy else sysid_obs
        act = self.actor.get_student_action(obs)
        return act.cpu().numpy() if as_numpy else act

    def step(self, sysid_obs, priv_tail_torch: torch.Tensor) -> None:
        """Stores one transition's supervision pair: history_flat and the teacher latent z*."""
        z_star = self.actor.teacher_latent(priv_tail_torch.to(self.device, dtype=torch.float32))[:, :self.latent_dim]
        hist = sysid_obs[:, :self.history_dim]
        self.storage.add_obs(hist.astype(np.float32, copy=False) if isinstance(hist, np.ndarray) else hist, z_star)

    # ---- update --------------------------------------------------------------------------------------------------------------
    def _minibatch(self, hist: torch.Tensor, zstar: torch.Tensor) -> None:
        enc = self.actor.id_encoder
        rc = _lib.lib().dagger_sysid_minibatch_step_f32(
            _lib.ptr(enc.flat), _lib.ptr(hist), ctypes.c_int64(hist.shape[1]), _lib.ptr(zstar), ctypes.c_int32(enc.input_size),
            ctypes.c_int32(enc.tsteps), ctypes.c_int32(enc.output_size), _lib.ptr(self.grads), _lib.ptr(self.scratch), _lib.ptr(self.exp_avg),
            _lib.ptr(self.exp_avg_sq), _lib.ptr(self.lr), _lib.ptr(self.adam_step), ctypes.c_int32(self._parity), _lib.ptr(self._mse),
            ctypes.c_int64(hist.shape[0]), _lib.stream())
        _lib.check(rc, "dagger_sysid_minibatch_step_f32")
        self._parity ^= 1

    def _run_epochs(self, minibatch) -> float:
        """num_learning_epochs x the in-order minibatches of the time-major batch (rows [b * mb, (b + 1) * mb)): minibatch(row0, mb)
        launches one training step each; then StepLR.  -> the last epoch's mean minibatch loss: the update's one host read."""
        self.itr += 1
        self.actor.set_itr(self.itr)
        mb = (self.num_envs * self.num_transitions_per_env) // self.num_mini_batches
        for _epoch in range(self.num_learning_epochs):
            self._mse.zero_()
            for b in range(self.num_mini_batches):
                minibatch(b * mb, mb)
        avg = float(self._mse.item()) / max(1, self.num_mini_batches)
        self.lr.fill_(self.base_lr * (0.1 ** (self.itr // 200)))    # scheduler.step(): StepLR(step_size=200, gamma=0.1)
        return avg

    def _train_step(self) -> float:
        hist, zstar = self.storage._flat()                              # the views mini_batch_generator_inorder slices
        return self._run_epochs(lambda r0, mb: self._minibatch(hist[r0:r0 + mb], zstar[r0:r0 + mb]))

    def update(self) -> dict:
        mse = self._train_step()
        obs_all = self.storage.obs.view(-1, self.history_dim)
        zstar_all = self.storage.expert.view(-1, self.latent_dim)
        metrics = latent_metrics(mse, self.actor.id_encoder(obs_all), zstar_all)
        self.storage.clear()
        return metrics

    # ---- checkpoints: the student's weights + Adam state ----------------------------------------------------------------------------
    def state_dict(self) -> dict:
        return {"id_encoder_state_dict": self.actor.id_encoder.state_dict(), "exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(),
                "step": int(self.adam_step[self._parity].item()), "itr": self.itr}

    def load_state_dict(self, sd: dict) -> None:
        self.actor.id_encoder.load_state_dict(sd["id_encoder_state_dict"])
        if "exp_avg" in sd:
            self.exp_avg.copy_(sd["exp_avg"]); self.exp_avg_sq.copy_(sd["exp_avg_sq"])
            self.adam_step.fill_(int(sd.get("step", 0)))
        self.itr = int(sd.get("itr", 0))
        self.lr.fill_(self.base_lr * (0.1 ** (self.itr // 200)))


def latent_metrics(mse: float, zhat_all: torch.Tensor, zstar_all: torch.Tensor) -> dict:
    """USVSysIDTrainer.update()'s dict: the update's mse, then the R^2 / variance guardrails of the collected batch
    [ref: dagger.py:150-176], a few reductions over (B, latent) tensors once per update."""
    metrics = {"mse": mse}
    metrics["zstar_var_mean"] = float(torch.var(zstar_all, dim=0, unbiased=False).mean())
    metrics["zhat_var_mean"] = float(torch.var(zhat_all, dim=0, unbiased=False).mean())
    sse = torch.sum((zhat_all - zstar_all) ** 2, dim=0)
    sst = torch.sum((zstar_all - zstar_all.mean(dim=0, keepdim=True)) ** 2, dim=0)
    r2 = (1.0 - sse / (sst + 1e-8)).tolist()
    for i in range(zstar_all.shape[1]):
        metrics[f"r2_dim{i}"] = r2[i]
    metrics["r2_total"] = float(1.0 - sse.sum() / (sst.sum() + 1e-8))
    return metrics


def _mlp_args(mlp: FlatMLP) -> list:
    """A FlatMLP as the C ABI's (params, layers, dims, weight offsets, bias offsets, last activation)."""
    nl, I32 = len(mlp.layers), ctypes.c_int32
    return [_lib.ptr(mlp._flat()), I32(nl), (I32 * (nl + 1))(*mlp.dims), (I32 * nl)(*[l[0] for l in mlp.layers]),
            (I32 * nl)(*[l[1] for l in mlp.layers]), I32(mlp.last_activation)]


# ---- deployment: save the distilled student, play it closed-loop ------------------------------------------------------------------------
def student_meta(meta: dict) -> dict:
    """The checkpoint's `meta` entry, checked against STUDENT_META (every key present, each of its type, a known fill mode)."""
    missing = [k for k in STUDENT_META if k not in meta]
    if missing:
        raise KeyError(f"student checkpoint meta lacks {missing}")
    out = {k: t(meta[k]) for k, t in STUDENT_META.items()}
    if out["fill_history_on_reset"] not in FILL_MODES:
        raise ValueError(f"fill_history_on_reset must be one of {FILL_MODES}, got {out['fill_history_on_reset']!r}")
    return out


def student_checkpoint(trainer_state: dict, teacher_state: dict, **meta) -> dict:
    """One self-contained file: USVSysIDTrainer.state_dict() keys unchanged (load_state_dict reads it), `teacher` = the loopz
    PPO.state_dict() the student was distilled from (frozen action head, action_scale), `meta` = STUDENT_META."""
    return {**trainer_state, "teacher": teacher_state, "meta": student_meta(meta)}


class USVSysIDStudentPolicy:
    """The distilled student as a deployable policy: each control step is ONE launch of dagger_student_act_f32, which appends the
    current non-privileged frame to a per-env history ring on the device, runs the id_encoder on the window and the frozen action head on
    [frame | z^].  mu is bit-identical to USVSysIDAgent.get_student_action on USVSysIDVecEnv's history (same window semantics, quirks
    included), without the wrapper's roll / cat passes.  The ring and its slot index live on the device, so act() can be captured in a
    CUDA graph.  CUDA tensors only."""

    def __init__(self, *, id_encoder: StateHistoryEncoder, frozen_action_head: FlatMLP, history_len: int, obs_nonpriv_dim: int,
                 fill_history_on_reset: str = "zeros") -> None:
        self.id_encoder, self.head = id_encoder, frozen_action_head
        self.history_len, self.obs_nonpriv_dim = int(history_len), int(obs_nonpriv_dim)
        if id_encoder.tsteps != self.history_len or id_encoder.input_size != self.obs_nonpriv_dim:
            raise ValueError("id_encoder was built for another history shape")
        if fill_history_on_reset not in FILL_MODES:
            raise ValueError(f"fill_history_on_reset must be one of {FILL_MODES}")
        if frozen_action_head.dims[0] != self.obs_nonpriv_dim + id_encoder.output_size:
            raise ValueError(f"action head input {frozen_action_head.dims[0]} != obs_nonpriv_dim + latent_dim "
                             f"({self.obs_nonpriv_dim} + {id_encoder.output_size})")
        self.fill_history_on_reset = fill_history_on_reset
        self.device = id_encoder.device
        self.ring = None                                                      # (N, T, D), allocated by reset()
        self.slot = torch.zeros(2, dtype=torch.int32, device=self.device)     # {slot of the oldest frame, CTA arrivals}
        self.action_scale = None                                              # set by from_checkpoint (the teacher's)
        self.meta = None

    def _prepare(self, obs: torch.Tensor, dones, init: bool):
        """Checks obs and dones, allocates the ring on init; -> dones as contiguous int64 (or None)."""
        if not torch.is_tensor(obs) or not obs.is_cuda:
            raise _lib.UsvLibraryError("USVSysIDStudentPolicy needs CUDA tensors (there is no CPU fallback)")
        if obs.dtype != torch.float32 or obs.dim() != 2 or obs.stride(1) != 1 or obs.shape[1] < self.obs_nonpriv_dim:
            raise ValueError(f"obs must be fp32 [N, >= {self.obs_nonpriv_dim}] with unit column stride, got {obs.dtype} {tuple(obs.shape)}")
        n, T, D = obs.shape[0], self.history_len, self.obs_nonpriv_dim
        if init:
            if self.ring is None or self.ring.shape[0] != n:
                self.ring = torch.zeros((n, T, D), dtype=torch.float32, device=self.device)
                self.slot.zero_()
        elif self.ring is None or self.ring.shape[0] != n:
            raise RuntimeError("reset(obs) initialises the history before the first act(obs)")
        if dones is not None:
            dones = dones.reshape(-1)
            if dones.numel() != n:
                raise ValueError(f"dones has {dones.numel()} entries for {n} envs")
            dones = dones if dones.dtype == torch.int64 and dones.is_contiguous() else dones.to(torch.int64).contiguous()
        return dones

    def _launch(self, obs: torch.Tensor, dones, init: bool, latent_out) -> torch.Tensor:
        dones = self._prepare(obs, dones, init)
        n, T, D, lat = obs.shape[0], self.history_len, self.obs_nonpriv_dim, self.id_encoder.output_size
        if latent_out is not None and (latent_out.shape != (n, lat) or latent_out.dtype != torch.float32):
            raise ValueError(f"latent_out must be fp32 [{n}, {lat}]")
        mu = torch.empty((n, self.head.dims[-1]), dtype=torch.float32, device=self.device)
        I32 = ctypes.c_int32
        rc = _lib.lib().dagger_student_act_f32(
            _lib.ptr(self.id_encoder.flat), *_mlp_args(self.head), _lib.ptr(self.ring), _lib.ptr(self.slot), ctypes.c_void_p(obs.data_ptr()),
            ctypes.c_int64(obs.stride(0)), I32(D), I32(T), I32(lat),
            _lib.ptr(dones), I32(FILL_MODES.index(self.fill_history_on_reset)), I32(int(init)), _lib.ptr(mu), _lib.ptr(latent_out),
            ctypes.c_int64(n), _lib.stream())
        _lib.check(rc, "dagger_student_act_f32")
        return mu

    def reset(self, obs: torch.Tensor, latent_out=None) -> torch.Tensor:
        """USVSysIDVecEnv.reset(): fills every env's window from obs[:, :D] ("zeros" or "repeat"); -> mu of that window."""
        return self._launch(obs, None, True, latent_out)

    def act(self, obs: torch.Tensor, dones=None, latent_out=None) -> torch.Tensor:
        """One control step: appends obs[:, :D] to the history (dones: the flags of the step that produced obs, used by "repeat");
        -> the head's raw output mu (N, 2).  latent_out (N, latent_dim), if given, receives z^."""
        return self._launch(obs, dones, False, latent_out)

    def history(self) -> torch.Tensor:
        """(N, T, D) copy of the window, oldest frame first (USVSysIDVecEnv._history_torch).  Not for the hot path."""
        if self.ring is None:
            raise RuntimeError("no history before reset(obs)")
        idx = (torch.arange(self.history_len, device=self.device) + self.slot[0].long()) % self.history_len
        return self.ring.index_select(1, idx)

    @classmethod
    def from_checkpoint(cls, path, device) -> "USVSysIDStudentPolicy":
        """A student file written by scripts/dagger_usv_sysid_loopz.py --save: id_encoder from the trainer state, the frozen action head
        and action_scale from the embedded teacher."""
        sd = torch.load(path, map_location=device, weights_only=False)
        meta = student_meta(sd["meta"])
        T, D, lat, priv = meta["history_len"], meta["obs_nonpriv_dim"], meta["latent_dim"], meta["priv_dim"]
        enc = StateHistoryEncoder("LeakyReLU", D, T, lat, device)
        enc.load_state_dict(sd["id_encoder_state_dict"])
        teacher = sd["teacher"]
        arch_sd = teacher["actor_architecture_state_dict"]
        n_act = int(arch_sd["architecture.action_mlp.4.weight"].shape[0])
        with torch.random.fork_rng(devices=[]):                           # MLPEncode's init draws; the loaded weights replace them
            arch = MLPEncode([H, H], "LeakyReLU", D + priv, n_act, "Tanh", speed_dim=3, mass_dim=priv, mass_latent_dim=lat,
                             mass_encoder_shape=[E1, E2])
        arch.load_state_dict(arch_sd, "architecture.")
        arch.flat = arch.flat.to(enc.device)
        pol = cls(id_encoder=enc, frozen_action_head=arch.action_mlp, history_len=T, obs_nonpriv_dim=D,
                  fill_history_on_reset=meta["fill_history_on_reset"])
        pol.action_scale = torch.as_tensor(teacher["actor_distribution_state_dict"]["action_scale"], dtype=torch.float32).to(enc.device)
        pol.meta = meta
        return pol


class USVSysIDDistiller:
    """USVSysIDTrainer's distillation with the collection on the fused student step.  Each control step is ONE launch of
    dagger_sysid_collect_f32: the policy's history ring, encoder and action head (mu, bit-identical to USVSysIDStudentPolicy.act), the
    frame into a store that keeps each frame of the rollout once, and the teacher's label z* = mass_encoder(priv tail).  update()
    rebuilds every sample's window from the store inside the training and forward kernels.  The update is bit-identical to
    USVSysIDTrainer.update() on what USVSysIDVecEnv + USVSysIDTrainer.step would have stored: same Adam state, lr / StepLR, itr and
    metrics, kept in the trainer (state_dict / load_state_dict unchanged).

    Store: [N, T - 1 + H, D] fp32 (T = history_len, H = the trainer's num_transitions_per_env), refill indices [H, N] int32, labels
    [H, N, latent] fp32; the windows are the rule of dagger_sysid_collect_f32 (include/usv_b200.h).  The trainer's ObsStorage
    ([H, N, T * D], T times the store) is released: with a distiller, update() here replaces USVSysIDTrainer.update().  CUDA tensors only."""

    def __init__(self, trainer: USVSysIDTrainer, policy: USVSysIDStudentPolicy) -> None:
        agent = trainer.actor
        if policy.id_encoder is not agent.id_encoder:
            raise ValueError("the policy must act with the trainer's id_encoder")
        self.trainer, self.policy, self.teacher = trainer, policy, agent.teacher_mass_encoder
        self.T, self.D, self.H, self.N = policy.history_len, policy.obs_nonpriv_dim, trainer.num_transitions_per_env, trainer.num_envs
        self.latent_dim = trainer.latent_dim
        if self.teacher.dims[-1] != self.latent_dim:
            raise ValueError(f"teacher mass encoder gives {self.teacher.dims[-1]} latents, the trainer regresses {self.latent_dim}")
        self.priv_dim = self.teacher.dims[0]
        dev = agent.id_encoder.device
        self.store = torch.zeros((self.N, self.T - 1 + self.H, self.D), dtype=torch.float32, device=dev)
        self.refill = torch.zeros((self.H, self.N), dtype=torch.int32, device=dev)
        self.zstar = torch.zeros((self.H, self.N, self.latent_dim), dtype=torch.float32, device=dev)
        self.step = 0                                                       # rollout steps collected since the last update
        trainer.storage = None

    def _collect(self, obs: torch.Tensor, dones, init: bool) -> torch.Tensor:
        if self.step >= self.H:
            raise AssertionError(f"Rollout buffer overflow: {self.H} steps collected, update() first")
        pol = self.policy
        if torch.is_tensor(obs) and (obs.dim() != 2 or obs.shape[0] != self.N or obs.shape[1] < self.D + self.priv_dim):
            raise ValueError(f"obs must be [{self.N}, >= {self.D + self.priv_dim}] (the trainer's envs; frame, then the priv tail), "
                             f"got {tuple(obs.shape)}")
        dones = pol._prepare(obs, dones, init)
        mu = torch.empty((self.N, pol.head.dims[-1]), dtype=torch.float32, device=self.store.device)
        I32 = ctypes.c_int32
        rc = _lib.lib().dagger_sysid_collect_f32(
            _lib.ptr(pol.id_encoder.flat), *_mlp_args(pol.head), *_mlp_args(self.teacher), _lib.ptr(pol.ring), _lib.ptr(pol.slot),
            ctypes.c_void_p(obs.data_ptr()), ctypes.c_int64(obs.stride(0)), I32(self.D), I32(self.T), I32(self.latent_dim), _lib.ptr(dones),
            I32(FILL_MODES.index(pol.fill_history_on_reset)), I32(int(init)), _lib.ptr(self.store), _lib.ptr(self.refill), _lib.ptr(self.zstar),
            I32(self.step), I32(self.H), _lib.ptr(mu), ctypes.c_int64(self.N), _lib.stream())
        _lib.check(rc, "dagger_sysid_collect_f32")
        self.step += 1
        return mu

    def reset(self, obs: torch.Tensor) -> torch.Tensor:
        """USVSysIDVecEnv.reset() + the first sample of a rollout: fills every env's window from obs[:, :D]; -> mu of that window."""
        if self.step != 0:
            raise RuntimeError("reset(obs) starts a rollout: call it before the first act() or right after update()")
        return self._collect(obs, None, True)

    def act(self, obs: torch.Tensor, dones=None) -> torch.Tensor:
        """One control step and one sample: appends obs[:, :D] to the history (dones: the flags of the step that produced obs), stores
        the frame and z* of obs's priv tail; -> the head's raw output mu (N, 2), what USVSysIDTrainer.observe returns."""
        return self._collect(obs, dones, False)

    def windows(self) -> torch.Tensor:
        """(H * N, T * D) windows of the rollout, time-major (ObsStorage.obs's rows), rebuilt from the store.  Not for the hot path."""
        k = torch.arange(self.T, device=self.store.device)
        t = torch.arange(self.H, device=self.store.device).view(-1, 1, 1)
        idx = torch.maximum(t + k, self.refill.long().unsqueeze(-1))                         # [H, N, T]
        e = torch.arange(self.N, device=self.store.device).view(1, -1, 1)
        return self.store[e, idx].reshape(self.H * self.N, self.T * self.D)

    def _minibatch(self, row0: int, mb: int) -> None:
        tr, enc = self.trainer, self.policy.id_encoder
        I32, I64 = ctypes.c_int32, ctypes.c_int64
        rc = _lib.lib().dagger_sysid_minibatch_step_store_f32(
            _lib.ptr(enc.flat), _lib.ptr(self.store), _lib.ptr(self.refill), I64(self.N), I32(self.H), I64(row0), _lib.ptr(self.zstar),
            I32(enc.input_size), I32(enc.tsteps), I32(enc.output_size), _lib.ptr(tr.grads), _lib.ptr(tr.scratch), _lib.ptr(tr.exp_avg),
            _lib.ptr(tr.exp_avg_sq), _lib.ptr(tr.lr), _lib.ptr(tr.adam_step), I32(tr._parity), _lib.ptr(tr._mse), I64(mb), _lib.stream())
        _lib.check(rc, "dagger_sysid_minibatch_step_store_f32")
        tr._parity ^= 1

    def update(self) -> dict:
        """USVSysIDTrainer.update() on the collected rollout: same keys, same definitions, same bits."""
        if self.step != self.H:
            raise RuntimeError(f"update() needs a full rollout: {self.step} of {self.H} steps collected")
        mse = self.trainer._run_epochs(self._minibatch)
        enc, M = self.policy.id_encoder, self.H * self.N
        zhat = torch.empty((M, self.latent_dim), dtype=torch.float32, device=self.store.device)
        rc = _lib.lib().dagger_history_encoder_forward_store_f32(
            _lib.ptr(enc.flat), _lib.ptr(self.store), _lib.ptr(self.refill), ctypes.c_int64(self.N), ctypes.c_int32(self.H), ctypes.c_int64(0),
            ctypes.c_int32(enc.input_size), ctypes.c_int32(enc.tsteps), ctypes.c_int32(enc.output_size), _lib.ptr(zhat), ctypes.c_int64(M),
            _lib.stream())
        _lib.check(rc, "dagger_history_encoder_forward_store_f32")
        self.step = 0
        return latent_metrics(mse, zhat, self.zstar.view(M, self.latent_dim))
