"""Actor / critic / distribution surfaces of the loopz PPO on the C-ABI kernels (csrc/ppo_loopz.cu).

Mirrors `omniisaacgymenvs/algo/ppo/module.py` of the reference for the classes the USV pipeline instantiates
(`rlgames_train_loopz.py:784-822`): `MLPEncode_wrap` (:363-390) around `MLPEncode` (:184-361), `Actor` (:54-96),
`Critic` (:98-115) and `SquashedGaussianDiagonalCovariance` (:517-659).  The networks are not `nn.Module`s here: all
parameters live in ONE flat fp32 CUDA vector in the order of the reference's optimiser
(`[*actor.parameters(), *critic.parameters()]`, ppo.py:60) so that the fused gradient / clip / Adam kernels work on one
span; `state_dict()` / `load_state_dict()` use the reference's key names, so its `.pt` checkpoints
(`actor_architecture_state_dict`, `actor_distribution_state_dict`, `critic_architecture_state_dict`) interchange.

There is no CPU path: the networks compute only on CUDA tensors through libusv_b200.so."""
from __future__ import annotations

import ctypes
import math
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from ... import _lib

H = _lib.ENUMS["PPO_HIDDEN"]
E1, E2, E3 = _lib.ENUMS["PPO_LOOPZ_ENC1"], _lib.ENUMS["PPO_LOOPZ_ENC2"], _lib.ENUMS["PPO_LOOPZ_LATENT"]


def _is_leaky_relu(fn) -> bool:
    name = fn if isinstance(fn, str) else getattr(fn, "__name__", type(fn).__name__)
    return str(name).lower().replace("_", "") in ("leakyrelu",)


def _is_tanh(fn) -> bool:
    name = fn if isinstance(fn, str) else getattr(fn, "__name__", type(fn).__name__)
    return str(name).lower() == "tanh"


def net_param_shapes(obs_dim: int, mass_dim: int, out: int):
    """(name, shape) in nn.Module registration order: mass_encoder first, then action_mlp  [ref module.py:250-310]."""
    IN = obs_dim - mass_dim + E3
    return [("mass_encoder.0.weight", (E1, mass_dim)), ("mass_encoder.0.bias", (E1,)),
            ("mass_encoder.2.weight", (E2, E1)), ("mass_encoder.2.bias", (E2,)),
            ("mass_encoder.4.weight", (E3, E2)), ("mass_encoder.4.bias", (E3,)),
            ("action_mlp.0.weight", (H, IN)), ("action_mlp.0.bias", (H,)),
            ("action_mlp.2.weight", (H, H)), ("action_mlp.2.bias", (H,)),
            ("action_mlp.4.weight", (out, H)), ("action_mlp.4.bias", (out,))]


class MLPEncode:
    """Parameter holder + shape contract of the reference's MLPEncode (the compute lives in the kernels)."""

    def __init__(self, shape, actionvation_fn, input_size, output_size, output_activation_fn=None, small_init=False,
                 speed_dim=3, mass_dim=4, mass_latent_dim: int = 8, mass_encoder_shape=(64, 16)):
        self.obs_dim, self.speed_dim, self.mass_dim = int(input_size), int(speed_dim), int(mass_dim)
        if self.speed_dim <= 0 or self.mass_dim <= 0:
            raise ValueError(f"speed_dim and mass_dim must be > 0, got speed_dim={self.speed_dim}, mass_dim={self.mass_dim}")
        self.task_dim = self.obs_dim - self.speed_dim - self.mass_dim
        if self.task_dim <= 0:
            raise ValueError(f"Invalid obs split: input_size={self.obs_dim}, speed_dim={self.speed_dim}, mass_dim={self.mass_dim} "
                             f"=> task_dim={self.task_dim}")
        if mass_encoder_shape is None:
            mass_encoder_shape = (64, 16)
        if not isinstance(mass_encoder_shape, (list, tuple)):
            raise TypeError(f"mass_encoder_shape must be list/tuple, got {type(mass_encoder_shape)}")
        # the kernels are compiled for the configuration the reference ships (cfg/task/USV/IROS2024/cfg.yaml:34-43)
        if [int(x) for x in shape] != [H, H] or [int(x) for x in mass_encoder_shape] != [E1, E2] or int(mass_latent_dim) != E3:
            raise NotImplementedError(f"loopz kernels support policy/value nets [{H},{H}] with mass encoder [{E1},{E2}] -> {E3} "
                                      f"(got {list(shape)}, {list(mass_encoder_shape)} -> {mass_latent_dim})")
        if not _is_leaky_relu(actionvation_fn):
            raise NotImplementedError("loopz kernels implement nn.LeakyReLU hidden activations (rlgames_train_loopz.py:793,810)")
        if output_activation_fn is not None and not _is_tanh(output_activation_fn):
            raise NotImplementedError("output activation must be None or nn.Tanh (rlgames_train_loopz.py:159-161)")
        if self.mass_dim > _lib.ENUMS["PPO_LOOPZ_MAX_MASS"] or self.obs_dim > _lib.ENUMS["PPO_MAX_OBS"]:
            raise NotImplementedError("mass_dim <= 8 and obs_dim <= 64")
        self.tanh_out = output_activation_fn is not None
        self.out = int(output_size)
        self.input_shape = [input_size]
        self.output_shape = [output_size]
        self._shapes = net_param_shapes(self.obs_dim, self.mass_dim, self.out)
        self.flat = torch.zeros(sum(math.prod(s) for _, s in self._shapes), dtype=torch.float32)
        self.init_weights(small_init)

    def init_weights(self, small_init=False):
        """orthogonal_(gain=sqrt 2) on every Linear weight, nn.Linear's default bias init  [ref module.py:312-338]."""
        for name, t in self.views().items():
            if name.endswith(".weight"):
                w = torch.empty(t.shape)
                torch.nn.init.orthogonal_(w, gain=math.sqrt(2))
                if small_init and name == "action_mlp.4.weight":
                    w *= 1e-6
                t.copy_(w)
            else:
                fan_in = self.views()[name.replace(".bias", ".weight")].shape[1]
                t.copy_(torch.empty(t.shape).uniform_(-1.0 / math.sqrt(fan_in), 1.0 / math.sqrt(fan_in)))

    def views(self) -> Dict[str, torch.Tensor]:
        out, off = {}, 0
        for name, shp in self._shapes:
            n = math.prod(shp)
            out[name] = self.flat[off:off + n].view(shp)
            off += n
        return out

    def parameters(self) -> List[torch.Tensor]:
        return list(self.views().values())

    def _submodule(self, prefix: str, last_activation: int) -> "FlatMLP":
        layers, off = [], 0
        for name, shp in self._shapes:
            n = math.prod(shp)
            if name.startswith(prefix) and name.endswith(".weight"):
                layers.append((off, off + n, int(shp[1]), int(shp[0])))           # weight offset, bias offset, in, out
            off += n
        return FlatMLP(lambda: self.flat, layers, last_activation)

    @property
    def mass_encoder(self) -> "FlatMLP":
        """The privileged-tail encoder as a callable (priv [M, mass_dim] -> latent [M, 8]); reads this network's live parameters.
        The SysID script takes it as the frozen teacher  [ref: dagger_usv_sysid_loopz.py ; module.py:250-270]."""
        return self._submodule("mass_encoder.", 0)

    @property
    def action_mlp(self) -> "FlatMLP":
        """The trunk on [speed | task | latent] as a callable ([M, obs_dim - mass_dim + 8] -> [M, out]); the SysID script's frozen action head."""
        return self._submodule("action_mlp.", 1 if self.tanh_out else 2)

    def state_dict(self, prefix: str = "") -> Dict[str, torch.Tensor]:
        return {prefix + k: v.detach().clone() for k, v in self.views().items()}

    def load_state_dict(self, sd, prefix: str = ""):
        v = self.views()
        missing = [k for k in v if prefix + k not in sd]
        if missing:
            raise KeyError(f"missing keys in state_dict: {missing}")
        for k, t in v.items():
            t.copy_(torch.as_tensor(sd[prefix + k], dtype=torch.float32).reshape(t.shape))


class FlatMLP:
    """<= 3 nn.Linear layers with LeakyReLU between them, evaluated by dagger_mlp_forward_f32 out of a flat CUDA parameter vector.
    `flat` is a callable returning that vector (a view of its owner's storage, so a parameter update is seen without re-binding)."""

    def __init__(self, flat, layers, last_activation: int):
        self._flat, self.layers, self.last_activation = flat, list(layers), int(last_activation)
        if not 1 <= len(self.layers) <= 3:
            raise NotImplementedError("FlatMLP: 1..3 layers")
        self.dims = [self.layers[0][2]] + [l[3] for l in self.layers]

    def to(self, device):
        return self

    def parameters(self):
        return []                                # frozen: nothing for an optimiser

    def __call__(self, x) -> torch.Tensor:
        flat = self._flat()
        if not flat.is_cuda:
            raise _lib.UsvLibraryError("FlatMLP needs its network bound to a CUDA Actor / Critic (no CPU fallback)")
        x = _as_dev(x, flat.device)
        if x.shape[1] < self.dims[0]:
            raise ValueError(f"input width {x.shape[1]} < {self.dims[0]}")
        M = x.shape[0]
        y = torch.empty((M, self.dims[-1]), dtype=torch.float32, device=flat.device)
        n = len(self.layers)
        I32 = ctypes.c_int32
        rc = _lib.lib().dagger_mlp_forward_f32(ctypes.c_void_p(flat.data_ptr()), I32(n), (I32 * (n + 1))(*self.dims),
                                               (I32 * n)(*[l[0] for l in self.layers]), (I32 * n)(*[l[1] for l in self.layers]),
                                               I32(self.last_activation), _lib.ptr(x), ctypes.c_int64(x.shape[1]), _lib.ptr(y),
                                               ctypes.c_int64(M), _lib.stream())
        _lib.check(rc, "dagger_mlp_forward_f32")
        return y


CONV_STACKS = {50: ((8, 4), (5, 1), (5, 1)), 20: ((6, 2), (4, 2)), 10: ((4, 2), (2, 1))}


class StateHistoryEncoder:
    """The SysID student [ref: OIGE/algo/ppo/module.py:392-448]: a history of `tsteps` non-privileged observations -> latent.
    Same constructor and call as the reference's nn.Module; parameters are ONE flat fp32 CUDA vector in `parameters()` order
    (encoder.0, conv_layers.{0,2,(4)}, linear_output.0), `state_dict()` uses the reference's keys.  forward runs
    dagger_history_encoder_forward_f32 (one warp per sample, weights in shared memory); training is USVSysIDTrainer's kernel."""

    def __init__(self, activation_fn, input_size, tsteps, output_size, device="cuda:0", seed: Optional[int] = None):
        if not _is_leaky_relu(activation_fn):
            raise NotImplementedError("StateHistoryEncoder kernels implement nn.LeakyReLU (dagger_usv_sysid_loopz.py passes it)")
        if int(tsteps) not in CONV_STACKS:
            raise NotImplementedError(f"tsteps {tsteps}: the reference defines 50, 20 and 10")
        self.tsteps, self.input_size, self.output_size = int(tsteps), int(input_size), int(output_size)
        self.input_shape, self.output_shape = self.input_size * self.tsteps, self.output_size
        self.device = _cuda_device(device)
        P = int(_lib.lib().dagger_history_encoder_param_count(ctypes.c_int32(self.input_size), ctypes.c_int32(self.tsteps),
                                                              ctypes.c_int32(self.output_size)))
        if P < 0:
            raise NotImplementedError("StateHistoryEncoder kernels: input_size <= 32, output_size <= 8")
        self._shapes = [("encoder.0.weight", (32, self.input_size)), ("encoder.0.bias", (32,))]
        for i, (k, _) in enumerate(CONV_STACKS[self.tsteps]):
            self._shapes += [(f"conv_layers.{2 * i}.weight", (32, 32, k)), (f"conv_layers.{2 * i}.bias", (32,))]
        self._shapes += [("linear_output.0.weight", (self.output_size, 96)), ("linear_output.0.bias", (self.output_size,))]
        assert sum(math.prod(s) for _, s in self._shapes) == P
        self.flat = torch.zeros(P, dtype=torch.float32, device=self.device)
        g = torch.Generator().manual_seed(int(seed)) if seed is not None else None
        for name, t in self.views().items():     # nn.Linear / nn.Conv1d defaults: U(+-1/sqrt(fan_in)) for weight and bias
            w = self.views()[name.replace(".bias", ".weight")]
            bound = 1.0 / math.sqrt(math.prod(w.shape[1:]))
            t.copy_(((torch.rand(t.shape, generator=g) * 2 - 1) * bound).to(self.device))

    def views(self) -> Dict[str, torch.Tensor]:
        out, off = {}, 0
        for name, shp in self._shapes:
            n = math.prod(shp)
            out[name] = self.flat[off:off + n].view(shp)
            off += n
        return out

    def parameters(self) -> List[torch.Tensor]:
        return list(self.views().values())

    def state_dict(self) -> Dict[str, torch.Tensor]:
        return {k: v.detach().clone() for k, v in self.views().items()}

    def load_state_dict(self, sd) -> None:
        for k, t in self.views().items():
            t.copy_(torch.as_tensor(sd[k], dtype=torch.float32).reshape(t.shape))

    def to(self, device):
        if torch.device(device) != self.device:
            raise _lib.UsvLibraryError("StateHistoryEncoder lives on the CUDA device it was built on")
        return self

    def forward(self, obs: torch.Tensor, row_stride: Optional[int] = None) -> torch.Tensor:
        """obs [bs, tsteps * input_size] (or wider rows: only the first tsteps * input_size columns are read) -> [bs, output_size]."""
        obs = _as_dev(obs, self.device)
        M = obs.shape[0]
        out = torch.empty((M, self.output_size), dtype=torch.float32, device=self.device)
        rc = _lib.lib().dagger_history_encoder_forward_f32(_lib.ptr(self.flat), _lib.ptr(obs), ctypes.c_int64(obs.shape[1]),
                                                           ctypes.c_int32(self.input_size), ctypes.c_int32(self.tsteps),
                                                           ctypes.c_int32(self.output_size), _lib.ptr(out), ctypes.c_int64(M), _lib.stream())
        _lib.check(rc, "dagger_history_encoder_forward_f32")
        return out

    __call__ = forward


class MLPEncode_wrap:
    """`.architecture` holds the real network, shapes are passed through  [ref module.py:363-390]."""

    def __init__(self, shape, actionvation_fn, input_size, output_size, output_activation_fn=None, small_init=False, speed_dim=3,
                 mass_dim=4, mass_latent_dim: int = 8, mass_encoder_shape=(64, 16)):
        self.architecture = MLPEncode(shape, actionvation_fn, input_size, output_size, output_activation_fn, small_init,
                                      speed_dim=speed_dim, mass_dim=mass_dim, mass_latent_dim=mass_latent_dim,
                                      mass_encoder_shape=mass_encoder_shape)
        self.input_shape = self.architecture.input_shape
        self.output_shape = self.architecture.output_shape

    def parameters(self):
        return self.architecture.parameters()

    def state_dict(self):
        return self.architecture.state_dict("architecture.")

    def load_state_dict(self, sd):
        self.architecture.load_state_dict(sd, "architecture.")

    def to(self, device):
        return self


class SquashedGaussianDiagonalCovariance:
    """a = tanh(u) * action_scale, u ~ Normal(mean, std); std is a free parameter  [ref module.py:517-659]."""

    def __init__(self, dim, init_std, action_scale=1.0, eps: float = 1e-6):
        self.dim = int(dim)
        if self.dim != 2:
            raise NotImplementedError("the USV action space has 2 dimensions (left / right thruster)")
        self.std = float(init_std) * torch.ones(self.dim)
        self.eps = float(eps)
        scale = torch.as_tensor(action_scale, dtype=torch.float32).reshape(-1)
        if scale.numel() not in (1, self.dim):
            raise ValueError(f"action_scale must be scalar or shape ({self.dim},), got {tuple(scale.shape)}")
        if scale.numel() == self.dim and not bool((scale == scale[0]).all()):
            raise NotImplementedError("per-dimension action_scale: the USV pipeline passes the scalar clipActions")
        self.action_scale = scale[:1].repeat(self.dim).clone()

    def parameters(self):
        return [self.std]

    def to(self, device):
        return self

    def state_dict(self):
        return {"std": self.std.detach().clone(), "action_scale": self.action_scale.clone()}

    def load_state_dict(self, sd):
        self.std.copy_(torch.as_tensor(sd["std"], dtype=torch.float32).reshape(self.dim))
        if "action_scale" in sd:
            # the kernels read the scale from the PpoLoopzNet struct the bound Actor was built with: a checkpoint with another (or a
            # per-dimension) scale cannot be honoured by swapping this attribute, so it is refused instead of silently ignored
            new = torch.as_tensor(sd["action_scale"], dtype=torch.float32).reshape(-1).cpu()
            if new.numel() not in (1, self.dim) or not bool((new == new[0]).all()):
                raise NotImplementedError("per-dimension action_scale in the checkpoint: the kernels take one scalar scale")
            if abs(float(new[0]) - float(self.action_scale.reshape(-1)[0])) > 1e-6 * max(1.0, abs(float(new[0]))):
                raise ValueError(f"checkpoint action_scale {float(new[0])} != {float(self.action_scale.reshape(-1)[0])} of this distribution "
                                 "(construct SquashedGaussianDiagonalCovariance with the checkpoint's scale)")

    def enforce_minimum_std(self, min_std):
        if not self.std.is_cuda:
            raise _lib.UsvLibraryError("distribution is not bound to an Actor on a CUDA device")
        lo = torch.as_tensor(min_std, dtype=torch.float32, device=self.std.device).reshape(self.dim).contiguous()
        rc = _lib.lib().ppo_loopz_enforce_min_std_f32(ctypes.c_void_p(self.std.data_ptr()), _lib.ptr(lo), ctypes.c_int32(self.dim), _lib.stream())
        _lib.check(rc, "ppo_loopz_enforce_min_std_f32")


class _Store:
    """The flat parameter vector [actor architecture | std | critic architecture] the kernels read."""

    def __init__(self, net: "_lib.PpoLoopzNet", device):
        L = _lib.lib()
        L.ppo_loopz_param_count.restype = ctypes.c_int64
        L.ppo_loopz_actor_param_count.restype = ctypes.c_int64
        self.net = net
        self.P = int(L.ppo_loopz_param_count(ctypes.byref(net)))
        self.PA = int(L.ppo_loopz_actor_param_count(ctypes.byref(net)))
        if self.P < 0:
            raise NotImplementedError("unsupported loopz network shape")
        self.flat = torch.zeros(self.P, dtype=torch.float32, device=device)
        self.seed = 0
        self.counter = 0
        # device-side part of the sampling counter: a captured rollout graph adds to it at the end of each replay, the kernels see
        # (counter - _offset_host) + *counter_offset == counter at every launch (same scheme as FusedUsvEnv.step_offset)
        self.counter_offset = torch.zeros(1, dtype=torch.int64, device=device)
        self._offset_host = 0
        self.row_offset = 0          # global id of the first env this process samples for (rank x num_envs on `world` ranks)

    def advance_counter_offset(self, calls: int) -> None:
        """Inside a CUDA-graph capture containing `calls` sampling launches: the next replay draws fresh Philox samples."""
        self.counter_offset += calls

    def note_graph_replay(self, calls: int) -> None:
        self.counter += calls
        self._offset_host += calls


def _as_dev(x, device) -> torch.Tensor:
    if isinstance(x, np.ndarray):
        x = torch.from_numpy(x)
    x = x.to(device=device, dtype=torch.float32)
    return x if x.is_contiguous() else x.contiguous()


def _cuda_device(device) -> torch.device:
    d = torch.device(device)
    if d.type != "cuda":
        raise _lib.UsvLibraryError("the loopz PPO kernels run on CUDA only (no CPU fallback)")
    return d


def _net_struct(arch: MLPEncode, action_scale: float, eps: float, tanh_out: bool) -> "_lib.PpoLoopzNet":
    return _lib.STRUCTS["PpoLoopzNet"](arch.obs_dim, arch.mass_dim, int(tanh_out), float(action_scale), float(eps))


def _act(store: _Store, actor_obs, critic_obs, eval_actions, actions, log_prob, means, values, M, sample: bool):
    L = _lib.lib()
    if sample:
        store.counter += 1
    rc = L.ppo_loopz_act_f32(_lib.ptr(store.flat), ctypes.byref(store.net), _lib.ptr(actor_obs), _lib.ptr(critic_obs),
                             ctypes.c_uint64(store.seed), ctypes.c_uint64(store.counter - store._offset_host), _lib.ptr(store.counter_offset),
                             ctypes.c_int64(store.row_offset),
                             _lib.ptr(eval_actions), _lib.ptr(actions), _lib.ptr(log_prob), _lib.ptr(means), _lib.ptr(values),
                             ctypes.c_int64(M), _lib.stream())
    _lib.check(rc, "ppo_loopz_act_f32")


class Actor:
    def __init__(self, architecture: MLPEncode_wrap, distribution: SquashedGaussianDiagonalCovariance, device="cuda:0", seed: int = 0):
        self.architecture = architecture
        self.distribution = distribution
        self.device = _cuda_device(device)
        arch = architecture.architecture
        if arch.out != distribution.dim:
            raise ValueError("actor output size must equal the action dimension")
        net = _net_struct(arch, float(distribution.action_scale[0]), distribution.eps, arch.tanh_out)
        store = _Store(net, self.device)
        store.seed = int(seed)
        store.flat[:store.PA].copy_(arch.flat)
        store.flat[store.PA:store.PA + 2].copy_(distribution.std)
        self._bind(store)

    def _bind(self, store: _Store):
        self._store = store
        self.architecture.architecture.flat = store.flat[:store.PA]
        self.distribution.std = store.flat[store.PA:store.PA + 2]

    def sample(self, obs):
        """-> (actions [M,2], log_prob [M]) on the device (the reference moves them to the CPU, module.py:67-70)."""
        obs = _as_dev(obs, self.device)
        M = obs.shape[0]
        actions = torch.empty((M, 2), dtype=torch.float32, device=self.device)
        logp = torch.empty(M, dtype=torch.float32, device=self.device)
        _act(self._store, obs, None, None, actions, logp, None, None, M, True)
        return actions, logp

    def evaluate(self, obs, actions):
        """-> ((log_prob, entropy), action_mean); entropy is the reference's single-sample estimate -log_prob (module.py:632-637)."""
        obs, actions = _as_dev(obs, self.device), _as_dev(actions, self.device)
        M = obs.shape[0]
        logp = torch.empty(M, dtype=torch.float32, device=self.device)
        means = torch.empty((M, 2), dtype=torch.float32, device=self.device)
        _act(self._store, obs, None, actions, None, logp, means, None, M, False)
        return (logp, -logp), means

    def noiseless_action(self, obs):
        obs = _as_dev(obs, self.device)
        means = torch.empty((obs.shape[0], 2), dtype=torch.float32, device=self.device)
        _act(self._store, obs, None, None, None, None, means, None, obs.shape[0], False)
        return means

    def parameters(self):
        return [*self.architecture.parameters(), *self.distribution.parameters()]

    def deterministic_parameters(self):
        return self.architecture.parameters()

    @property
    def obs_shape(self):
        return self.architecture.input_shape

    @property
    def action_shape(self):
        return self.architecture.output_shape


class Critic:
    def __init__(self, architecture: MLPEncode_wrap, device="cuda:0"):
        self.architecture = architecture
        self.device = _cuda_device(device)
        arch = architecture.architecture
        if arch.out != 1:
            raise ValueError("critic output size must be 1")
        store = _Store(_net_struct(arch, 1.0, 1e-6, True), self.device)
        store.flat[store.PA + 2:].copy_(arch.flat)
        self._bind(store)

    def _bind(self, store: _Store):
        self._store = store
        self.architecture.architecture.flat = store.flat[store.PA + 2:]

    def predict(self, obs, out: Optional[torch.Tensor] = None):
        obs = _as_dev(obs, self.device)
        M = obs.shape[0]
        values = out if out is not None else torch.empty((M, 1), dtype=torch.float32, device=self.device)
        _act(self._store, None, obs, None, None, None, None, values, M, False)
        return values

    evaluate = predict

    def parameters(self):
        return [*self.architecture.parameters()]

    @property
    def obs_shape(self):
        return self.architecture.input_shape
