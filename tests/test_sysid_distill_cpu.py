"""CPU suite of the SysID distillation from a frame store: the three entry points behind USVSysIDDistiller reject bad arguments before any
CUDA call, and the distiller refuses CPU tensors, a rollout longer than the trainer's horizon and observations of another shape."""
import ctypes
from types import SimpleNamespace

import pytest
import torch

from omniisaacgymenvs_loop_b200 import _lib
from omniisaacgymenvs_loop_b200.algo.ppo.dagger import USVSysIDDistiller, USVSysIDStudentPolicy, USVSysIDTrainer

I32, I64, P = ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p
D, LAT, PRIV = 25, 8, 8


def _collect(**over):
    """dagger_sysid_collect_f32 with valid arguments (pointers that are never dereferenced, M = 0) except for the overrides."""
    a = dict(enc=256, head=256, nl=3, dims=[D + LAT, 128, 128, 2], last=1, teacher=256, tnl=3, tdims=[PRIV, 64, 16, LAT], tlast=0, ring=256,
             slot=256, obs=256, obs_ld=D + PRIV, D=D, T=50, lat=LAT, dones=None, fill=0, init=0, store=256, refill=256, zstar=256, t=0, H=16,
             mu=256, M=0)
    a.update(over)
    z3 = (I32 * 3)(0, 0, 0)
    return _lib.lib().dagger_sysid_collect_f32(
        P(a["enc"]), P(a["head"]), I32(a["nl"]), (I32 * len(a["dims"]))(*a["dims"]), z3, z3, I32(a["last"]), P(a["teacher"]), I32(a["tnl"]),
        (I32 * len(a["tdims"]))(*a["tdims"]), z3, z3, I32(a["tlast"]), P(a["ring"]), P(a["slot"]), P(a["obs"]), I64(a["obs_ld"]), I32(a["D"]),
        I32(a["T"]), I32(a["lat"]), P(a["dones"]), I32(a["fill"]), I32(a["init"]), P(a["store"]), P(a["refill"]), P(a["zstar"]), I32(a["t"]),
        I32(a["H"]), P(a["mu"]), I64(a["M"]), None)


def test_collect_rejects_bad_arguments_before_any_cuda_call():
    E = _lib.ENUMS
    assert _collect() == E["USV_OK"]                                              # valid, no envs: nothing to launch
    assert _collect(fill=1, init=1, dones=256, T=10, tdims=[4, 64, 16, LAT], obs_ld=D + 4, t=0, H=1) == E["USV_OK"]
    assert _collect(t=15) == E["USV_OK"]
    for name in ("enc", "head", "teacher", "ring", "slot", "obs", "store", "refill", "zstar", "mu"):
        assert _collect(**{name: None}) == E["USV_E_NULL"], name
    for T in (0, 5, 30, 49, 51):
        assert _collect(T=T) == E["USV_E_UNSUPPORTED"], T
    assert _collect(obs_ld=D + PRIV - 1) == E["USV_E_SIZE"]                        # the priv tail must be inside the row
    for t, H in ((-1, 16), (16, 16), (0, 0), (3, 2)):
        assert _collect(t=t, H=H) == E["USV_E_SIZE"], (t, H)
    assert _collect(dims=[D + LAT + 1, 128, 128, 2]) == E["USV_E_SIZE"]           # head input != D + latent_dim
    assert _collect(tdims=[PRIV, 64, 16, LAT - 1]) == E["USV_E_SIZE"]              # teacher output != latent_dim
    assert _collect(tnl=4) == E["USV_E_SIZE"] and _collect(tdims=[PRIV, 0, 16, LAT]) == E["USV_E_SIZE"]
    assert _collect(M=-1) == E["USV_E_SIZE"]
    for fill in (-1, 2):
        assert _collect(fill=fill) == E["USV_E_PARAM"], fill
    assert _collect(tlast=3) == E["USV_E_PARAM"] and _collect(last=-1) == E["USV_E_PARAM"]
    assert _collect(init=1, t=1) == E["USV_E_PARAM"]                              # a rollout's store starts with the reset window


def _forward(**over):
    a = dict(prm=256, store=256, refill=256, N=37, H=16, row0=0, In=D, T=50, Out=LAT, out=256, M=0)
    a.update(over)
    return _lib.lib().dagger_history_encoder_forward_store_f32(P(a["prm"]), P(a["store"]), P(a["refill"]), I64(a["N"]), I32(a["H"]),
                                                               I64(a["row0"]), I32(a["In"]), I32(a["T"]), I32(a["Out"]), P(a["out"]),
                                                               I64(a["M"]), None)


def _train(**over):
    a = dict(prm=256, store=256, refill=256, N=37, H=16, row0=0, zstar=256, In=D, T=50, Out=LAT, grads=256, scratch=256, m=256, v=256, lr=256,
             step=256, parity=0, mse=None, M=0)
    a.update(over)
    return _lib.lib().dagger_sysid_minibatch_step_store_f32(
        P(a["prm"]), P(a["store"]), P(a["refill"]), I64(a["N"]), I32(a["H"]), I64(a["row0"]), P(a["zstar"]), I32(a["In"]), I32(a["T"]),
        I32(a["Out"]), P(a["grads"]), P(a["scratch"]), P(a["m"]), P(a["v"]), P(a["lr"]), P(a["step"]), I32(a["parity"]), P(a["mse"]),
        I64(a["M"]), None)


def test_store_forward_and_train_reject_bad_arguments_before_any_cuda_call():
    E = _lib.ENUMS
    assert _forward() == E["USV_OK"] and _forward(row0=16 * 37) == E["USV_OK"]
    for name in ("prm", "store", "refill", "out"):
        assert _forward(**{name: None}) == E["USV_E_NULL"], name
    for name in ("prm", "store", "refill", "zstar", "grads", "scratch", "m", "v", "lr", "step"):
        assert _train(**{name: None}, M=8) == E["USV_E_NULL"], name
    for T in (0, 49, 100):
        assert _forward(T=T) == E["USV_E_UNSUPPORTED"] and _train(T=T, M=8) == E["USV_E_UNSUPPORTED"], T
    # the minibatch must lie inside the H * N windows of the store
    for row0, M in ((0, 16 * 37 + 1), (16 * 37 - 7, 8), (-1, 4), (16 * 37, 1)):
        assert _forward(row0=row0, M=M) == E["USV_E_SIZE"] and _train(row0=row0, M=M) == E["USV_E_SIZE"], (row0, M)
    for bad in (dict(N=0), dict(H=0), dict(In=0), dict(In=33), dict(Out=0), dict(Out=9), dict(M=-1)):
        assert _forward(**bad) == E["USV_E_SIZE"] and _train(**{"M": 8, **bad}) == E["USV_E_SIZE"], bad
    assert _train(M=0) == E["USV_E_SIZE"]                                         # a training step needs samples
    assert _train(parity=2, M=8) == E["USV_E_PARAM"]


def _fake_distiller(N=37, T=10, H=4, teacher_out=LAT):
    """A USVSysIDDistiller over CPU stand-ins of the trainer and the policy (only what its constructor and checks read)."""
    enc = SimpleNamespace(device=torch.device("cpu"), tsteps=T, input_size=D, output_size=LAT)
    pol = USVSysIDStudentPolicy.__new__(USVSysIDStudentPolicy)
    pol.__dict__.update(id_encoder=enc, head=SimpleNamespace(dims=[D + LAT, 128, 128, 2]), history_len=T, obs_nonpriv_dim=D,
                        fill_history_on_reset="zeros", ring=None, device=enc.device)
    tr = USVSysIDTrainer.__new__(USVSysIDTrainer)
    tr.__dict__.update(actor=SimpleNamespace(id_encoder=enc, teacher_mass_encoder=SimpleNamespace(dims=[PRIV, 64, 16, teacher_out])),
                       num_transitions_per_env=H, num_envs=N, latent_dim=LAT, storage=object())
    return USVSysIDDistiller(tr, pol), tr, pol


def test_distiller_layout_and_refusals():
    N, T, H = 37, 10, 4
    dist, tr, pol = _fake_distiller(N, T, H)
    assert dist.store.shape == (N, T - 1 + H, D) and dist.refill.shape == (H, N) and dist.zstar.shape == (H, N, LAT)
    assert tr.storage is None                                                     # the frames live in the store now
    obs = torch.zeros((N, D + PRIV))
    with pytest.raises(_lib.UsvLibraryError):                                     # CUDA tensors only: no CPU fallback
        dist.reset(obs)
    with pytest.raises(_lib.UsvLibraryError):
        dist.act(obs)
    for shape in ((N + 1, D + PRIV), (N, D + PRIV - 1), (N,)):
        with pytest.raises(ValueError):
            dist.act(torch.zeros(shape))
    dist.step = H                                                                 # a full rollout: the next sample would overflow
    with pytest.raises(AssertionError):
        dist.act(obs)
    with pytest.raises(RuntimeError):
        dist.reset(obs)
    dist.step = H - 1
    with pytest.raises(RuntimeError):                                             # update() wants the whole rollout
        dist.update()
    with pytest.raises(ValueError):
        _fake_distiller(teacher_out=LAT - 1)
    other, _, pol2 = _fake_distiller()
    pol2.id_encoder = SimpleNamespace(device=torch.device("cpu"))
    with pytest.raises(ValueError):
        USVSysIDDistiller(tr, pol2)
