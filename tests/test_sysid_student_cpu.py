"""CPU suite of the deployed SysID student: dagger_student_act_f32 rejects bad arguments before any CUDA call, the student checkpoint's
`meta` round-trips through a file, and scripts/play_loopz.py refuses privileged-tail interventions for the student."""
import ctypes

import pytest
import torch

from omniisaacgymenvs_loop_b200 import _lib
from omniisaacgymenvs_loop_b200.algo.ppo.dagger import STUDENT_META, student_checkpoint, student_meta

I32 = ctypes.c_int32
D, LAT = 25, 8


def _call(**over):
    """dagger_student_act_f32 with valid arguments (pointers that are never dereferenced, M = 0) except for the overrides."""
    a = dict(enc=256, head=256, nl=3, dims=[D + LAT, 128, 128, 2], last=1, ring=256, slot=256, obs=256, obs_ld=33, D=D, T=50, lat=LAT,
             dones=None, fill=0, init=0, mu=256, latent=None, M=0)
    a.update(over)
    nl, dims = a["nl"], a["dims"]
    return _lib.lib().dagger_student_act_f32(
        ctypes.c_void_p(a["enc"]), ctypes.c_void_p(a["head"]), I32(nl), (I32 * len(dims))(*dims), (I32 * 3)(0, 0, 0), (I32 * 3)(0, 0, 0),
        I32(a["last"]), ctypes.c_void_p(a["ring"]), ctypes.c_void_p(a["slot"]), ctypes.c_void_p(a["obs"]), ctypes.c_int64(a["obs_ld"]),
        I32(a["D"]), I32(a["T"]), I32(a["lat"]), ctypes.c_void_p(a["dones"]), I32(a["fill"]), I32(a["init"]), ctypes.c_void_p(a["mu"]),
        ctypes.c_void_p(a["latent"]), ctypes.c_int64(a["M"]), None)


def test_student_act_rejects_bad_arguments_before_any_cuda_call():
    E = _lib.ENUMS
    assert _call() == E["USV_OK"]                                                 # valid, no envs: nothing to launch
    assert _call(fill=1, init=1, dones=256, latent=256, T=10, D=21, obs_ld=21, dims=[21 + LAT, 128, 128, 2]) == E["USV_OK"]
    for name in ("enc", "head", "ring", "slot", "obs", "mu"):
        assert _call(**{name: None}) == E["USV_E_NULL"], name
    for T in (0, 5, 30, 49, 51, 100):
        assert _call(T=T) == E["USV_E_UNSUPPORTED"], T
    assert _call(obs_ld=D - 1) == E["USV_E_SIZE"]
    assert _call(dims=[D + LAT + 1, 128, 128, 2]) == E["USV_E_SIZE"]             # head input != D + latent_dim
    assert _call(dims=[D, 128, 128, 2]) == E["USV_E_SIZE"]
    assert _call(M=-1) == E["USV_E_SIZE"]
    for fill in (-1, 2):
        assert _call(fill=fill) == E["USV_E_PARAM"], fill
    assert _call(init=2) == E["USV_E_PARAM"] and _call(last=3) == E["USV_E_PARAM"]


def test_student_checkpoint_meta_round_trips(tmp_path):
    meta = dict(history_len=50, priv_dim=8, obs_nonpriv_dim=25, latent_dim=8, fill_history_on_reset="repeat", seed=1234)
    trainer_sd = {"id_encoder_state_dict": {"encoder.0.weight": torch.randn(32, 25)}, "exp_avg": torch.zeros(3), "exp_avg_sq": torch.zeros(3),
                  "step": 32, "itr": 2}
    teacher_sd = {"actor_distribution_state_dict": {"action_scale": torch.ones(2)}}
    path = tmp_path / "student.pt"
    torch.save(student_checkpoint(trainer_sd, teacher_sd, **meta), path)
    back = torch.load(path, weights_only=False)
    assert student_meta(back["meta"]) == meta and set(back["meta"]) == set(STUDENT_META)
    assert set(trainer_sd) <= set(back) and back["step"] == 32 and torch.equal(back["id_encoder_state_dict"]["encoder.0.weight"],
                                                                               trainer_sd["id_encoder_state_dict"]["encoder.0.weight"])
    with pytest.raises(KeyError):
        student_checkpoint(trainer_sd, teacher_sd, **{k: v for k, v in meta.items() if k != "seed"})
    with pytest.raises(ValueError):
        student_checkpoint(trainer_sd, teacher_sd, **{**meta, "fill_history_on_reset": "last"})


def test_play_rejects_privileged_tail_interventions_for_the_student():
    from scripts.play_loopz import parse_args
    a = parse_args(["--student", "s.pt"])
    assert a.policy == "student" and a.mass_mode == "normal"
    assert parse_args([]).policy == "teacher"
    assert parse_args(["--student", "s.pt", "--policy", "teacher", "--mass-mode", "zero"]).policy == "teacher"
    for policy in ("student", "both"):
        for extra in (["--mass-mode", "shuffle"], ["--obs-source", "base"], ["--obs-source", "both"]):
            with pytest.raises(SystemExit):
                parse_args(["--student", "s.pt", "--policy", policy, *extra])
    with pytest.raises(SystemExit):
        parse_args(["--policy", "both"])                                            # no student file

