"""CPU suite: the C-ABI library loads, exports every symbol include/usv_b200.h declares, and the
ctypes mirror generated from the header matches the library's struct sizes.  No compute calls."""
import ctypes
import dataclasses
import glob
import os

import pytest

from omniisaacgymenvs_loop_b200 import _lib
from omniisaacgymenvs_loop_b200.config import UsvEnvConfig, parse_penalty_lambda, load_task_yaml, PenaltyTerm
from omniisaacgymenvs_loop_b200 import config as C
from oracle import ref_shim

# the reference project's YAML files are not part of this repository: point USV_REFERENCE_ROOT at a checkout of it to run these
needs_reference = pytest.mark.skipif(not ref_shim.reference_available(), reason="needs a checkout of the reference project (USV_REFERENCE_ROOT)")


def test_library_loads_and_exports_every_declared_symbol():
    L = _lib.lib()
    syms = _lib.exported_symbols()
    assert "usv_step_fused_f32" in syms and "ppo_gae_f32" in syms and len(syms) >= 14
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/usv_b200.h but not exported by libusv_b200.so"
    assert L.usv_b200_abi_version() == _lib.ENUMS["USV_B200_ABI_VERSION"]


def test_struct_sizes_match_library():
    L = _lib.lib()
    for name, st in _lib.STRUCTS.items():
        assert L.usv_b200_sizeof(name.encode()) == ctypes.sizeof(st), name
    assert L.usv_b200_sizeof(b"NoSuchStruct") == -1


def test_error_strings():
    L = _lib.lib()
    assert L.usv_b200_error_string(0) == b"ok"
    assert b"NULL" in L.usv_b200_error_string(_lib.ENUMS["USV_E_NULL"])
    with pytest.raises(RuntimeError):
        _lib.check(_lib.ENUMS["USV_E_SIZE"], "x")


def test_product_fails_loudly_without_cuda_tensors():
    import torch
    with pytest.raises(_lib.UsvLibraryError):
        _lib.ptr(torch.zeros(4))
    from omniisaacgymenvs_loop_b200.engine import FusedUsvEnv
    with pytest.raises(_lib.UsvLibraryError):
        FusedUsvEnv(UsvEnvConfig(), 8, device="cpu")
    from omniisaacgymenvs_loop_b200.envs.USV.Hydrostatics import HydrostaticsObject
    with pytest.raises(_lib.UsvLibraryError):
        HydrostaticsObject(4, "cpu", 1000, -9.81, 0.5, 0.65, 275, 1.0, 0.0, 1.0, 0.3, -10.0)
    # the evaluation player has no torch-module fallback either: its policy is the CUDA kernel
    import numpy as np
    from omniisaacgymenvs_loop_b200.rl.players import PpoPlayerContinuous, rescale_actions
    from omniisaacgymenvs_loop_b200.utils.spaces import Box, Dict

    class _Env:
        def get_env_info(self):
            return {"action_space": Box(-1.0, 1.0, (2,)), "observation_space": Dict({"state": Box(-np.inf, np.inf, (13,))})}
    with pytest.raises(_lib.UsvLibraryError):
        PpoPlayerContinuous(_Env(), {"games_num": 1}, device="cpu")
    lo, hi = torch.tensor([-2.0, 0.0]), torch.tensor([2.0, 1.0])
    assert torch.equal(rescale_actions(lo, hi, torch.tensor([[1.0, -1.0], [0.0, 0.0]])), torch.tensor([[2.0, 0.0], [0.0, 0.5]]))


def test_params_roundtrip():
    cfg = UsvEnvConfig().full_dr()
    p = cfg.to_params(step_counter=7, env_id_offset=4096, first_call=True)
    assert p.seed == 1234 and p.step_counter == 7 and p.env_id_offset == 4096 and p.first_call == 1
    assert p.n_substeps == 5 and p.max_episode_length == 3000 and abs(p.lag_alpha - 0.6703200340270996) < 1e-9
    assert p.pen_energy.form == C.PEN_EXP_NEG_SUMSQ and abs(p.pen_energy.c1 - 0.01) < 1e-9
    assert p.pen_angular_vel_variation.form == C.PEN_EXP_NEG_ABS and abs(p.pen_angular_vel_variation.k - 0.033) < 1e-9
    assert abs(p.force_const_max - 2.5 / 2 ** 0.5) < 1e-6 and abs(p.lin_rand[1] - 9.999) < 1e-5
    assert p.use_sin_force == 1 and p.mass_rand == 1


def test_penalty_lambda_closed_set():
    f = parse_penalty_lambda
    assert f("lambda x,step : -torch.sum(x, dim=-1)*0.005") == PenaltyTerm(C.PEN_NEG_SUM, 0.005)
    assert f("lambda x,step : (torch.exp(-torch.sum(x**2, dim=-1)) - 1.0) * 0.01") == PenaltyTerm(C.PEN_EXP_NEG_SUMSQ, 0.01)
    assert f("lambda x,step: -torch.norm(x, dim=-1)*0.01") == PenaltyTerm(C.PEN_NEG_ABS, 0.01)
    assert f("lambda x,step : -torch.abs(x)*0.01 + 0.0") == PenaltyTerm(C.PEN_NEG_ABS, 0.01, 0.0)
    assert f("lambda x,step: -torch.clamp(torch.abs(x)-0.4, min=0)*0.02") == PenaltyTerm(C.PEN_NEG_DEADZONE, 0.02, 0.0, 0.4)
    assert f("lambda x,step: (torch.exp(-0.033 * torch.abs(x)) - 1.0) * 1.0") == PenaltyTerm(C.PEN_EXP_NEG_ABS, 1.0, 0.0, 0.033)
    assert f("lambda x,step: torch.exp(c1 * torch.abs(x)) - 1.0", c1=-0.033) == PenaltyTerm(C.PEN_EXP_NEG_ABS, 1.0, 0.0, 0.033)
    with pytest.raises(NotImplementedError):
        f("lambda x,step: torch.tanh(x)")


@needs_reference
def test_reference_yamls_parse():
    snap = os.path.join(ref_shim.snapshot_dir(), "USV_Virtual_CaptureXY_SysID-TEST.yaml")
    cfg = UsvEnvConfig.from_task_cfg(load_task_yaml(snap))
    assert dataclasses.asdict(cfg) == dataclasses.asdict(UsvEnvConfig())   # defaults ARE the classic snapshot
    for y in glob.glob(os.path.join(ref_shim.REFERENCE_ROOT, "omniisaacgymenvs/cfg/task/USV/IROS2024/USV_Virtual_CaptureXY_*DR50.yaml")):
        c = UsvEnvConfig.from_task_cfg(load_task_yaml(y, num_envs=64))
        assert c.num_envs == 64 and c.use_sin_force and c.drag_rand and c.thr_rand and c.n_substeps == 5


def test_live_task_cfg_round_trip():
    """live_task_cfg() emits the YAML tree the live USVVirtual reads; parsing it back gives the same configs."""
    from omniisaacgymenvs_loop_b200.config import UsvLiveConfig, live_default_config, live_env_config, live_task_cfg
    cfg, live = live_default_config(num_envs=96), UsvLiveConfig()
    t = live_task_cfg(cfg, live)
    assert dataclasses.asdict(live_env_config(t)) == dataclasses.asdict(cfg)
    assert UsvLiveConfig.from_task_cfg(t) == live
    lp = live.to_params()
    assert lp.priv_mode == 2 and list(lp.priv_a) == [1.0, 0.5, 0.5, 1.0] and list(lp.priv_active) == [1, 1, 1, 1]
    # mass.masscom_obs_source: base  [ref: OIGE/tasks/USV_Virtual.py:468-472,859-880]: round trip + the neutral parameters of each encoding
    base = dataclasses.replace(live, masscom_obs_base=True)
    tb = live_task_cfg(cfg, base)
    assert tb["env"]["disturbances"]["mass"]["masscom_obs_source"] == "base" and UsvLiveConfig.from_task_cfg(tb) == base
    lpb = base.to_params()
    assert lpb.masscom_obs_base == 1 and lp.masscom_obs_base == 0 and list(lpb.priv_neutral) == [1.25, 0.75, 0.75, 1.25]   # minmax: mid-range
    assert list(dataclasses.replace(base, priv_mode=1).to_params().priv_neutral) == [1.0] * 4                              # centered / raw: 1.0
    tb["env"]["disturbances"]["mass"]["masscom_obs_source"] = "other"
    with pytest.raises(ValueError):
        UsvLiveConfig.from_task_cfg(tb)


@needs_reference
def test_reference_live_yaml_parses_to_the_shipped_defaults():
    from omniisaacgymenvs_loop_b200.config import UsvLiveConfig, live_default_config, live_env_config
    y = load_task_yaml(os.path.join(ref_shim.REFERENCE_ROOT, "omniisaacgymenvs/cfg/task/USV/IROS2024/USV_Virtual_CaptureXY_SysID-TEST.yaml"),
                       num_envs=128)
    assert dataclasses.asdict(live_env_config(y)) == dataclasses.asdict(live_default_config(num_envs=128))
    assert UsvLiveConfig.from_task_cfg(y) == UsvLiveConfig()
