#!/usr/bin/env python
"""TEST INFRASTRUCTURE ONLY.  Runs the UNMODIFIED reference classes of the USV SysID distillation step (StateHistoryEncoder,
USVSysIDAgent, USVSysIDTrainer, ObsStorage; OIGE/algo/ppo/{module,dagger,storage}.py) on seeded inputs and freezes
tests/golden/dagger_sysid.npz.  Needs a reference checkout:  USV_REFERENCE_ROOT=<reference checkout> python oracle/make_golden_dagger.py"""
import os
import sys

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402


def main():
    ref_shim.install()
    import omniisaacgymenvs.algo.ppo.dagger as D
    import omniisaacgymenvs.algo.ppo.module as M

    torch.set_num_threads(1)
    out = {}
    g = torch.Generator().manual_seed(77)
    OD, LAT, PRIV = 25, 8, 8                                          # obs_nonpriv_dim (33 - 8), latent, privileged tail
    for T_hist in (50, 20, 10):
        torch.manual_seed(100 + T_hist)
        enc = M.StateHistoryEncoder(nn.LeakyReLU, OD, T_hist, LAT)
        hist = torch.randn((6, T_hist * OD), generator=g)
        out[f"enc{T_hist}_params"] = torch.cat([p.detach().reshape(-1) for p in enc.parameters()])
        out[f"enc{T_hist}_in"], out[f"enc{T_hist}_out"] = hist, enc(hist).detach()
    # agent + trainer at the script's configuration (history 50, 4 epochs x 4 in-order minibatches, Adam 5e-4)
    torch.manual_seed(5)
    T_hist, N, T = 50, 6, 4
    teacher = nn.Sequential(nn.Linear(PRIV, 64), nn.LeakyReLU(), nn.Linear(64, 16), nn.LeakyReLU(), nn.Linear(16, LAT), nn.LeakyReLU())
    head = nn.Sequential(nn.Linear(OD + LAT, 128), nn.LeakyReLU(), nn.Linear(128, 128), nn.LeakyReLU(), nn.Linear(128, 2), nn.Tanh())
    enc = M.StateHistoryEncoder(nn.LeakyReLU, OD, T_hist, LAT)
    agent = D.USVSysIDAgent(teacher_mass_encoder=teacher, id_encoder=enc, frozen_action_head=head, history_len=T_hist, obs_nonpriv_dim=OD, device="cpu")
    trainer = D.USVSysIDTrainer(actor=agent, num_envs=N, num_transitions_per_env=T, history_dim=T_hist * OD, latent_dim=LAT, device="cpu")
    out["tr_params0"] = torch.cat([p.detach().reshape(-1) for p in enc.parameters()])
    out["teacher_params"] = torch.cat([p.detach().reshape(-1) for p in teacher.parameters()])
    out["head_params"] = torch.cat([p.detach().reshape(-1) for p in head.parameters()])
    sysid = torch.randn((T, N, T_hist * OD + OD), generator=g)
    priv = torch.rand((T, N, PRIV), generator=g) * 2 - 1
    out["tr_sysid_obs"], out["tr_priv"] = sysid, priv
    out["tr_actions0"] = torch.from_numpy(trainer.observe(sysid[0].numpy()))
    out["tr_zstar"] = torch.stack([agent.teacher_latent(priv[t]).detach() for t in range(T)])
    metrics = []
    for upd in range(2):
        for t in range(T):
            trainer.step(sysid[t].numpy(), priv[t])
        m = trainer.update()
        metrics.append([m["mse"], m["zstar_var_mean"], m["zhat_var_mean"], m["r2_total"]] + [m[f"r2_dim{i}"] for i in range(LAT)])
        out[f"tr_params{upd + 1}"] = torch.cat([p.detach().reshape(-1) for p in enc.parameters()])
    out["tr_metrics"] = torch.tensor(metrics, dtype=torch.float64)
    out["tr_lr_after"] = torch.tensor(trainer.optimizer.param_groups[0]["lr"])
    path = os.path.join(ROOT, "tests", "golden", "dagger_sysid.npz")
    np.savez_compressed(path, **{k: v.numpy() for k, v in out.items()})
    print("wrote", path, {k: tuple(v.shape) for k, v in out.items() if v.dim() > 1})


if __name__ == "__main__":
    main()
