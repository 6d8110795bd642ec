"""GPU tests of the SysID distillation from a frame store (USVSysIDDistiller over dagger_sysid_collect_f32 and the store training
kernels): the fused loop against the unfused loop it replaces (USVSysIDVecEnv + USVSysIDTrainer, scripts/dagger_usv_sysid_loopz.py
build / run), side by side from one seed on the live env, bit for bit; and the fused script's --save file."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

from omniisaacgymenvs_loop_b200.algo.ppo.dagger import USVSysIDAgent, USVSysIDStudentPolicy, USVSysIDTrainer  # noqa: E402
from omniisaacgymenvs_loop_b200.algo.ppo.module import StateHistoryEncoder  # noqa: E402

DEV = "cuda:0"
H, UPDATES = 16, 5
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# both fill modes x every history length x priv 8 / 4 (D = 25 either way on the live env) x ragged N.  Episodes of at most 15 steps put
# several "repeat" refills inside one T = 50 window and move the timeouts across the rollout's steps; windows of a rollout's first steps
# straddle the previous rollout.
CASES = [("zeros", 50, 8, 37), ("repeat", 50, 4, 4133), ("repeat", 50, 8, 1), ("zeros", 20, 4, 4133), ("repeat", 20, 8, 37),
         ("repeat", 10, 4, 37), ("zeros", 10, 8, 4133), ("repeat", 10, 8, 4133)]


@pytest.mark.parametrize("fill,T,priv,n", CASES)
def test_fused_distillation_equals_the_unfused_loop(fill, T, priv, n):
    from scripts.dagger_usv_sysid_loopz import build_fused, build_with_teacher
    seed = 7 + T + n + priv
    kw = dict(history_len=T, priv_dim=priv, horizon=H, fill_history_on_reset=fill, max_episode_length=15)
    torch.manual_seed(seed)
    env_u, trainer, ppo_u = build_with_teacher(n, DEV, seed, **kw)
    torch.manual_seed(seed)
    env_f, dist, ppo_f = build_fused(n, DEV, seed, **kw)
    tr_f, enc_u, enc_f = dist.trainer, trainer.actor.id_encoder, dist.policy.id_encoder
    assert env_u.obs_nonpriv_dim == 25 and dist.D == 25 and dist.priv_dim == priv
    assert torch.equal(ppo_u.actor.architecture.architecture.flat, ppo_f.actor.architecture.architecture.flat)
    assert torch.equal(enc_u.flat, enc_f.flat)
    env_u.reset()
    env_f.reset()
    dones, done_steps = None, set()
    for upd in range(UPDATES):
        for t in range(H):
            sysid_obs = env_u.observe_sysid_obs(as_numpy=False)        # run(): the unfused loop's step
            trainer.step(sysid_obs, env_u.get_priv_tail())
            want = trainer.observe(sysid_obs)
            obs = env_f.observe(as_numpy=False)
            if dones is not None and bool(dones.any()):
                done_steps.add(t)
            mu = dist.reset(obs) if upd == 0 and t == 0 else dist.act(obs, dones)
            assert torch.equal(mu, want), f"action differs at update {upd} step {t}: {float((mu - want).abs().max())}"
            assert torch.equal(dist.zstar[t], trainer.storage.expert[t]), f"label differs at update {upd} step {t}"
            env_u.step(want)
            _, dones = env_f.step(mu)
        assert torch.equal(dist.windows(), trainer.storage.obs.view(H * n, -1)), f"rebuilt windows differ at update {upd}"
        m_u, m_f = trainer.update(), dist.update()
        assert m_f == m_u, f"metrics differ at update {upd}: {m_f} vs {m_u}"
        assert torch.equal(enc_f.flat, enc_u.flat), f"encoder parameters differ after update {upd}"
        assert torch.equal(tr_f.exp_avg, trainer.exp_avg) and torch.equal(tr_f.exp_avg_sq, trainer.exp_avg_sq), f"Adam moments, update {upd}"
        assert torch.equal(tr_f.adam_step, trainer.adam_step) and tr_f._parity == trainer._parity and tr_f.itr == trainer.itr == upd + 1
    if fill == "repeat":
        assert int(dist.refill.max()) > T - 1                                  # refills happened inside the rollout
    if n > 1000:                                                               # early terminations spread the dones over the rollout
        assert {0, H - 1} <= done_steps, f"dones seen at rollout steps {sorted(done_steps)}"


def test_fused_save_file_loads(tmp_path):
    """scripts/dagger_usv_sysid_loopz.py (the fused loop) --save: the file loads as a deployable policy and into a trainer."""
    path = tmp_path / "s.pt"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "dagger_usv_sysid_loopz.py"), "--envs", "64", "--updates", "2",
                        "--horizon", "8", "--history-len", "20", "--seed", "3", "--save", str(path)], cwd=ROOT, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    assert "frames/s" in r.stdout and f"wrote the student to {path}" in r.stdout
    pol = USVSysIDStudentPolicy.from_checkpoint(str(path), DEV)
    assert pol.meta == dict(history_len=20, priv_dim=8, obs_nonpriv_dim=25, latent_dim=8, fill_history_on_reset="zeros", seed=3)
    sd = torch.load(path, map_location=DEV, weights_only=False)
    enc = StateHistoryEncoder("LeakyReLU", 25, 20, 8, DEV, seed=99)
    agent = USVSysIDAgent(teacher_mass_encoder=None, id_encoder=enc, frozen_action_head=None, history_len=20, obs_nonpriv_dim=25, device=DEV)
    fresh = USVSysIDTrainer(actor=agent, num_envs=64, num_transitions_per_env=8, history_dim=20 * 25, latent_dim=8, device=DEV)
    fresh.load_state_dict(sd)
    assert torch.equal(enc.flat, pol.id_encoder.flat) and fresh.itr == 4 and sd["step"] == 4 * 4 * 4   # 2 warm-up + 2 updates
    assert torch.equal(fresh.exp_avg, sd["exp_avg"].to(DEV))
