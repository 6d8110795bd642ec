"""GPU tests of the deployed SysID student (USVSysIDStudentPolicy over dagger_student_act_f32): the fused control step against the
unfused path it replaces (USVSysIDVecEnv's history + USVSysIDAgent.get_student_action), bit for bit; CUDA-graph replay; closed-loop play;
the student checkpoint written by scripts/dagger_usv_sysid_loopz.py."""
import csv
import dataclasses
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from omniisaacgymenvs_loop_b200 import _lib  # noqa: E402
from omniisaacgymenvs_loop_b200.algo.ppo.dagger import USVSysIDAgent, USVSysIDStudentPolicy, USVSysIDTrainer  # noqa: E402
from omniisaacgymenvs_loop_b200.algo.ppo.module import StateHistoryEncoder  # noqa: E402
from omniisaacgymenvs_loop_b200.config import UsvLiveConfig, live_default_config, live_task_cfg  # noqa: E402
from omniisaacgymenvs_loop_b200.envs.usv_raisim_vecenv import USVSysIDVecEnv  # noqa: E402

DEV = "cuda:0"
LAT = 8


def live_env(n, priv, seed, max_len):
    from scripts.train_loopz import make_env
    cfg = dataclasses.replace(live_default_config(num_envs=n, seed=seed), max_episode_length=max_len)
    return make_env(live_task_cfg(cfg, UsvLiveConfig(priv_dim=priv)), DEV, seed)


def student_parts(base, T, priv, seed):
    """-> (USVSysIDAgent, USVSysIDStudentPolicy factory) sharing one id_encoder and one frozen action head (a seeded random teacher)."""
    from scripts.train_loopz import build_learner
    D = base.num_obs - priv
    arch = build_learner(base, DEV, 16, seed, mass_dim=priv, use_cuda_graph=False).actor.architecture.architecture
    enc = StateHistoryEncoder("LeakyReLU", D, T, LAT, DEV, seed=seed)
    agent = USVSysIDAgent(teacher_mass_encoder=arch.mass_encoder, id_encoder=enc, frozen_action_head=arch.action_mlp, history_len=T,
                          obs_nonpriv_dim=D, device=DEV)

    def policy(fill):
        return USVSysIDStudentPolicy(id_encoder=enc, frozen_action_head=arch.action_mlp, history_len=T, obs_nonpriv_dim=D,
                                     fill_history_on_reset=fill)
    return agent, policy


# both fill modes x every history length; obs 33 wide (task priv_dim 8, D = 25) and 29 wide (task priv_dim 4, D = 29 - 8 = 21); ragged N
CASES = [("zeros", 50, 33, 4133), ("repeat", 50, 29, 37), ("repeat", 50, 33, 1), ("zeros", 20, 29, 1), ("repeat", 20, 33, 4133),
         ("zeros", 10, 33, 37), ("repeat", 10, 29, 4133), ("zeros", 20, 33, 37)]


@pytest.mark.parametrize("fill,T,width,n", CASES)
def test_fused_act_equals_the_unfused_student_path(fill, T, width, n):
    """One live env drives both paths with the same observations, dones and raw actions for 3 T + 7 control steps (the ring wraps three
    times, episodes of 12 steps end and restart): mu, the window and z^ must be bit-identical every step."""
    seed = 11 + T + n
    base = live_env(n, 8 if width == 33 else 4, seed, max_len=12)
    env = USVSysIDVecEnv(base._env, history_len=T, priv_dim=8, fill_history_on_reset=fill, device=DEV)
    agent, make_policy = student_parts(base, T, 8, seed)
    pol = make_policy(fill)
    D = env.obs_nonpriv_dim
    assert env.num_obs == width and D == width - 8
    lat = torch.empty((n, LAT), device=DEV)
    env.reset()
    mu = pol.reset(env.observe(as_numpy=False), latent_out=lat)
    n_done = 0
    for k in range(3 * T + 7):
        want = agent.get_student_action(env.observe_sysid_obs(as_numpy=False))
        hist = env.observe_history(as_numpy=False)
        assert torch.equal(mu, want), f"mu differs at step {k}: {float((mu - want).abs().max())}"
        assert torch.equal(pol.history(), hist.view(n, T, D)), f"history differs at step {k}"
        assert torch.equal(lat, agent.id_encoder(hist)), f"latent differs at step {k}"
        _, dones = env.step(want)
        n_done += int(dones.sum())
        mu = pol.act(env.observe(as_numpy=False), dones, latent_out=lat)
    assert n_done >= n and int(pol.slot[1]) == 0
    with pytest.raises(_lib.UsvLibraryError):
        pol.act(env.observe(as_numpy=False).cpu())


@pytest.mark.parametrize("fill,T,n", [("repeat", 20, 37), ("zeros", 50, 300)])
def test_graph_replay_equals_eager_steps(fill, T, n):
    """K act() launches captured in one CUDA graph and replayed twice give the bits of 2 K eager calls on the same inputs: the slot index
    advances on the device."""
    D, K = 25, T + 3
    g = torch.Generator(device=DEV).manual_seed(T)
    obs = [torch.randn((n, 33), device=DEV, generator=g) for _ in range(K + 1)]
    dones = [(torch.rand(n, device=DEV, generator=g) < 0.2).long() for _ in range(K)]
    base = live_env(8, 8, 5, max_len=40)
    _, make_policy = student_parts(base, T, 8, 5)
    eager, graphed = make_policy(fill), make_policy(fill)
    eager.reset(obs[0])
    want = [eager.act(obs[k + 1], dones[k]).clone() for k in range(K)] + [eager.act(obs[k + 1], dones[k]).clone() for k in range(K)]
    graphed.reset(obs[0])
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = [graphed.act(obs[k + 1], dones[k]) for k in range(K)]
    got = []
    for _ in range(2):
        graph.replay()
        got += [o.clone() for o in outs]
    torch.cuda.synchronize()
    for k, (a, b) in enumerate(zip(got, want)):
        assert torch.equal(a, b), f"graph step {k}"
    assert torch.equal(graphed.history(), eager.history()) and torch.equal(graphed.slot, eager.slot)
    assert int(graphed.slot[0]) == (1 + 2 * K) % T                        # reset() is a launch too


def _same_rows(a, b, skip=()):
    assert len(a) == len(b) and len(a) > 0
    for ra, rb in zip(a, b):
        assert list(ra) == list(rb)
        for key in ra:
            if key in skip:
                continue
            x, y = ra[key], rb[key]
            same = x == y or (isinstance(x, float) and isinstance(y, float) and math.isnan(x) and math.isnan(y))
            assert same, (key, x, y)


class UnfusedStudent:
    """play_student's policy interface on the unfused path: the USVSysIDVecEnv being played keeps the history, the agent reads it."""

    def __init__(self, env, agent, action_scale):
        self.env, self.agent, self.action_scale = env, agent, action_scale

    def reset(self, obs):
        return self.agent.get_student_action(self.env.observe_sysid_obs(as_numpy=False))

    def act(self, obs, dones):
        return self.agent.get_student_action(self.env.observe_sysid_obs(as_numpy=False))


@pytest.mark.parametrize("fill", ["zeros", "repeat"])
def test_play_student_rows_equal_the_unfused_path(fill):
    from scripts.play_loopz import play_student
    n, seed, T = 256, 23, 50
    scale = torch.ones(2, device=DEV)
    fused_env = live_env(n, 8, seed, max_len=60)
    agent, make_policy = student_parts(fused_env, T, 8, seed)
    pol = make_policy(fill)
    pol.action_scale = scale
    rows = play_student(fused_env, pol, 300, run_id="student", ckpt="none", seed=seed).rows
    ref_env = USVSysIDVecEnv(live_env(n, 8, seed, max_len=60)._env, history_len=T, priv_dim=8, fill_history_on_reset=fill, device=DEV)
    ref = play_student(ref_env, UnfusedStudent(ref_env, agent, scale), 300, run_id="student", ckpt="none", seed=seed).rows
    assert len(rows) >= 300
    _same_rows(rows, ref)                                      # every column, the obstacle hash included


@pytest.fixture(scope="module")
def student_file(tmp_path_factory):
    """Two distillation updates on 64 envs, saved the way `dagger_usv_sysid_loopz.py --save` saves."""
    from scripts.dagger_usv_sysid_loopz import build_with_teacher, run, save_student
    torch.manual_seed(3)
    env, trainer, ppo = build_with_teacher(64, DEV, seed=3, history_len=50, priv_dim=8, horizon=8)
    run(env, trainer, 2, horizon=8, quiet=True)
    path = str(tmp_path_factory.mktemp("student") / "s.pt")
    save_student(path, env, trainer, ppo, seed=3)
    teacher = str(tmp_path_factory.mktemp("teacher") / "t.pt")
    torch.save(ppo.state_dict(), teacher)
    return path, teacher, trainer, ppo


def test_student_checkpoint_round_trip(student_file):
    path, _, trainer, ppo = student_file
    pol = USVSysIDStudentPolicy.from_checkpoint(path, DEV)
    assert pol.meta == dict(history_len=50, priv_dim=8, obs_nonpriv_dim=25, latent_dim=LAT, fill_history_on_reset="zeros", seed=3)
    assert torch.equal(pol.id_encoder.flat, trainer.actor.id_encoder.flat)
    arch = ppo.actor.architecture.architecture
    assert torch.equal(pol.head._flat(), arch.flat) and pol.head.layers == arch.action_mlp.layers
    assert pol.head.last_activation == arch.action_mlp.last_activation
    assert torch.equal(pol.action_scale.cpu(), ppo.actor.distribution.action_scale.cpu())
    enc = StateHistoryEncoder("LeakyReLU", 25, 50, LAT, DEV, seed=99)
    agent = USVSysIDAgent(teacher_mass_encoder=None, id_encoder=enc, frozen_action_head=None, history_len=50, obs_nonpriv_dim=25, device=DEV)
    fresh = USVSysIDTrainer(actor=agent, num_envs=64, num_transitions_per_env=8, history_dim=50 * 25, latent_dim=LAT, device=DEV)
    fresh.load_state_dict(torch.load(path, map_location=DEV, weights_only=False))
    assert torch.equal(enc.flat, trainer.actor.id_encoder.flat) and fresh.itr == 2 and torch.equal(fresh.exp_avg, trainer.exp_avg)


def test_play_both_teacher_rows_equal_teacher_only_play(student_file, tmp_path):
    from scripts.play_loopz import main
    path, teacher, _, _ = student_file
    both, alone = tmp_path / "both.csv", tmp_path / "alone.csv"
    common = ["--num-envs", "256", "--episodes", "150", "--seed", "7"]
    main(["--student", path, "--policy", "both", "--csv", str(both), *common])
    main(["--checkpoint", teacher, "--csv", str(alone), *common])
    rows_both = list(csv.DictReader(open(both)))
    rows_alone = list(csv.DictReader(open(alone)))
    teacher_rows = [r for r in rows_both if r["run_id"] == "play"]
    student_rows = [r for r in rows_both if r["run_id"] == "student"]
    assert len(student_rows) >= 150 and len(teacher_rows) == len(rows_alone)
    _same_rows(teacher_rows, rows_alone, skip=("ckpt",))       # ckpt names the file the teacher came from
