"""TEST INFRASTRUCTURE ONLY.  Generates tests/golden/*.npz by executing the UNMODIFIED reference
modules (a reference checkout, CPU torch, fp32) under oracle/ref_shim.py on seeded synthetic inputs.

Run where a checkout of the reference exists:
    USV_REFERENCE_ROOT=<reference checkout> python -m oracle.make_golden
The fixtures are small (N=32) and committed; tests/test_oracle_cpu.py checks the oracle restatement
against them and tests/test_gpu_parity.py checks the CUDA kernels against them.

Synthetic inputs follow SURVEY 8(d): pos ~ U(-12,12)^2, yaw ~ U(-pi,pi), vx,vy ~ U(-1.5,1.5),
r ~ U(-1,1), 6-DOF variant with random unit quaternions / N(0,0.3) heave-roll-pitch rates.
"""
from __future__ import annotations

import math
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
N = 32


def gen():
    return torch.Generator().manual_seed(1234)


def t2n(d):
    return {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in d.items()}


DRAG_CFG = dict(use_drag_randomization=False, u_linear_rand=0.1, v_linear_rand=0.1, w_linear_rand=0.0,
                p_linear_rand=0.0, q_linear_rand=0.0, r_linear_rand=0.1, u_quad_rand=0.1, v_quad_rand=0.1,
                w_quad_rand=0.0, p_quad_rand=0.0, q_quad_rand=0.0, r_quad_rand=0.1)
LIN = [0.0, 99.99, 99.99, 13.0, 13.0, 0.82985084]
QUAD = [17.257603, 99.99, 10.0, 5.0, 5.0, 17.33600724]
LUT_CLASSIC_L = [-3.8, -3.8, -3.6, -3.6, -1.6, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 4.0, 10.0, 15.0, 21.0, 23.0, 22.0]
LUT_CLASSIC_R = [-5.0, -5.0, -5.0, -4.6, -2.2, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 4.6, 10.0, 17.0, 24.0, 24.0, 23.0]
LUT_LIVE = [0.0] * 11 + [8.0 * i for i in range(1, 11)]
LUT_NOMINAL = [-19.88, -16.52, -12.6, -5.6, -1.4, 0.0, 2.24, 9.52, 21.28, 28.0, 33.6]
THR_CFG = dict(use_thruster_randomization=False, thruster_rand=0.5, use_separate_randomization=False,
               left_rand=0.5, right_rand=0.5)


def force_modules():
    hs, hd, td = ref_shim.load_force_modules()
    g = gen()
    out = {}
    # ---- inputs: 6-DOF variant
    q = torch.randn((N, 4), generator=g)
    q = q / q.norm(dim=1, keepdim=True)
    q[0] = torch.tensor([1.0, 0, 0, 0])
    q[1] = torch.tensor([math.cos(math.pi / 6), 0, 0, math.sin(math.pi / 6)])
    q[2] = q[2] * 1.7  # non-unit quaternion: two_s = 2/|q|^2 must absorb it
    yaw = (torch.rand(N, generator=g) * 2 - 1) * math.pi
    q_planar = torch.stack([torch.cos(yaw / 2), torch.zeros(N), torch.zeros(N), torch.sin(yaw / 2)], 1)
    vel6 = torch.zeros((N, 6))
    vel6[:, 0:2] = torch.rand((N, 2), generator=g) * 3 - 1.5
    vel6[:, 2:5] = torch.randn((N, 3), generator=g) * 0.3
    vel6[:, 5] = torch.rand(N, generator=g) * 2 - 1
    vel6[0] = torch.tensor([1.0, 0.5, 0, 0, 0, 0.3])
    vel6[1] = torch.tensor([-0.4, 1.2, 0, 0, 0, -0.7])
    vel6_planar = vel6.clone()
    vel6_planar[:, 2:5] = 0
    vol = torch.rand(N, generator=g) * 0.05
    rpy = torch.randn((N, 3), generator=g) * 0.1
    out.update(quat=q, quat_planar=q_planar, yaw=yaw, vel6=vel6, vel6_planar=vel6_planar, vol=vol, rpy=rpy)

    # ---- A1 hydrostatics  (ctor args as USV_Virtual.get_USV_dynamics passes them)
    H = hs.HydrostaticsObject(N, "cpu", 1000, -9.81, 0.5, 0.65, 275, 1.0, 0.0, 1.0, 0.3, -10.0)
    out["hs_out"] = H.compute_archimedes_metacentric_local(vol, rpy, q).clone()
    out["hs_force_global"] = H.archimedes_force_global.clone()
    out["hs_torque_global"] = H.archimedes_torque_global.clone()
    out["hs_out_planar"] = H.compute_archimedes_metacentric_local(vol, rpy * 0, q_planar).clone()
    H2 = hs.HydrostaticsObject(N, "cpu", 1025.0, -9.80665, 0.4, 0.7, 300.0, 2.5, 0.0, 1.0, 0.3, -10.0)
    out["hs_out_alt"] = H2.compute_archimedes_metacentric_local(vol, rpy, q).clone()

    # ---- A2 hydrodynamics
    def mk(cfg_extra=None, **kw):
        cfg = dict(DRAG_CFG)
        cfg.update(cfg_extra or {})
        args = dict(task_cfg=cfg, num_envs=N, device="cpu", water_density=1000, gravity=-9.81, linear_damping=LIN,
                    quadratic_damping=QUAD, linear_damping_forward_speed=[0.0] * 6, offset_linear_damping=0.0,
                    offset_lin_forward_damping_speed=0.0, offset_nonlin_damping=0.0, scaling_damping=1.0,
                    offset_added_mass=0.0, scaling_added_mass=1.0, alpha=0.3, last_time=-10.0)
        args.update(kw)
        return hd.HydrodynamicsObject(**args)

    D = mk()
    out["hd_drag"] = D.ComputeHydrodynamicsEffects(0.01, q, vel6, False, [0.0, 0.0, 0.0]).clone()
    out["hd_local_vel"] = D.local_velocities.clone()
    out["hd_drag_planar"] = D.ComputeHydrodynamicsEffects(0.01, q_planar, vel6_planar, False, [0.0, 0.0, 0.0]).clone()
    out["hd_drag_current"] = D.ComputeHydrodynamicsEffects(0.01, q, vel6, True, [0.3, -0.2, 0.05]).clone()
    # per-env coefficients + drag scale + non-trivial offsets/scaling
    D2 = mk(dict(use_drag_scale_randomization=True, k_drag_min=1.0, k_drag_max=1.5),
            linear_damping_forward_speed=[0.1, 0.2, 0.0, 0.0, 0.0, 0.05], offset_linear_damping=0.5,
            offset_lin_forward_damping_speed=0.25, offset_nonlin_damping=0.125, scaling_damping=1.25)
    lin = torch.tensor([LIN] * N) * (1 + 0.1 * (torch.rand((N, 6), generator=g) * 2 - 1))
    quad = torch.tensor([QUAD] * N) * (1 + 0.1 * (torch.rand((N, 6), generator=g) * 2 - 1))
    kd = 1.0 + 0.5 * torch.rand((N, 1), generator=g)
    D2.linear_damping[:] = lin
    D2.quadratic_damping[:] = quad
    D2.drag_scale[:] = kd
    out.update(hd2_lin=lin, hd2_quad=quad, hd2_kdrag=kd)
    out["hd2_drag"] = D2.ComputeHydrodynamicsEffects(0.01, q, vel6, False, [0.0, 0.0, 0.0]).clone()
    out["hd2_drag_planar"] = D2.ComputeHydrodynamicsEffects(0.01, q_planar, vel6_planar, False, [0.0, 0.0, 0.0]).clone()

    # ---- A4/A5 thrusters
    def mkthr(L, R, cfg_extra=None, n_interp=1000):
        cfg = dict(THR_CFG)
        cfg.update(cfg_extra or {})
        return td.DynamicsFirstOrder(cfg, N, "cpu", 0.05, 0.02, n_interp, L, R, [0.0] * 5, [0.0] * 5, -1.0, 1.0)

    cmd = torch.rand((N, 2), generator=g) * 2 - 1
    cmd[0] = torch.tensor([0.73, 0.5005])
    cmd[1] = torch.tensor([0.0, 1.0])
    cmd[2] = torch.tensor([-1.0, -0.999])
    cmd[3] = torch.tensor([1.0 / 999.0, 3.0 / 999.0])    # half-integer indices after the affine map
    cmd[4] = torch.tensor([-1.5, 1.5])                   # out of range -> clamp
    out["thr_cmd"] = cmd
    for name, (L, R) in {"classic": (LUT_CLASSIC_L, LUT_CLASSIC_R), "live": (LUT_LIVE, LUT_LIVE),
                         "nominal": (LUT_NOMINAL, LUT_NOMINAL)}.items():
        T = mkthr(L, R)
        out[f"lut_{name}_left"] = T.y_linear_interp_left.clone()
        out[f"lut_{name}_right"] = T.y_linear_interp_right.clone()
        out[f"lut_{name}_points_left"] = torch.tensor(L)
        out[f"lut_{name}_points_right"] = torch.tensor(R)
        T.set_target_force(cmd)
        out[f"thr_{name}_before"] = T.thruster_forces_before_dynamics.clone()
        lag = []
        for _ in range(6):
            lag.append(T.update_forces().clone())
        out[f"thr_{name}_lag6"] = torch.stack(lag)           # (6, N, 6)
    # multipliers (separate + shared)
    Ts = mkthr(LUT_CLASSIC_L, LUT_CLASSIC_R, dict(use_thruster_randomization=True, use_separate_randomization=True))
    ml = 0.5 + torch.rand((N, 1), generator=g)
    mr = 0.5 + torch.rand((N, 1), generator=g)
    Ts.thruster_left_multiplier = ml
    Ts.thruster_right_multiplier = mr
    Ts.set_target_force(cmd)
    out.update(thr_mult_left=ml, thr_mult_right=mr, thr_sep_after=Ts.thruster_forces_after_randomization.clone())
    lag = [Ts.update_forces().clone() for _ in range(3)]
    out["thr_sep_lag3"] = torch.stack(lag)
    out["thr_alpha"] = torch.exp(torch.tensor(-0.02 / 0.05))
    np.savez(os.path.join(OUT, "force_modules.npz"), **t2n(out))
    print("force_modules.npz:", len(out), "arrays")


def disturbances():
    d = ref_shim.load_disturbances()
    g = gen()
    fcfg = dict(use_force_disturbance=True, use_constant_force=True, use_sinusoidal_force=True,
                force_const_min=0.0, force_const_max=2.5, force_sin_min=0.0, force_sin_max=2.5,
                force_min_freq=0.25, force_max_freq=3.0, force_min_shift=0.0, force_max_shift=100.0)
    tcfg = dict(use_torque_disturbance=True, use_constant_torque=True, use_sinusoidal_torque=True,
                torque_const_min=0.0, torque_const_max=1.0, torque_sin_min=0.0, torque_sin_max=1.0,
                torque_min_freq=0.25, torque_max_freq=3.0, torque_min_shift=0.0, torque_max_shift=100.0)
    UF = d.ForceDisturbance(fcfg, N, "cpu")
    TD = d.TorqueDisturbance(tcfg, N, "cpu")
    torch.manual_seed(7)
    ids = torch.arange(N)
    UF.generate_force(ids, N)
    TD.generate_torque(ids, N)
    root_pos = torch.zeros((N, 3))
    root_pos[:, :2] = torch.rand((N, 2), generator=g) * 60 - 30
    out = dict(root_pos=root_pos, f_const=UF.disturbance_forces_const.clone(), fxf=UF._force_x_freq.clone(),
               fyf=UF._force_y_freq.clone(), fxs=UF._force_x_shift.clone(), fys=UF._force_y_shift.clone(),
               famp=UF._force_amp.clone(), t_const=TD.disturbance_torques_const.clone(), tf=TD._torque_freq.clone(),
               ts=TD._torque_shift.clone(), tamp=TD._torque_amp.clone())
    out["forces"] = UF.get_disturbance_forces(root_pos).clone()
    out["torques"] = TD.get_torque_disturbance(root_pos).clone()
    out["ranges"] = torch.tensor([UF._const_min, UF._const_max, UF._sin_min, UF._sin_max])
    np.savez(os.path.join(OUT, "disturbances.npz"), **t2n(out))
    print("disturbances.npz")


def classic_task():
    """K steps of the classic CaptureXYTask + Penalties on a synthetic trajectory, with a reset batch
    in the middle  [SNAP/USV_capture_xy.py, SNAP/USV_task_rewards.py]."""
    core, rew, cap = ref_shim.load_classic()
    cfg = ref_shim.classic_yaml()
    g = gen()
    K = 6
    with ref_shim.quiet():
        task = cap.CaptureXYTask(cfg["env"]["task_parameters"], cfg["env"]["reward_parameters"], N, "cpu")
        pen = core.parse_data_dict(rew.Penalties(), cfg["env"]["penalties_parameters"])
    task._target_positions[:] = torch.rand((N, 2), generator=g) * 2 - 1
    pos = torch.rand((N, 2), generator=g) * 24 - 12
    yaw = (torch.rand(N, generator=g) * 2 - 1) * math.pi
    vel = torch.rand((N, 2), generator=g) * 3 - 1.5
    w = torch.rand(N, generator=g) * 2 - 1
    # crafted rows: inside tolerance & slow (goal), beyond kill distance, heading wrap cases
    pos[0] = task._target_positions[0] + torch.tensor([0.03, 0.02]); vel[0] = torch.tensor([0.01, 0.02])
    pos[1] = torch.tensor([-21.0, 0.0]); vel[1] = torch.tensor([0.0, 0.0])
    pos[2] = task._target_positions[2] + torch.tensor([0.03, 0.02]); vel[2] = torch.tensor([0.2, 0.0])   # in tol, too fast
    pos[3] = torch.tensor([5.0, 2.0]); yaw[3] = 3.1; task._target_positions[3] = torch.tensor([4.0, -2.0])
    pos[4] = torch.tensor([5.0, 2.0]); yaw[4] = 3.0; task._target_positions[4] = torch.tensor([-4.0, 1.0])
    pos[5] = torch.tensor([3.0, 0.0]); task._target_positions[5] = torch.tensor([0.0, 0.0])             # d = 3.0 zone
    pos[6] = torch.tensor([2.0, 0.0]); task._target_positions[6] = torch.tensor([0.0, 0.0])             # d = 2.0 zone
    pos[7] = torch.tensor([1.0, 0.0]); task._target_positions[7] = torch.tensor([0.0, 0.0])             # d = 1.0 zone
    out = dict(target=task._target_positions.clone())
    S = {k: [] for k in ("pos", "yaw", "vel", "w", "actions", "obs", "reward", "penalty", "die", "goal_reached",
                         "distance_reward", "alignment_reward", "speed_reward")}
    reset_ids = torch.tensor([1, 9, 17, 30])
    for k in range(K):
        actions = torch.rand((N, 2), generator=g) * 2.2 - 1.1
        if k == 3:
            task.reset(reset_ids)
            pos[reset_ids] = torch.rand((4, 2), generator=g) * 10 - 5
        heading = torch.stack([torch.cos(yaw), torch.sin(yaw)], 1)
        state = {"position": pos.clone(), "orientation": heading, "linear_velocity": vel.clone(),
                 "angular_velocity": w.clone()}
        with ref_shim.quiet():
            obs = task.get_state_observations(state, "local").clone()
            r = task.compute_reward(state, actions).clone()
            p = pen.compute_penalty(state, actions, 0.0).clone()
            die = task.update_kills(0).clone()
        for name, v in (("pos", pos), ("yaw", yaw), ("vel", vel), ("w", w), ("actions", actions), ("obs", obs),
                        ("reward", r), ("penalty", p), ("die", die), ("goal_reached", task._goal_reached),
                        ("distance_reward", task.distance_reward), ("alignment_reward", task.alignment_reward),
                        ("speed_reward", task.a)):
            S[name].append(v.clone())
        # synthetic motion
        pos = pos + 0.1 * vel
        yaw = yaw + 0.1 * w
        vel = vel * 0.9 + 0.1 * (torch.rand((N, 2), generator=g) * 3 - 1.5)
        w = w * 0.9 + 0.1 * (torch.rand(N, generator=g) * 2 - 1)
        vel[0] = torch.tensor([0.01, 0.02]); pos[0] = task._target_positions[0] + torch.tensor([0.03, 0.02])
    out.update({k: torch.stack(v) for k, v in S.items()})
    out["reset_step"] = np.int64(3)
    out["reset_ids"] = reset_ids
    np.savez(os.path.join(OUT, "capture_xy_classic.npz"), **t2n(out))
    print("capture_xy_classic.npz")


def gae():
    rl = ref_shim.load_rl_games()
    g = gen()
    out = {}
    for tag, (T, n) in {"a": (16, 32), "b": (16, 37), "c": (4, 2), "d": (1, 5)}.items():
        ns = types.SimpleNamespace(horizon_length=T, gamma=0.99, tau=0.95)
        rew = torch.randn((T, n, 1), generator=g) * 0.1
        val = torch.randn((T, n, 1), generator=g)
        dones = (torch.rand((T, n), generator=g) < 0.15).to(torch.uint8)
        last_d = (torch.rand((n,), generator=g) < 0.15).to(torch.uint8)
        last_v = torch.randn((n, 1), generator=g)
        if tag == "c":  # SURVEY appendix D.5
            rew = torch.tensor([[0.1, 0], [0.2, -0.1], [0, 0.3], [0.5, 0.05]]).unsqueeze(-1)
            val = torch.tensor([[1.0, 0.5], [0.9, 0.4], [1.1, 0.6], [0.8, 0.2]]).unsqueeze(-1)
            dones = torch.tensor([[0, 0], [0, 1], [0, 0], [1, 0]], dtype=torch.uint8)
            last_d = torch.tensor([0, 1], dtype=torch.uint8)
            last_v = torch.tensor([[0.7], [0.3]])
        adv = rl.a2c_common.A2CBase.discount_values(ns, last_d.float(), last_v, dones.float(), val, rew)
        out.update({f"{tag}_rewards": rew, f"{tag}_values": val, f"{tag}_dones": dones, f"{tag}_last_dones": last_d,
                    f"{tag}_last_values": last_v, f"{tag}_adv": adv, f"{tag}_returns": adv + val})
    np.savez(os.path.join(OUT, "gae.npz"), **t2n(out))
    print("gae.npz")


def ppo():
    """rl_games model / losses / optimizer on a seeded minibatch  [RLG/algos_torch/*, RLG/common/common_losses.py]"""
    rl = ref_shim.load_rl_games()
    torch.manual_seed(7)
    D, M = 13, 200
    with ref_shim.quiet():
        net = rl.model_builder.ModelBuilder().load({
            "model": {"name": "continuous_a2c_logstd"},
            "network": {"name": "actor_critic_mlp_dict", "separate": False,
                        "space": {"continuous": {"mu_activation": "None", "sigma_activation": "None", "mu_init": {"name": "default"},
                                                 "sigma_init": {"name": "const_initializer", "val": 0}, "fixed_sigma": True}},
                        "mlp": {"units": [128, 128], "activation": "tanh", "d2rl": False, "initializer": {"name": "default"},
                                "regularizer": {"name": "None"}}}})
        model = net.build({"actions_num": 2, "input_shape": {"state": (D,)}, "num_seqs": 1, "value_size": 1,
                           "normalize_value": True, "normalize_input": True, "normalize_input_keys": ["state"]})
    g = gen()
    with torch.no_grad():
        # biases are zero-initialised in the reference; perturb everything so every gradient path is exercised
        for prm in model.parameters():
            prm.add_(0.05 * torch.randn(prm.shape, generator=g))
        model.a2c_network.sigma.copy_(torch.tensor([-0.3, 0.2]))
    rms = model.running_mean_std.running_mean_std["state"]
    out = {"param_names": np.array([n for n, _ in model.named_parameters()])}
    obs0 = torch.randn((64, D), generator=g) * torch.linspace(0.5, 6.0, D) + torch.linspace(-2, 2, D)
    model.train()
    rms(obs0)                                  # one training-mode update of the obs normaliser
    vms = model.value_mean_std
    vms(torch.randn((64, 1), generator=g) * 2.0 + 0.5)
    model.eval()
    out.update(rms_update_obs=obs0, obs_mean=rms.running_mean.clone(), obs_var=rms.running_var.clone(), obs_count=rms.count.clone(),
               val_mean=vms.running_mean.clone(), val_var=vms.running_var.clone(), val_count=vms.count.clone())
    params0 = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    out["params0"] = params0.clone()
    obs = torch.randn((M, D), generator=g) * torch.linspace(0.5, 6.0, D) * 1.5 + torch.linspace(-2, 2, D)
    obs[0] = 100.0                              # exercises the +-5 clamp of the normaliser
    with torch.no_grad():
        r = model({"is_train": False, "prev_actions": None, "obs": {"state": obs.clone()}, "rnn_states": None})
    out.update(obs=obs, inf_mus=r["mus"], inf_sigmas=r["sigmas"], inf_values=r["values"], inf_actions=r["actions"],
               inf_neglogpacs=r["neglogpacs"])
    # a minibatch as prepare_dataset would hand it over
    actions = r["actions"] + 0.3 * torch.randn((M, 2), generator=g)
    actions[1] = torch.tensor([3.0, -3.0])
    old_nlp = r["neglogpacs"] + 0.2 * torch.randn(M, generator=g)
    adv = torch.randn(M, generator=g)
    old_v = torch.randn((M, 1), generator=g) * 0.5
    ret = old_v + torch.randn((M, 1), generator=g) * 0.5
    old_mu = r["mus"] + 0.05 * torch.randn((M, 2), generator=g)
    old_sigma = r["sigmas"] * (1 + 0.05 * torch.randn((M, 2), generator=g))
    out.update(mb_actions=actions, mb_old_neglogp=old_nlp, mb_adv=adv, mb_old_values=old_v, mb_returns=ret, mb_old_mu=old_mu,
               mb_old_sigma=old_sigma)
    opt = torch.optim.Adam(model.parameters(), 3e-4, eps=1e-08, weight_decay=0.0)
    ns = types.SimpleNamespace(bounds_loss_coef=1e-4)
    lr = 3e-4
    sched = rl.schedulers.AdaptiveScheduler(0.016)
    for it in range(3):
        res = model({"is_train": True, "prev_actions": actions, "obs": {"state": obs.clone()}})
        a_loss = rl.common_losses.actor_loss(old_nlp, res["prev_neglogp"], adv, True, 0.2)
        c_loss = rl.common_losses.critic_loss(model, old_v, res["values"], 0.2, ret, True)
        b_loss = rl.a2c_continuous.A2CAgent.bound_loss(ns, res["mus"])
        a_m, c_m, e_m, b_m = a_loss.mean(), c_loss.mean(), res["entropy"].mean(), b_loss.mean()
        loss = a_m + 0.5 * c_m * 0.5 - e_m * 0.0 + b_m * 1e-4
        for prm in model.parameters():
            prm.grad = None
        loss.backward()
        grads = torch.cat([p.grad.reshape(-1) for p in model.parameters()])
        kl = rl.torch_ext.policy_kl(res["mus"].detach(), res["sigmas"].detach(), old_mu, old_sigma, True)
        norm = torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        for gp in opt.param_groups:
            gp["lr"] = lr
        opt.step()
        new_lr, _ = sched.update(lr, 0.0, 0, 0, kl.item())
        out.update({f"it{it}_loss": loss.detach(), f"it{it}_a_loss": a_m.detach(), f"it{it}_c_loss": c_m.detach(),
                    f"it{it}_entropy": e_m.detach(), f"it{it}_b_loss": b_m.detach(), f"it{it}_kl": kl, f"it{it}_grads": grads.clone(),
                    f"it{it}_grad_norm": norm, f"it{it}_train_values": res["values"].detach(), f"it{it}_train_neglogp": res["prev_neglogp"].detach(),
                    f"it{it}_mus": res["mus"].detach(), f"it{it}_lr": torch.tensor(lr), f"it{it}_new_lr": torch.tensor(new_lr),
                    f"it{it}_params_after": torch.cat([p.detach().reshape(-1) for p in model.parameters()])})
        old_mu, old_sigma = res["mus"].detach(), res["sigmas"].detach()     # dataset.update_mu_sigma
        lr = new_lr
    np.savez(os.path.join(OUT, "ppo.npz"), **t2n(out))
    print("ppo.npz")


def ppo_epoch():
    """Two whole PPO epochs of the reference's own loop on fixed rollouts: ContinuousA2CBase.train_epoch -> prepare_dataset ->
    PPODataset -> calc_gradients / trancate_gradients_and_step / legacy adaptive-KL schedule, executed UNMODIFIED on a bare
    a2c_continuous.A2CAgent instance whose play_steps() hands over a recorded rollout (the env / experience buffer / writers of
    __init__ are Isaac Sim + config plumbing)  [RLG/common/a2c_common.py:1152-1320, common/datasets.py:25-77,
    algos_torch/a2c_continuous.py:78-196].  T=16, 64 actors, 2 minibatches of 512, 2 mini-epochs."""
    rl = ref_shim.load_rl_games()
    A2C, base = rl.a2c_continuous.A2CAgent, rl.a2c_common
    torch.manual_seed(11)
    D, T, NA, MB, ME = 13, 16, 64, 512, 2
    with ref_shim.quiet():
        net = rl.model_builder.ModelBuilder().load({
            "model": {"name": "continuous_a2c_logstd"},
            "network": {"name": "actor_critic_mlp_dict", "separate": False,
                        "space": {"continuous": {"mu_activation": "None", "sigma_activation": "None", "mu_init": {"name": "default"},
                                                 "sigma_init": {"name": "const_initializer", "val": 0}, "fixed_sigma": True}},
                        "mlp": {"units": [128, 128], "activation": "tanh", "d2rl": False, "initializer": {"name": "default"},
                                "regularizer": {"name": "None"}}}})
        model = net.build({"actions_num": 2, "input_shape": {"state": (D,)}, "num_seqs": 1, "value_size": 1,
                           "normalize_value": True, "normalize_input": True, "normalize_input_keys": ["state"]})
    g = gen()
    with torch.no_grad():
        for prm in model.parameters():
            prm.add_(0.03 * torch.randn(prm.shape, generator=g))
        model.a2c_network.sigma.copy_(torch.tensor([-0.2, 0.1]))
    rms = model.running_mean_std.running_mean_std["state"]
    vms = model.value_mean_std
    model.train()
    rms(torch.randn((256, D), generator=g) * torch.linspace(0.5, 4.0, D) + torch.linspace(-1, 1, D))
    vms(torch.randn((256, 1), generator=g) * 1.5 + 0.3)
    model.eval()
    ag = object.__new__(A2C)
    ag.__dict__.update(
        model=model, value_mean_std=vms, normalize_value=True, normalize_input=True, normalize_advantage=True, normalize_rms_advantage=False,
        is_rnn=False, has_central_value=False, has_value_loss=True, multi_gpu=False, mixed_precision=False, ppo=True, ppo_device="cpu",
        device="cpu", e_clip=0.2, clip_value=True, bound_loss_type="bound", bounds_loss_coef=1e-4, critic_coef=0.5, entropy_coef=0.0,
        truncate_grads=True, grad_norm=1.0, schedule_type="legacy", scheduler=rl.schedulers.AdaptiveScheduler(0.016), last_lr=1e-4,
        epoch_num=0, frame=0, mini_epochs_num=ME, gamma=0.99, tau=0.95, horizon_length=T, batch_size=T * NA, seq_len=4, zero_rnn_on_done=False,
        actor_loss_func=rl.common_losses.actor_loss, diagnostics=base.DefaultDiagnostics(),
        algo_observer=types.SimpleNamespace(after_steps=lambda: None), vec_env=types.SimpleNamespace(set_train_info=lambda *a: None),
        scaler=torch.cuda.amp.GradScaler(enabled=False),
        dataset=rl.datasets.PPODataset(T * NA, MB, False, False, "cpu", 4))
    ag.optimizer = torch.optim.Adam(model.parameters(), 1e-4, eps=1e-08, weight_decay=0.0)
    flat = lambda: torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    moments = lambda key: torch.cat([ag.optimizer.state[p][key].reshape(-1) for p in model.parameters()])
    out = dict(params0=flat(), obs_mean0=rms.running_mean.clone(), obs_var0=rms.running_var.clone(), obs_count0=rms.count.clone(),
               val_mean0=vms.running_mean.clone(), val_var0=vms.running_var.clone(), val_count0=vms.count.clone(),
               shape=np.array([D, T, NA, MB, ME]), lr0=np.float32(1e-4))
    for ep in range(2):
        # a rollout as play_steps leaves it in the experience buffer: (T, N, ...) tensors  [a2c_common.py:670-760]
        obses = torch.randn((T, NA, D), generator=g) * torch.linspace(0.5, 4.0, D) * (1.0 + 0.3 * ep) + torch.linspace(-1, 1, D)
        with torch.no_grad():
            r = model({"is_train": False, "prev_actions": None, "obs": {"state": obses.reshape(T * NA, D).clone()}, "rnn_states": None})
        actions, neglogpacs = r["actions"].reshape(T, NA, 2), r["neglogpacs"].reshape(T, NA)
        values, mus, sigmas = r["values"].reshape(T, NA, 1), r["mus"].reshape(T, NA, 2), r["sigmas"].reshape(T, NA, 2)
        rewards = (torch.randn((T, NA, 1), generator=g) * 0.05 + 0.02)
        dones = (torch.rand((T, NA), generator=g) < 0.08).to(torch.uint8)
        last_values = torch.randn((NA, 1), generator=g) * 0.5 + 0.3
        last_dones = (torch.rand(NA, generator=g) < 0.08).to(torch.uint8)
        advs = A2C.discount_values(ag, last_dones.float(), last_values, dones.float(), values, rewards)
        returns = advs + values
        fl = base.swap_and_flatten01
        batch = dict(obses={"state": fl(obses)}, returns=fl(returns), dones=fl(dones), values=fl(values), actions=fl(actions),
                     neglogpacs=fl(neglogpacs), mus=fl(mus).clone(), sigmas=fl(sigmas).clone(), played_frames=T * NA, step_time=0.0)
        ag.play_steps = lambda b=batch: dict(b)
        out.update({f"ep{ep}_obses": obses, f"ep{ep}_actions": actions, f"ep{ep}_neglogpacs": neglogpacs, f"ep{ep}_values": values,
                    f"ep{ep}_mus": mus.clone(), f"ep{ep}_sigmas": sigmas.clone(), f"ep{ep}_rewards": rewards, f"ep{ep}_dones": dones,
                    f"ep{ep}_last_values": last_values, f"ep{ep}_last_dones": last_dones, f"ep{ep}_returns": returns})
        # record what every minibatch step saw and left behind
        trace = []
        orig = A2C.train_actor_critic

        def traced(self, input_dict, _t=trace):
            lr_used = self.optimizer.param_groups[0]["lr"]
            res = orig(self, input_dict)
            _t.append(dict(a_loss=res[0].detach().clone(), c_loss=res[1].detach().clone(), kl=res[3].detach().clone(), lr=torch.tensor(lr_used),
                           mu=res[6].clone(), sigma=res[7].clone(), params=flat(), obs_mean=rms.running_mean.clone(),
                           obs_count=rms.count.clone()))
            return res

        ag.train_actor_critic = types.MethodType(traced, ag)
        with ref_shim.quiet():
            res = A2C.train_epoch(ag)
        ds = ag.dataset.values_dict
        out.update({f"ep{ep}_ds_old_values": ds["old_values"], f"ep{ep}_ds_returns": ds["returns"], f"ep{ep}_ds_advantages": ds["advantages"],
                    f"ep{ep}_ds_obs": ds["obs"]["state"], f"ep{ep}_ds_actions": ds["actions"], f"ep{ep}_ds_old_logp_actions": ds["old_logp_actions"],
                    f"ep{ep}_ds_mu_final": ds["mu"], f"ep{ep}_ds_sigma_final": ds["sigma"],
                    f"ep{ep}_params": flat(), f"ep{ep}_exp_avg": moments("exp_avg"), f"ep{ep}_exp_avg_sq": moments("exp_avg_sq"),
                    f"ep{ep}_last_lr": torch.tensor(ag.last_lr), f"ep{ep}_obs_mean": rms.running_mean.clone(), f"ep{ep}_obs_var": rms.running_var.clone(),
                    f"ep{ep}_obs_count": rms.count.clone(), f"ep{ep}_val_mean": vms.running_mean.clone(), f"ep{ep}_val_var": vms.running_var.clone(),
                    f"ep{ep}_val_count": vms.count.clone(), f"ep{ep}_obs_rms_training_after": torch.tensor(int(model.running_mean_std.training))})
        for k in trace[0]:
            if k != "params" or ep == 0:          # per-minibatch parameter snapshots for the first epoch only (fixture size)
                out[f"ep{ep}_mb_{k}"] = torch.stack([t[k] for t in trace])
        ag.epoch_num += 1
    np.savez(os.path.join(OUT, "ppo_epoch.npz"), **t2n(out))
    print("ppo_epoch.npz", {k: tuple(v.shape) for k, v in out.items() if k.startswith("ep1_mb")})


def variant_b():
    """Live CaptureXY with static obstacles (Variant B): spawn + potential-field build + K steps of obs / reward / kills,
    with a reset batch in the middle  [OIGE/tasks/USV/USV_capture_xy_static_obs.py, d_multi_gemini.py]."""
    live, dmap = ref_shim.load_live()
    cfg = ref_shim.live_yaml()
    NB, K = 12, 6
    torch.manual_seed(21)
    g = gen()
    with ref_shim.quiet():
        task = live.CaptureXYTask(cfg["env"]["task_parameters"], cfg["env"]["reward_parameters"], NB, "cpu", priv_dim=8)
    task._env = types.SimpleNamespace(_env_pos=torch.zeros((NB, 3)))
    ids = torch.arange(NB)
    out = {}
    with ref_shim.quiet():
        task.reset(ids)
        task.get_goals(ids, torch.zeros((NB, 3)), torch.zeros((NB, 4)))
        pos0, rot0 = task.get_spawns(ids, torch.zeros((NB, 3)), torch.zeros((NB, 4)))
    out.update(obstacles0=task.xunlian_pos[:, :, :2].clone(), field0=task.global_potential_field.clone(), target=task._target_positions.clone(),
               spawn_pos=pos0[:, :2].clone(), spawn_quat=rot0.clone())
    # intermediate products of the field builder for env 0..NB (fresh call, same obstacles): occupancy, sdf, cost
    occ, sdf = task.gpu_map.compute_occupancy_and_sdf(task.xunlian_pos[:, :, :2])
    cost = task.gpu_map.compute_cost_field_wavefront(occ, task._target_positions)
    out.update(occupancy0=occ.to(torch.uint8), sdf0=sdf.clone(), cost0=cost.clone())
    pos = pos0[:, :2].clone()
    yaw = (torch.rand(NB, generator=g) * 2 - 1) * math.pi
    vel = torch.rand((NB, 2), generator=g) * 2 - 1
    w = torch.rand(NB, generator=g) * 1.2 - 0.6
    # crafted rows: next to an obstacle (collision), inside the goal tolerance, far away, high-potential region
    obs_xy = task.xunlian_pos[:, :, :2]
    pos[0] = obs_xy[0, 0] + torch.tensor([0.9, 0.3])
    pos[1] = task._target_positions[1] + torch.tensor([0.3, -0.2])
    pos[2] = torch.tensor([-20.5, 1.0])
    pos[3] = obs_xy[3, 1] + torch.tensor([1.6, 0.2])
    S = {k: [] for k in ("pos", "yaw", "vel", "w", "prev_action", "priv", "obs", "reward", "die", "goal_reached", "done_success", "done_collision",
                         "distance_reward", "alignment_reward", "potential_shaping", "turn_hazard", "speed_reward", "angular_reward",
                         "heading_improve", "collision_penalty", "goal_reward", "danger", "potential")}
    reset_ids = torch.tensor([2, 5, 9])
    for k in range(K):
        if k == 3:
            with ref_shim.quiet():
                task.reset(reset_ids)
                p_new, _ = task.get_spawns(reset_ids, torch.zeros((NB, 3)), torch.zeros((NB, 4)))
            pos[reset_ids] = p_new[reset_ids, :2]
            out.update(obstacles1=task.xunlian_pos[:, :, :2].clone(), field1=task.global_potential_field.clone())
        heading = torch.stack([torch.cos(yaw), torch.sin(yaw)], 1)
        state = {"position": pos.clone(), "orientation": heading, "linear_velocity": vel.clone(), "angular_velocity": w.clone()}
        prev_action = torch.rand((NB, 2), generator=g) * 2 - 1
        priv = torch.rand((NB, 8), generator=g) * 2 - 1
        actions = torch.rand((NB, 2), generator=g)
        with ref_shim.quiet():
            obs = task.get_state_observations(state, "local", prev_action=prev_action, priv_tail=priv).clone()
            r = task.compute_reward(state, actions).clone()
            die = task.update_kills(0, state).clone()
        for name, v in (("pos", pos), ("yaw", yaw), ("vel", vel), ("w", w), ("prev_action", prev_action), ("priv", priv), ("obs", obs), ("reward", r),
                        ("die", die), ("goal_reached", task._goal_reached), ("done_success", task._done_success), ("done_collision", task._done_collision),
                        ("distance_reward", task.distance_reward), ("alignment_reward", task.alignment_reward),
                        ("potential_shaping", task.potential_shaping_reward), ("turn_hazard", task._turn_hazard_penalty),
                        ("speed_reward", task._speed_reward), ("angular_reward", task._angular_reward), ("heading_improve", task._heading_improve_reward),
                        ("collision_penalty", task.collision_penalty), ("goal_reward", task._goal_reward), ("danger", task._danger_factor),
                        ("potential", task._get_potential_values(state["position"]))):
            S[name].append(v.clone())
        pos = pos + 0.15 * vel
        yaw = yaw + 0.15 * w
        vel = vel * 0.9 + 0.1 * (torch.rand((NB, 2), generator=g) * 2 - 1)
        w = w * 0.8 + 0.2 * (torch.rand(NB, generator=g) * 1.2 - 0.6)
    out.update({k: torch.stack(v) for k, v in S.items()})
    out["reset_step"] = np.int64(3)
    out["reset_ids"] = reset_ids
    d = t2n(out)
    for k in ("field0", "field1", "sdf0", "cost0"):
        d[k] = d[k].astype(np.float32)
    np.savez_compressed(os.path.join(OUT, "capture_xy_live.npz"), **d)
    print("capture_xy_live.npz")


def variant_b_pd4():
    """The live CaptureXYTask with the 4-wide privileged tail (priv_dim = 4: obs = 3 + 20 + 2 + 4 = 29)
    [OIGE/tasks/USV/USV_core.py:23-52,127-170 ; USV_capture_xy_static_obs.py:193-299].  Same seed and call order as variant_b(), so
    obstacles / field / targets equal capture_xy_live.npz (asserted here) and only the states and the 29-wide observations are stored."""
    live, dmap = ref_shim.load_live()
    cfg = ref_shim.live_yaml()
    NB, K = 12, 3
    torch.manual_seed(21)
    g = gen()
    with ref_shim.quiet():
        task = live.CaptureXYTask(cfg["env"]["task_parameters"], cfg["env"]["reward_parameters"], NB, "cpu", priv_dim=4)
    task._env = types.SimpleNamespace(_env_pos=torch.zeros((NB, 3)))
    ids = torch.arange(NB)
    with ref_shim.quiet():
        task.reset(ids)
        task.get_goals(ids, torch.zeros((NB, 3)), torch.zeros((NB, 4)))
        pos0, rot0 = task.get_spawns(ids, torch.zeros((NB, 3)), torch.zeros((NB, 4)))
    G8 = np.load(os.path.join(OUT, "capture_xy_live.npz"))
    assert np.array_equal(G8["obstacles0"], task.xunlian_pos[:, :, :2].numpy()) and np.array_equal(G8["target"], task._target_positions.numpy())
    assert np.allclose(G8["field0"], task.global_potential_field.numpy(), rtol=0, atol=1e-6)
    pos = pos0[:, :2].clone()
    yaw = (torch.rand(NB, generator=g) * 2 - 1) * math.pi
    vel = torch.rand((NB, 2), generator=g) * 2 - 1
    w = torch.rand(NB, generator=g) * 1.2 - 0.6
    S = {k: [] for k in ("pos", "yaw", "vel", "w", "prev_action", "priv", "obs")}
    for k in range(K):
        heading = torch.stack([torch.cos(yaw), torch.sin(yaw)], 1)
        state = {"position": pos.clone(), "orientation": heading, "linear_velocity": vel.clone(), "angular_velocity": w.clone()}
        prev_action = torch.rand((NB, 2), generator=g) * 2 - 1
        priv = torch.rand((NB, 4), generator=g) * 2 - 1
        with ref_shim.quiet():
            obs = task.get_state_observations(state, "local", prev_action=prev_action, priv_tail=priv).clone()
        assert obs.shape == (NB, 29)
        for name, v in (("pos", pos), ("yaw", yaw), ("vel", vel), ("w", w), ("prev_action", prev_action), ("priv", priv), ("obs", obs)):
            S[name].append(v.clone())
        pos = pos + 0.15 * vel
        yaw = yaw + 0.15 * w
        vel = vel * 0.9 + 0.1 * (torch.rand((NB, 2), generator=g) * 2 - 1)
        w = w * 0.8 + 0.2 * (torch.rand(NB, generator=g) * 1.2 - 0.6)
    np.savez_compressed(os.path.join(OUT, "capture_xy_live_pd4.npz"), **t2n({k: torch.stack(v) for k, v in S.items()}))
    print("capture_xy_live_pd4.npz")


def live_virtual():
    """The live USVVirtual's own host-side chains that sit around the task (driven on a bare instance, no Isaac Sim):
    pre_physics_step action path (A12), get_observations privileged tail (B1), _apply_mass_driven_coupling (A11)
    [OIGE/tasks/USV_Virtual.py:837-1101]."""
    ref_shim.install()
    ref_shim.load_live()
    hs, hd, td = ref_shim.load_force_modules()
    dist = ref_shim.load_disturbances()
    with ref_shim.quiet():
        import omniisaacgymenvs.tasks.USV_Virtual as V
    cfg = ref_shim.live_yaml()
    env, dyn = cfg["env"], cfg["dynamics"]
    d = env["disturbances"]
    n = 24
    g = gen()
    out = {}

    def bare():
        me = object.__new__(V.USVVirtual)
        me._device, me._num_envs = "cpu", n
        me._task_cfg = cfg
        return me

    thr = dyn["thrusters"]
    def thrusters():
        with ref_shim.quiet():
            return td.DynamicsFirstOrder(d["thruster"], n, "cpu", thr["timeConstant"], cfg["sim"]["dt"],
                                         thr["interpolation"]["numberOfPointsForInterpolation"],
                                         thr["interpolation"]["interpolationPointsFromRealDataLeft"],
                                         thr["interpolation"]["interpolationPointsFromRealDataRight"],
                                         thr["leastSquareMethod"]["neg_cmd_coeff"], thr["leastSquareMethod"]["pos_cmd_coeff"],
                                         thr["cmd_lower_range"], thr["cmd_upper_range"])

    # ---- A12: action path, with and without the initial bias, with a reset subset ----------------------------------------
    for tag, count in (("bias", 0), ("nobias", 10 ** 9)):
        me = bare()
        me._env = types.SimpleNamespace(_world=types.SimpleNamespace(is_playing=lambda: True))
        me.reset_buf = torch.zeros(n, dtype=torch.long)
        me.reset_buf[[1, 7, 20]] = 1
        me.reset_idx = lambda ids: None
        me._discrete_actions = "Continuous"
        me.prev_thrust_cmds = torch.full((n, 2), 9.0)
        ap = env["action_processing"]
        me._initial_action_bias, me._initial_action_bias_steps = float(ap["initial_action_bias"]), int(ap["initial_action_bias_steps"])
        me._action_bias_step_count = count
        me._use_affine_thrust_mapping = bool(ap["use_affine_thrust_mapping"])
        me.AN = dist.NoisyActions(dict(d["actions"], add_noise_on_act=False))
        me.thrust_cmds_before_rect = torch.zeros((n, 2))
        me.thrust_cmds_unit = torch.zeros((n, 2))
        me.thrusters_dynamics = thrusters()
        actions = torch.rand((n, 2), generator=g) * 2 - 1           # VecEnvRLGames has already clamped to +-1
        with ref_shim.quiet():
            V.USVVirtual.pre_physics_step(me, actions.clone())
        out.update({f"act_{tag}_in": actions, f"act_{tag}_prev": me.prev_thrust_cmds.clone(), f"act_{tag}_before_rect": me.thrust_cmds_before_rect.clone(),
                    f"act_{tag}_unit": me.thrust_cmds_unit.clone(), f"act_{tag}_target": me.thrusters_dynamics.thruster_forces_before_dynamics.clone()})
    out["act_reset_ids"] = torch.tensor([1, 7, 20])
    out.update(lut_points_left=torch.tensor(thr["interpolation"]["interpolationPointsFromRealDataLeft"], dtype=torch.float64),
               lut_points_right=torch.tensor(thr["interpolation"]["interpolationPointsFromRealDataRight"], dtype=torch.float64),
               n_lut=torch.tensor(int(thr["interpolation"]["numberOfPointsForInterpolation"])),
               act_bias=torch.tensor(float(env["action_processing"]["initial_action_bias"]), dtype=torch.float64))

    # ---- A11 + B1: mass -> coupling -> privileged tail, for the three encodings ------------------------------------------
    for mode in ("minmax", "centered", "raw"):
        me = bare()
        with ref_shim.quiet():
            me.MDD = dist.MassDistributionDisturbances(d["mass"], n, "cpu")
            me.hydrodynamics = hd.HydrodynamicsObject(d["drag"], n, "cpu", 1000, -9.81, dyn["hydrodynamics"]["linear_damping"],
                                                      dyn["hydrodynamics"]["quadratic_damping"], dyn["hydrodynamics"]["linear_damping_forward_speed"],
                                                      0.0, 0.0, 0.0, 1.0, 0.0, 1.0, 0.3, -10.0)
            me.thrusters_dynamics = thrusters()
        ids = torch.arange(n)
        torch.manual_seed(33)
        me.MDD.randomize_masses(ids, n)
        me.MDD.platforms_mass[0, 0] = me.MDD._base_mass
        me.MDD.platforms_mass[1, 0] = me.MDD._max_mass
        me._mass_driven_coupling_enabled = True
        me._mass_driven_couple_drag = me._mass_driven_couple_thruster = me._mass_driven_couple_yaw_inertia = True
        me._k_drag_min, me._k_drag_max = float(d["drag"]["k_drag_min"]), float(d["drag"]["k_drag_max"])
        me._thruster_rand_for_priv = float(d["thruster"]["thruster_rand"])
        me._k_iz_min, me._k_iz_max = float(d["inertia"]["k_Iz_min"]), float(d["inertia"]["k_Iz_max"])
        me.mass_ratio_r = torch.zeros((n, 1))
        me.k_Iz = torch.ones((n, 1))
        me._base_inertias0 = torch.ones((n, 9))
        me._maybe_init_base_inertias0 = lambda: None
        me._heron = types.SimpleNamespace(name="heron")
        with ref_shim.quiet():
            V.USVVirtual._apply_mass_driven_coupling(me, ids)
        captured = {}
        me.update_state = lambda: None
        me.current_state = None
        me._masscom_obs_source, me._mass_obs_mode, me._com_obs_mode = "sim", d["mass"]["mass_obs_mode"], d["mass"]["com_obs_mode"]
        hsd = dyn["hydrostatics"]
        me._com_obs_scale = [float(hsd["box_length"]), float(hsd["box_width"]), float(max(hsd["heron_zero_height"], 1.0))]
        me._priv_dim = 8
        me._privileged_params_mode, me._privileged_params_nominal = mode, 1.0
        me._use_drag_scale_randomization_priv = me._use_thruster_randomization_priv = me._use_yaw_inertia_randomization = True
        me.obs_buf = {}
        me._observation_frame = "local"
        me.prev_thrust_cmds = torch.zeros((n, 2))
        me.task = types.SimpleNamespace(get_state_observations=lambda st, fr, mass, com, prev_action=None, priv_tail=None:
                                        captured.update(priv=priv_tail.clone()) or torch.zeros((n, 33)))
        with ref_shim.quiet():
            V.USVVirtual.get_observations(me)
        out.update({f"priv_{mode}": captured["priv"]})
        # the ablation source: base mass / CoM encodings and neutral dynamics parameters for every env  (USV_Virtual.py:840-880)
        me._masscom_obs_source = "base"
        with ref_shim.quiet():
            V.USVVirtual.get_observations(me)
        out.update({f"priv_base_{mode}": captured["priv"]})
        me._masscom_obs_source = "sim"
        if mode == "minmax":
            out.update(cpl_mass=me.MDD.platforms_mass[:, 0].clone(), cpl_com=me.MDD.platforms_CoM.clone(), cpl_kdrag=me.hydrodynamics.drag_scale[:, 0].clone(),
                       cpl_thr=me.thrusters_dynamics.thruster_multiplier[:, 0].clone(), cpl_kiz=me.k_Iz[:, 0].clone(),
                       cpl_com_scale=torch.tensor(me._com_obs_scale))
    np.savez_compressed(os.path.join(OUT, "live_virtual.npz"), **t2n(out))
    print("live_virtual.npz")


def tier3():
    """GoToPose / KeepXY / TrackXYVelocity (SURVEY row T): the tasks cannot run end-to-end in the reference (broken wiring), so
    their methods are called one by one on a bare task object with `_task_data` pre-allocated (N,20), as SURVEY 8(c) prescribes.
    KeepXYTask.compute_reward reads an undefined `self.positionposition` (USV_keep_xy.py:137): the attribute is set on the instance,
    the source is not touched."""
    ref_shim.install()
    ref_shim.load_live()
    with ref_shim.quiet():
        import omniisaacgymenvs.tasks.USV.USV_go_to_pose as gtp
        import omniisaacgymenvs.tasks.USV.USV_keep_xy as kxy
        import omniisaacgymenvs.tasks.USV.USV_track_xy_velocity as txv
    n, K = 16, 5
    g = gen()
    out = {}
    specs = [("gotopose", gtp.GoToPoseTask, dict(name="GoToPose", position_tolerance=0.5, kill_after_n_steps_in_tolerance=3, max_spawn_dist=3.0,
                                                 min_spawn_dist=0.3, kill_dist=10.0),
              dict(name="GoToPose", position_reward_mode="exponential", heading_reward_mode="exponential", position_exponential_reward_coeff=0.25,
                   heading_exponential_reward_coeff=0.25, position_scale=1.0, heading_scale=5.0, sig_gain=3.0)),
             ("gotopose_sq", gtp.GoToPoseTask, dict(name="GoToPose", position_tolerance=0.5, kill_after_n_steps_in_tolerance=3, kill_dist=10.0),
              dict(name="GoToPose", position_reward_mode="square", heading_reward_mode="linear", position_scale=2.0, heading_scale=3.0, sig_gain=2.0)),
             ("keepxy", kxy.KeepXYTask, dict(name="KeepXY", position_tolerance=0.1, kill_after_n_steps_in_tolerance=500, kill_dist=8.0, boundary_cost=25.0),
              dict(name="KeepXY", reward_mode="exponential", exponential_reward_coeff=0.25)),
             ("keepxy_lin", kxy.KeepXYTask, dict(name="KeepXY", kill_dist=8.0), dict(name="KeepXY", reward_mode="linear")),
             ("trackxyvel", txv.TrackXYVelocityTask, dict(name="TrackXYVelocity", lin_vel_tolerance=0.3, kill_after_n_steps_in_tolerance=2, kill_dist=9.0,
                                                          goal_random_velocity=0.75),
              dict(name="TrackXYVelocity", reward_mode="exponential", exponential_reward_coeff=0.25))]
    for tag, cls, tp, rp in specs:
        with ref_shim.quiet():
            task = cls(tp, rp, n, "cpu", priv_dim=8)
        task._task_data = torch.zeros((n, 20))
        task.positionposition = None
        ids = torch.arange(n)
        target = torch.rand((n, 2), generator=g) * 2 - 1
        if hasattr(task, "_target_positions"):
            task._target_positions[:] = target
        if hasattr(task, "_target_headings"):
            task._target_headings[:] = torch.rand(n, generator=g) * 2 * math.pi
            out[f"{tag}_target_heading"] = task._target_headings.clone()
        if hasattr(task, "_target_velocities"):
            task._target_velocities[:] = torch.rand((n, 2), generator=g) * 1.5 - 0.75
            out[f"{tag}_target_vel"] = task._target_velocities.clone()
        task.reset(ids)
        pos = torch.rand((n, 2), generator=g) * 8 - 4
        pos[0] = target[0] + torch.tensor([0.1, 0.05])          # inside the tolerance
        pos[1] = target[1] + torch.tensor([11.0, 0.0])          # beyond kill_dist
        yaw = (torch.rand(n, generator=g) * 2 - 1) * math.pi
        vel = torch.rand((n, 2), generator=g) * 2 - 1
        vel[0] = torch.tensor([0.02, -0.03])
        if tag == "trackxyvel":
            vel[2] = task._target_velocities[2] + torch.tensor([0.05, -0.05])   # inside lin_vel_tolerance
        w = torch.rand(n, generator=g) * 1.2 - 0.6
        S = {k: [] for k in ("pos", "yaw", "vel", "w", "prev_action", "priv", "actions", "obs", "reward", "die", "goal_reached")}
        for k in range(K):
            state = {"position": pos.clone(), "orientation": torch.stack([torch.cos(yaw), torch.sin(yaw)], 1),
                     "linear_velocity": vel.clone(), "angular_velocity": w.clone()}
            actions = torch.rand((n, 2), generator=g) * 2 - 1
            priv = torch.rand((n, 8), generator=g) * 2 - 1
            with ref_shim.quiet():
                obs = task.get_state_observations(state, "local", prev_action=actions, priv_tail=priv).clone()
                r = task.compute_reward(state, actions).clone()
                die = (task.update_kills() if tag == "trackxyvel" else task.update_kills(0)).clone()
            for name, v in (("pos", pos), ("yaw", yaw), ("vel", vel), ("w", w), ("prev_action", actions), ("priv", priv), ("actions", actions),
                            ("obs", obs), ("reward", r), ("die", die), ("goal_reached", task._goal_reached)):
                S[name].append(v.clone())
            pos = pos + 0.1 * vel
            yaw = yaw + 0.1 * w
            vel = vel * 0.95
            vel[3:] = vel[3:] + 0.05 * (torch.rand((n - 3, 2), generator=g) * 2 - 1)
        out.update({f"{tag}_{k}": torch.stack(v) for k, v in S.items()})
        out[f"{tag}_target"] = target
    np.savez_compressed(os.path.join(OUT, "tier3_tasks.npz"), **t2n(out))
    print("tier3_tasks.npz")


def classic_curriculum():
    """Spawn-distance / kill-distance curriculum of the classic CaptureXYTask (rows A18, A19: optional, linear in `step`)
    [SNAP/USV_capture_xy.py:231-275,330-394]."""
    core, rew, cap = ref_shim.load_classic()
    cfg = ref_shim.classic_yaml()
    tp = dict(cfg["env"]["task_parameters"], spawn_curriculum=True, spawn_curriculum_min_dist=0.2, spawn_curriculum_max_dist=3.0,
              spawn_curriculum_kill_dist=30.0, spawn_curriculum_warmup=250, spawn_curriculum_end=1000, min_spawn_dist=0.5,
              max_spawn_dist=11.0, kill_dist=20.0)
    n = 64
    with ref_shim.quiet():
        task = cap.CaptureXYTask(tp, cfg["env"]["reward_parameters"], n, "cpu")
    steps = [0.0, 100.0, 249.9375, 250.0, 400.5, 625.0, 1000.0, 1000.0625, 1500.0]
    ids = torch.arange(n)
    dist = torch.linspace(15.0, 35.0, n)
    out = dict(steps=torch.tensor(steps, dtype=torch.float64), dist=dist, params=torch.tensor([0.2, 3.0, 30.0, 250, 1000, 0.5, 11.0, 20.0], dtype=torch.float64))
    U, R, D = [], [], []
    for st in steps:
        torch.manual_seed(int(st * 16))
        u = torch.rand(n)                                        # the first draw of get_spawns is r
        torch.manual_seed(int(st * 16))
        with ref_shim.quiet():
            pos, _ = task.get_spawns(ids, torch.zeros((n, 3)), torch.zeros((n, 4)), step=st)
        R.append(torch.norm(pos[:, :2] - task._target_positions, dim=1))
        U.append(u)
        task.position_dist = dist.clone()
        task.current_state = {"linear_velocity": torch.ones((n, 2))}
        task._goal_reached[:] = 0
        with ref_shim.quiet():
            D.append(task.update_kills(st).clone())
    out.update(u=torch.stack(U), r=torch.stack(R), die=torch.stack(D))
    np.savez(os.path.join(OUT, "classic_curriculum.npz"), **t2n(out))
    print("classic_curriculum.npz")


def loopz():
    """The loopz PPO learner: MLPEncode actor / critic, squashed Gaussian, RolloutStorage.compute_returns and PPO._train_step of the
    UNMODIFIED reference (OIGE/algo/ppo/{module,storage,ppo}.py) in the configuration rlgames_train_loopz.py:784-842 builds."""
    import tempfile

    import torch.nn as nn
    from torch.distributions import Normal

    ref_shim.install()
    import omniisaacgymenvs.algo.ppo.module as M
    import omniisaacgymenvs.algo.ppo.ppo as P

    D, MD, T, N = 33, 8, 8, 48
    torch.manual_seed(11)
    g = gen()

    def build(n_epochs, n_mb, lr, max_norm, state=None, sampling="in_order"):
        actor = M.Actor(M.MLPEncode_wrap([128, 128], nn.LeakyReLU, D, 2, nn.Tanh, False, speed_dim=3, mass_dim=MD, mass_latent_dim=8,
                                         mass_encoder_shape=[64, 16]),
                        M.SquashedGaussianDiagonalCovariance(2, 0.3, action_scale=1.0), "cpu")
        critic = M.Critic(M.MLPEncode_wrap([128, 128], nn.LeakyReLU, D, 1, speed_dim=3, mass_dim=MD, mass_latent_dim=8,
                                           mass_encoder_shape=[64, 16]), "cpu")
        with ref_shim.quiet():
            ppo_ = P.PPO(actor=actor, critic=critic, num_envs=N, num_transitions_per_env=T, num_learning_epochs=n_epochs, gamma=0.997,
                         lam=0.95, num_mini_batches=n_mb, device="cpu", log_dir=tempfile.mkdtemp(), mini_batch_sampling=sampling,
                         learning_rate=lr, max_grad_norm=max_norm)
        if state is not None:
            with torch.no_grad():
                for p_, s_ in zip([*actor.parameters(), *critic.parameters()], state):
                    p_.copy_(s_)
        return actor, critic, ppo_

    actor, critic, ppo_ = build(4, 4, 5e-4, 0.5)
    with torch.no_grad():
        for prm in [*actor.parameters(), *critic.parameters()]:
            prm.add_(0.05 * torch.randn(prm.shape, generator=g))
        actor.distribution.std.copy_(torch.tensor([0.3, 0.45]))
    plist = [*actor.parameters(), *critic.parameters()]
    state0 = [p_.detach().clone() for p_ in plist]
    out = {"param_names": np.array([n for n, _ in actor.architecture.named_parameters()] + ["distribution.std"] +
                                   [n for n, _ in critic.architecture.named_parameters()]),
           "param_sizes": np.array([p_.numel() for p_ in plist]), "params0": torch.cat([p_.reshape(-1) for p_ in state0])}

    # ---- inference: means / values / log-prob of a sample with known noise / evaluate() of given actions -------------------
    Mrows = 200
    obs = torch.randn((Mrows, D), generator=g) * torch.linspace(0.3, 2.0, D)
    obs[:, -MD:] = torch.rand((Mrows, MD), generator=g) * 2 - 1
    with torch.no_grad():
        means = actor.architecture.architecture(obs)
        values = critic.predict(obs)
        std = actor.distribution.std.reshape(2)
        noise = torch.randn((Mrows, 2), generator=g)
        u = means + std * noise
        logp_u = actor.distribution._log_prob_from_u(Normal(means, std), u)
        acts = torch.tanh(u) * actor.distribution.action_scale
        eval_actions = torch.rand((Mrows, 2), generator=g) * 2 - 1
        eval_actions[0] = torch.tensor([1.0, -1.0])            # the atanh clamp
        eval_actions[1] = torch.tensor([0.999999, 0.0])
        (logp_eval, ent_eval), mean_eval = actor.evaluate(obs, eval_actions)
    out.update(inf_obs=obs, inf_means=means, inf_values=values, inf_noise=noise, inf_u=u, inf_logp_u=logp_u, inf_actions=acts,
               eval_actions=eval_actions, eval_logp=logp_eval, eval_entropy=ent_eval, eval_means=mean_eval)

    # ---- a rollout in the storage + compute_returns ------------------------------------------------------------------------
    st = ppo_.storage
    roll_obs = torch.randn((T + 1, N, D), generator=g) * torch.linspace(0.3, 2.0, D)
    roll_obs[:, :, -MD:] = torch.rand((T + 1, N, MD), generator=g) * 2 - 1
    rewards = torch.randn((T, N), generator=g) * 0.05
    rewards[2, 5] = float("nan")                                # sanitised to 0 by add_transitions
    dones = (torch.rand((T, N), generator=g) < 0.12)
    for t in range(T):
        with torch.no_grad():
            m_ = actor.architecture.architecture(roll_obs[t])
            nz = torch.randn((N, 2), generator=g)
            u_ = m_ + std * nz
            a_ = torch.tanh(u_) * actor.distribution.action_scale
            lp_ = actor.distribution._log_prob_from_u(Normal(m_, std), u_)
            v_ = critic.predict(roll_obs[t])
        st.add_transitions(roll_obs[t].numpy(), roll_obs[t].numpy(), a_, rewards[t].numpy(), dones[t].numpy(), v_, lp_)
    with torch.no_grad():
        last_values = critic.predict(roll_obs[T])
    st.compute_returns(last_values, ppo_.gamma, ppo_.lam)
    out.update(roll_obs=roll_obs, roll_rewards=rewards, roll_dones=dones.to(torch.uint8), roll_actions=st.actions.clone(),
               roll_log_prob=st.actions_log_prob.clone(), roll_values=st.values.clone(), roll_last_values=last_values,
               roll_returns=st.returns.clone(), roll_advantages=st.advantages.clone(), gamma=np.float32(0.997), lam=np.float32(0.95))
    fields = ["actor_obs", "critic_obs", "rewards", "actions", "dones", "actions_log_prob", "values", "returns", "advantages"]
    filled = {k: getattr(st, k).clone() for k in fields}

    def fill(p2):
        for k in fields:
            setattr(p2.storage, k, filled[k].clone())
        p2.storage.step = T

    # ---- raw gradient of ONE minibatch (lr = 0, no clipping) over rows [0, 96) and over the full batch ----------------------
    for tag, n_mb in (("full", 1), ("quarter", 4)):
        a2, c2, p2 = build(1, n_mb, 0.0, 1e9, state0)
        fill(p2)
        if n_mb == 4:       # only the FIRST minibatch: stop after one step
            orig = p2.batch_sampler
            p2.batch_sampler = lambda k, _o=orig: (b for i, b in enumerate(_o(k)) if i == 0)
        with ref_shim.quiet():
            vl, sl, _ = p2._train_step()
        out[f"grad_{tag}"] = torch.cat([p_.grad.reshape(-1) for p_ in [*a2.parameters(), *c2.parameters()]])
        out[f"grad_{tag}_value_loss"] = np.float32(vl)
        out[f"grad_{tag}_surrogate"] = np.float32(sl)

    # ---- one full update as the live script configures it: 4 epochs x 4 in-order minibatches, lr 5e-4, clip 0.5 ---------------
    a3, c3, p3 = build(4, 4, 5e-4, 0.5, state0)
    fill(p3)
    with ref_shim.quiet():
        vl, sl, _ = p3._train_step()
    out.update(update_params_after=torch.cat([p_.detach().reshape(-1) for p_ in [*a3.parameters(), *c3.parameters()]]),
               update_value_loss=np.float32(vl), update_surrogate=np.float32(sl))
    a3.distribution.enforce_minimum_std(torch.tensor([0.05, 0.5]))
    out["min_std_after"] = a3.distribution.std.detach().clone()
    np.savez_compressed(os.path.join(OUT, "loopz_ppo.npz"), **t2n(out))
    print("loopz_ppo.npz")


def loopz_md4():
    """The 4-wide privileged tail (cfg.yaml mass_dim: 4, obs 29): forward, evaluate and one raw minibatch gradient of the reference."""
    import tempfile

    import torch.nn as nn

    ref_shim.install()
    import omniisaacgymenvs.algo.ppo.module as M
    import omniisaacgymenvs.algo.ppo.ppo as P

    D, MD, T, N = 29, 4, 4, 40
    torch.manual_seed(12)
    g = gen()
    arch = dict(speed_dim=3, mass_dim=MD, mass_latent_dim=8, mass_encoder_shape=[64, 16])
    actor = M.Actor(M.MLPEncode_wrap([128, 128], nn.LeakyReLU, D, 2, nn.Tanh, False, **arch),
                    M.SquashedGaussianDiagonalCovariance(2, 0.3, action_scale=1.0), "cpu")
    critic = M.Critic(M.MLPEncode_wrap([128, 128], nn.LeakyReLU, D, 1, **arch), "cpu")
    with ref_shim.quiet():
        ppo_ = P.PPO(actor=actor, critic=critic, num_envs=N, num_transitions_per_env=T, num_learning_epochs=1, gamma=0.997, lam=0.95,
                     num_mini_batches=1, device="cpu", log_dir=tempfile.mkdtemp(), mini_batch_sampling="in_order", learning_rate=0.0,
                     max_grad_norm=1e9)
    with torch.no_grad():
        for prm in [*actor.parameters(), *critic.parameters()]:
            prm.add_(0.05 * torch.randn(prm.shape, generator=g))
        actor.distribution.std.copy_(torch.tensor([0.25, 0.4]))
    plist = [*actor.parameters(), *critic.parameters()]
    out = {"params0": torch.cat([p_.detach().reshape(-1) for p_ in plist]), "param_sizes": np.array([p_.numel() for p_ in plist])}
    obs = torch.randn((T, N, D), generator=g)
    flat = obs.reshape(-1, D)
    with torch.no_grad():
        means = actor.architecture.architecture(flat)
        values = critic.predict(flat)
    actions = torch.tanh(torch.randn((T * N, 2), generator=g) * 1.2)
    with torch.no_grad():
        (logp, _), _ = actor.evaluate(flat, actions)
    st = ppo_.storage
    st.actor_obs.copy_(obs); st.critic_obs.copy_(obs); st.actions.copy_(actions.view(T, N, 2))
    st.actions_log_prob.copy_((logp + 0.05 * torch.randn(logp.shape, generator=g)).view(T, N, 1))
    st.values.copy_((values + 0.05 * torch.randn(values.shape, generator=g)).view(T, N, 1))
    st.returns.copy_(st.values + 0.5 * torch.randn(st.values.shape, generator=g))
    st.advantages.copy_(torch.randn(st.advantages.shape, generator=g))
    st.step = T
    cols = {k: getattr(st, k).clone() for k in ("actor_obs", "actions", "actions_log_prob", "values", "returns", "advantages")}
    with ref_shim.quiet():
        vl, sl, _ = ppo_._train_step()
    out.update(means=means, values=values, eval_logp=logp, grad=torch.cat([p_.grad.reshape(-1) for p_ in plist]),
               value_loss=np.float32(vl), surrogate=np.float32(sl), **{"st_" + k: v for k, v in cols.items()})
    np.savez_compressed(os.path.join(OUT, "loopz_ppo_md4.npz"), **t2n(out))
    print("loopz_ppo_md4.npz")


def config_branches():
    """Configuration branches of the live USVVirtual that no shipped YAML takes (VERDICT r01 "missing" 6), each driven on the reference's
    own code: mass-driven coupling with PARTIAL target lists (OIGE/tasks/USV_Virtual.py:988-1040), the independent episode-wise k_Iz
    draw in linear and log space (:153-170), and the legacy disc-shaped CoM randomisation (OIGE/tasks/USV/USV_disturbances.py:108-124).
    torch.rand cannot be matched by the kernels' Philox streams, so the uniforms the reference consumed are recorded beside its
    outputs (re-drawn from the same torch seed in the same call order) and the oracle / kernels are fed those."""
    ref_shim.install()
    ref_shim.load_live()
    hs, hd, td = ref_shim.load_force_modules()
    dist = ref_shim.load_disturbances()
    with ref_shim.quiet():
        import omniisaacgymenvs.tasks.USV_Virtual as V
    cfg = ref_shim.live_yaml()
    env, dyn = cfg["env"], cfg["dynamics"]
    d = env["disturbances"]
    n = 24
    out = {}
    thr = dyn["thrusters"]
    ids = torch.arange(n)
    for tag, targets in (("drag", ("drag_scale",)), ("thr_kiz", ("thruster", "yaw_inertia")), ("kiz", ("yaw_inertia",))):
        me = object.__new__(V.USVVirtual)
        me._device, me._num_envs, me._task_cfg = "cpu", n, cfg
        with ref_shim.quiet():
            me.MDD = dist.MassDistributionDisturbances(d["mass"], n, "cpu")
            me.hydrodynamics = hd.HydrodynamicsObject(d["drag"], n, "cpu", 1000, -9.81, dyn["hydrodynamics"]["linear_damping"],
                                                      dyn["hydrodynamics"]["quadratic_damping"], dyn["hydrodynamics"]["linear_damping_forward_speed"],
                                                      0.0, 0.0, 0.0, 1.0, 0.0, 1.0, 0.3, -10.0)
            me.thrusters_dynamics = td.DynamicsFirstOrder(d["thruster"], n, "cpu", thr["timeConstant"], cfg["sim"]["dt"],
                                                          thr["interpolation"]["numberOfPointsForInterpolation"],
                                                          thr["interpolation"]["interpolationPointsFromRealDataLeft"],
                                                          thr["interpolation"]["interpolationPointsFromRealDataRight"],
                                                          thr["leastSquareMethod"]["neg_cmd_coeff"], thr["leastSquareMethod"]["pos_cmd_coeff"],
                                                          thr["cmd_lower_range"], thr["cmd_upper_range"])
        torch.manual_seed(41)
        me.MDD.randomize_masses(ids, n)
        me.MDD.platforms_mass[0, 0] = me.MDD._base_mass
        me.MDD.platforms_mass[1, 0] = me.MDD._max_mass
        # what the independent randomisations left behind before the coupling runs (sentinels: the coupling must leave a
        # non-target untouched)
        me.hydrodynamics.drag_scale[:, 0] = 1.25
        me.thrusters_dynamics.thruster_multiplier[:] = 0.875
        me.thrusters_dynamics.thruster_left_multiplier[:] = 0.75
        me.thrusters_dynamics.thruster_right_multiplier[:] = 1.125
        me.k_Iz = torch.full((n, 1), 1.375)
        me._mass_driven_coupling_enabled = True
        me._mass_driven_couple_drag = "drag_scale" in targets
        me._mass_driven_couple_thruster = "thruster" in targets
        me._mass_driven_couple_yaw_inertia = "yaw_inertia" in targets
        me._k_drag_min, me._k_drag_max = float(d["drag"]["k_drag_min"]), float(d["drag"]["k_drag_max"])
        me._thruster_rand_for_priv = float(d["thruster"]["thruster_rand"])
        me._k_iz_min, me._k_iz_max = float(d["inertia"]["k_Iz_min"]), float(d["inertia"]["k_Iz_max"])
        me.mass_ratio_r = torch.zeros((n, 1))
        me._base_inertias0 = torch.ones((n, 9))
        me._maybe_init_base_inertias0 = lambda: None
        me._heron = types.SimpleNamespace(name="heron")
        with ref_shim.quiet():
            V.USVVirtual._apply_mass_driven_coupling(me, ids)
        tdm = me.thrusters_dynamics
        out.update({f"cpl_{tag}_mass": me.MDD.platforms_mass[:, 0].clone(), f"cpl_{tag}_kdrag": me.hydrodynamics.drag_scale[:, 0].clone(),
                    f"cpl_{tag}_thr_l": tdm.thruster_left_multiplier.reshape(n, -1)[:, 0].clone(),
                    f"cpl_{tag}_thr_r": tdm.thruster_right_multiplier.reshape(n, -1)[:, 0].clone(), f"cpl_{tag}_kiz": me.k_Iz[:, 0].clone()})
    f64 = lambda v: torch.tensor(v, dtype=torch.float64)        # configuration scalars are Python doubles in the reference
    out.update(cpl_mass_base=f64(float(d["mass"]["base_mass"])), cpl_mass_max=f64(float(d["mass"]["max_mass"])),
               cpl_kdrag_rng=f64([float(d["drag"]["k_drag_min"]), float(d["drag"]["k_drag_max"])]),
               cpl_thr_a=f64(float(d["thruster"]["thruster_rand"])),
               cpl_kiz_rng=f64([float(d["inertia"]["k_Iz_min"]), float(d["inertia"]["k_Iz_max"])]))

    # ---- independent k_Iz  (_sample_k_iz)
    for space in ("linear", "log"):
        me = object.__new__(V.USVVirtual)
        me._device = "cpu"
        me._k_iz_min, me._k_iz_max, me._k_iz_sample_space = 0.8, 1.7, space
        torch.manual_seed(43)
        k = V.USVVirtual._sample_k_iz(me, n)
        torch.manual_seed(43)
        u = torch.rand((n, 1), dtype=torch.float32)
        out.update({f"kiz_{space}": k[:, 0].clone(), f"kiz_{space}_u": u[:, 0].clone()})
    out["kiz_rng"] = f64([0.8, 1.7])

    # ---- legacy disc-shaped CoM  (MDD._randomize_com without com_displacement_xyz)
    mcfg = dict(d["mass"], add_mass_disturbances=True, CoM_max_displacement=0.12, base_com=[0.02, -0.01, 0.03])
    mcfg.pop("com_displacement_xyz", None)
    with ref_shim.quiet():
        mdd = dist.MassDistributionDisturbances(mcfg, n, "cpu")
    torch.manual_seed(47)
    mdd._randomize_com(ids, n)
    torch.manual_seed(47)
    ur = torch.rand((n,), dtype=torch.float32)
    uth = torch.rand((n,), dtype=torch.float32)
    out.update(com_disc=mdd.platforms_CoM.clone(), com_disc_u_r=ur, com_disc_u_theta=uth, com_disc_max=f64(0.12),
               com_disc_base=f64([0.02, -0.01, 0.03]))
    np.savez_compressed(os.path.join(OUT, "config_branches.npz"), **t2n(out))
    print("config_branches.npz")


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)
    force_modules()
    disturbances()
    classic_task()
    gae()
    ppo()
    ppo_epoch()
    variant_b()
    variant_b_pd4()
    live_virtual()
    tier3()
    classic_curriculum()
    loopz()
    loopz_md4()
    config_branches()


if __name__ == "__main__":
    if len(sys.argv) > 1:                 # python oracle/make_golden.py live_virtual tier3 ...
        os.makedirs(OUT, exist_ok=True)
        torch.set_num_threads(1)
        for name in sys.argv[1:]:
            globals()[name]()
    else:
        main()
