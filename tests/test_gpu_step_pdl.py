"""The fused step is launched as a programmatic dependent of the previous kernel in the stream (csrc/usv_step.cu, launch_pdl): it may
start while that kernel still runs and must not touch global memory before griddepcontrol.wait.  Torch kernels on the same stream write
the actions, the state of the first and last envs and some reset flags just before a step, and read obs / reward / done just after it;
some steps follow each other with nothing in between.  Everything must equal the same sequence with a device synchronize between every
pair of launches."""
import pytest
import torch

from omniisaacgymenvs_loop_b200.config import UsvEnvConfig
from omniisaacgymenvs_loop_b200.engine import FusedUsvEnv

DEV = "cuda:0"
K = 12


def _run(n, acts, sync):
    env = FusedUsvEnv(UsvEnvConfig(max_episode_length=7).full_dr(), n, DEV)
    a = torch.zeros((n, 2), device=DEV)                 # the buffer every step reads its actions from
    vx, r = env.field_view("USV_S_VX"), env.field_view("USV_S_R")
    seen_obs = torch.empty((K, n, 13), device=DEV)
    seen_rew = torch.empty((K, n), device=DEV)
    seen_done = torch.empty((K, n), dtype=torch.long, device=DEV)
    fence = torch.cuda.synchronize if sync else (lambda: None)
    for k in range(K):
        # k % 3 == 0: kernels before and after the step; 1: before only; 2: after only -- so steps 3m+1 and 3m+2 follow each other directly
        if k % 3 != 2:
            torch.neg(acts[k], out=a)
            fence()
            vx[:4].add_(0.25)                            # first 128 envs (first wave of CTAs)
            fence()
            r[-4:].sub_(0.125)                           # last tile rows (last wave)
            fence()
            env.reset_buf[k::997].fill_(1)
            fence()
        env.step(a)
        fence()
        if k % 3 != 1:
            torch.mul(env.obs, 1.0, out=seen_obs[k])
            fence()
            torch.mul(env.rew, 1.0, out=seen_rew[k])
            fence()
            torch.mul(env.reset_buf, 1, out=seen_done[k])
            fence()
    torch.cuda.synchronize()
    env.check_finite()
    return seen_obs, seen_rew, seen_done, env.state, env.consts


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4096 + 3, (1 << 20) + 37])
def test_step_pdl_orders_with_neighbouring_torch_kernels(n):
    g = torch.Generator(device=DEV).manual_seed(11)
    acts = [torch.rand((n, 2), device=DEV, generator=g) * 2 - 1 for _ in range(K)]
    got = _run(n, acts, sync=False)
    want = _run(n, acts, sync=True)
    for name, x, y in zip(("obs", "reward", "done", "state", "consts"), got, want):
        if name in ("obs", "reward", "done"):
            for k in range(K):
                if k % 3 != 1:
                    assert torch.equal(x[k], y[k]), (name, k)
        else:
            assert torch.equal(x, y), name
