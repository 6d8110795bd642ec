"""USVSysIDVecEnv (history wrapper of the DAgger / SysID path) over a scripted base env: against the reference's own class when the
reference tree is present, and against the expected window contents always  [ref: omniisaacgymenvs/envs/usv_raisim_vecenv.py:387-617]."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from omniisaacgymenvs_loop_b200.envs.usv_raisim_vecenv import USVSysIDVecEnv
from oracle import ref_shim

N, D, PRIV, H = 5, 9, 4, 6
# the reference project is not part of this repository: point USV_REFERENCE_ROOT at a checkout of it to run these
needs_reference = pytest.mark.skipif(not ref_shim.reference_available(), reason="needs a checkout of the reference project (USV_REFERENCE_ROOT)")


class ScriptedBase:
    """VecEnvRLGames-shaped: reset() / step(a) -> ({'obs': {'state': ...}}, rew, resets, extras), attribute _task."""

    def __init__(self, seed):
        self.g = torch.Generator().manual_seed(seed)
        self.num_envs = N
        self._task = SimpleNamespace(num_envs=N, num_observations=D, num_actions=2, device="cpu", rl_device="cpu")
        self.k = 0

    def _obs(self):
        return {"obs": {"state": torch.randn((N, D), generator=self.g)}, "states": torch.zeros((N, 0))}

    def reset(self):
        return self._obs()

    def step(self, a):
        self.k += 1
        done = (torch.rand(N, generator=self.g) < 0.3).long()
        return self._obs(), torch.rand(N, generator=self.g), done, {}


@pytest.mark.parametrize("fill", ["zeros", "repeat"])
def test_history_window_contents(fill):
    env = USVSysIDVecEnv(ScriptedBase(3), history_len=H, priv_dim=PRIV, fill_history_on_reset=fill)
    assert env.obs_nonpriv_dim == D - PRIV
    env.reset()
    frames = [env.observe_nonpriv(as_numpy=False).clone()]
    want = torch.zeros((N, H, D - PRIV))
    want[:] = frames[0].unsqueeze(1) if fill == "repeat" else 0.0
    want[:, -1] = frames[0]
    assert torch.equal(env.observe_history(as_numpy=False).reshape(N, H, -1), want)
    for _ in range(10):
        _, dones = env.step(torch.zeros((N, 2)))
        cur = env.observe_nonpriv(as_numpy=False)
        want = torch.roll(want, -1, 1)
        want[:, -1] = cur
        if fill == "repeat":
            want[dones.bool()] = cur[dones.bool()].unsqueeze(1).expand(-1, H, -1)
        # "zeros": the reference zeroes a copy, the old frames stay (usv_raisim_vecenv.py:613)
        assert torch.equal(env.observe_history(as_numpy=False).reshape(N, H, -1), want)
        s = env.observe_sysid_obs()
        assert s.shape == (N, H * (D - PRIV) + D - PRIV) and s.dtype == np.float32
        assert np.array_equal(s[:, -(D - PRIV):], cur.numpy()) and np.array_equal(s[:, : H * (D - PRIV)], want.reshape(N, -1).numpy())
        assert torch.equal(env.get_priv_tail(), env.observe(as_numpy=False)[:, -PRIV:])
        assert torch.equal(env.get_masscom(), env.observe(as_numpy=False)[:, -4:])
    with pytest.raises(ValueError):
        USVSysIDVecEnv(ScriptedBase(1), history_len=0)
    with pytest.raises(ValueError):
        USVSysIDVecEnv(ScriptedBase(1), priv_dim=D)
    env8 = USVSysIDVecEnv(ScriptedBase(1), history_len=3, priv_dim=8)
    env8.reset()
    assert torch.equal(env8.get_masscom(), env8.observe(as_numpy=False)[:, -8:-4])        # 8-wide tail: mass + CoM come first


@needs_reference
@pytest.mark.parametrize("fill", ["zeros", "repeat"])
def test_history_matches_reference_class(fill):
    ref_shim.install()
    import omniisaacgymenvs.envs.usv_raisim_vecenv as R
    ours = USVSysIDVecEnv(ScriptedBase(8), history_len=H, priv_dim=PRIV, fill_history_on_reset=fill)
    ref = R.USVSysIDVecEnv(ScriptedBase(8), history_len=H, priv_dim=PRIV, fill_history_on_reset=fill)
    ours.reset(); ref.reset()
    for _ in range(12):
        a = np.zeros((N, 2), dtype=np.float32)
        r1, d1 = ours.step(a)
        r2, d2 = ref.step(a)
        assert np.array_equal(r1, r2) and np.array_equal(d1, d2)
        assert np.array_equal(ours.observe_sysid_obs(), ref.observe_sysid_obs())
        assert np.array_equal(ours.observe_history(), ref.observe_history()) and np.array_equal(ours.observe_nonpriv(), ref.observe_nonpriv())
        assert torch.equal(ours.get_priv_tail(), ref.get_priv_tail())


def test_obs_storage_surface_and_generators():
    """ObsStorage [ref: omniisaacgymenvs/algo/ppo/storage.py:4-42]: time-major flattening, in-order blocks, overflow, shuffle = a partition."""
    from omniisaacgymenvs_loop_b200.algo.ppo import ObsStorage
    T, n, hd, lat = 3, 4, 5, 2
    st = ObsStorage(n, T, [hd], [lat], "cpu")
    g = torch.Generator().manual_seed(0)
    obs = torch.randn((T, n, hd), generator=g)
    tgt = torch.randn((T, n, lat), generator=g)
    for t in range(T):
        st.add_obs(obs[t].numpy() if t % 2 else obs[t], tgt[t])                  # numpy or tensor
    with pytest.raises(AssertionError):
        st.add_obs(obs[0], tgt[0])
    got = list(st.mini_batch_generator_inorder(4))
    assert len(got) == 4
    for b, (o, e) in enumerate(got):
        assert torch.equal(o, obs.reshape(-1, hd)[3 * b:3 * b + 3]) and torch.equal(e, tgt.reshape(-1, lat)[3 * b:3 * b + 3])
    rows = torch.cat([o for o, _ in st.mini_batch_generator_shuffle(4, generator=torch.Generator().manual_seed(1))])
    assert rows.shape == (12, hd) and torch.equal(rows.sort(dim=0).values, obs.reshape(-1, hd).sort(dim=0).values)
    assert len(list(st.mini_batch_generator_shuffle(5))) == 6                    # 12 // 5 = 2 rows per batch, drop_last
    st.clear()
    assert st.step == 0


@needs_reference
def test_obs_storage_matches_reference_class():
    """A cleared and refilled ObsStorage yields the reference class's in-order minibatches."""
    from omniisaacgymenvs_loop_b200.algo.ppo import ObsStorage
    ref_shim.install()
    import omniisaacgymenvs.algo.ppo.storage as RS
    T, n, hd, lat = 3, 4, 5, 2
    g = torch.Generator().manual_seed(0)
    obs = torch.randn((T, n, hd), generator=g)
    tgt = torch.randn((T, n, lat), generator=g)
    st = ObsStorage(n, T, [hd], [lat], "cpu")
    for t in range(T):
        st.add_obs(obs[t], tgt[t])
    st.clear()
    ref = RS.ObsStorage(n, T, [hd], [lat], "cpu")
    for t in range(T):
        st.add_obs(obs[t], tgt[t]); ref.add_obs(obs[t].numpy(), tgt[t])
    for (a, b), (c, d) in zip(st.mini_batch_generator_inorder(2), ref.mini_batch_generator_inorder(2)):
        assert torch.equal(a, c) and torch.equal(b, d)
