"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

Import shim that lets the *unmodified* reference modules of a reference checkout
(the directory named by the environment variable USV_REFERENCE_ROOT) be executed on
CPU (no Isaac Sim, no pytorch3d, no gym).  The reference is not part of this
repository.  The shim is used by ``oracle/make_golden*.py`` to generate the committed
fixtures in ``tests/golden/`` and by the tests that compare with the reference
directly, which skip when USV_REFERENCE_ROOT is unset.

What is faked (SURVEY.md section 8(c)):
  * ``omni.*``, ``pxr.*``, ``carb``, ``gym``, ``matplotlib``, ``ray``, ``tensorboardX``,
    ``cv2``, ``envpool`` -> permissive dummy modules (attribute access fabricates
    sub-modules for lower-case names and dummy classes for Capitalised names).
  * ``pytorch3d.transforms.quaternion_to_matrix`` -> a restatement of the public
    PyTorch3D formula (real-first (w,x,y,z), two_s = 2/|q|^2).  PyTorch3D is a
    third-party dependency of the reference that is neither vendored nor pinned
    (reference setup.py:12-18) -> "parity unpinned at that boundary"; we pin the
    restatement ourselves in tests/test_oracle_cpu.py.
  * the classic snapshot files (``811*/USV_core.py`` ...) are alias-loaded under the
    module names they import each other by.
"""
from __future__ import annotations

import contextlib
import glob
import importlib.abc
import importlib.machinery
import importlib.util
import io
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("USV_REFERENCE_ROOT", "")

_FAKE_ROOTS = (
    "omni", "pxr", "carb", "gym", "matplotlib", "ray", "tensorboardX", "cv2",
    "envpool", "gymnasium", "hydra", "omegaconf", "wandb",
)


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "omniisaacgymenvs"))


def snapshot_dir() -> str:
    hits = sorted(glob.glob(os.path.join(REFERENCE_ROOT, "811*")))
    if not hits:
        raise FileNotFoundError("classic snapshot folder (811*) not found under reference root")
    return hits[0]


class _DummyMeta(type):
    def __getattr__(cls, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Dummy


class _Dummy(metaclass=_DummyMeta):
    """Permissive stand-in for any class coming from a faked module."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Dummy()

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Dummy()


class _FakeModule(types.ModuleType):
    def __call__(self, *a, **k):  # e.g. gym.envs.register(...)
        return _Dummy()

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        full = f"{self.__name__}.{name}"
        if name[:1].isupper():
            cls = type(name, (_Dummy,), {"__module__": self.__name__})
            setattr(self, name, cls)
            return cls
        mod = sys.modules.get(full)
        if mod is None:
            mod = _FakeModule(full)
            mod.__path__ = []
            sys.modules[full] = mod
        setattr(self, name, mod)
        return mod


class _FakeFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path=None, target=None):
        if fullname.split(".")[0] in _FAKE_ROOTS:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        mod = _FakeModule(spec.name)
        mod.__path__ = []
        return mod

    def exec_module(self, module):
        pass


def _quaternion_to_matrix(quaternions):
    """Restatement of pytorch3d.transforms.quaternion_to_matrix (public formula)."""
    import torch

    r, i, j, k = torch.unbind(quaternions, -1)
    two_s = 2.0 / (quaternions * quaternions).sum(-1)
    o = torch.stack(
        (
            1 - two_s * (j * j + k * k),
            two_s * (i * j - k * r),
            two_s * (i * k + j * r),
            two_s * (i * j + k * r),
            1 - two_s * (i * i + k * k),
            two_s * (j * k - i * r),
            two_s * (i * k - j * r),
            two_s * (j * k + i * r),
            1 - two_s * (i * i + j * j),
        ),
        -1,
    )
    return o.reshape(quaternions.shape[:-1] + (3, 3))


_installed = False


def install() -> None:
    """Install the fake modules and put the reference on sys.path (idempotent)."""
    global _installed
    if _installed:
        return
    if not reference_available():
        raise FileNotFoundError(f"no reference checkout at USV_REFERENCE_ROOT={REFERENCE_ROOT!r}: set it to the reference project's root")
    sys.meta_path.insert(0, _FakeFinder())

    p3d = types.ModuleType("pytorch3d")
    p3d.__path__ = []
    p3dt = types.ModuleType("pytorch3d.transforms")
    p3dt.quaternion_to_matrix = _quaternion_to_matrix
    p3d.transforms = p3dt
    sys.modules["pytorch3d"] = p3d
    sys.modules["pytorch3d.transforms"] = p3dt

    # a real-enough gym.spaces for rl_games / the task classes
    gym = _FakeModule("gym")
    gym.__path__ = []
    spaces = _FakeModule("gym.spaces")
    spaces.__path__ = []

    class Box:
        def __init__(self, low, high, shape=None, dtype=None):
            import numpy as np

            self.low = np.asarray(low, dtype=np.float32)
            self.high = np.asarray(high, dtype=np.float32)
            self.shape = tuple(shape) if shape is not None else self.low.shape
            self.dtype = dtype or np.float32

    class Dict:
        def __init__(self, spaces_):
            self.spaces = dict(spaces_)

        def __getitem__(self, k):
            return self.spaces[k]

        def items(self):
            return self.spaces.items()

    class Discrete:
        def __init__(self, n):
            self.n = n

    class Tuple(tuple):
        def __new__(cls, seq):
            return super().__new__(cls, seq)

    spaces.Box, spaces.Dict, spaces.Discrete, spaces.Tuple = Box, Dict, Discrete, Tuple
    gym.spaces = spaces
    sys.modules["gym"] = gym
    sys.modules["gym.spaces"] = spaces

    # visual-marker helpers pull in pxr types at import time -> pre-seed fakes
    for name in ("omniisaacgymenvs.utils.pin", "omniisaacgymenvs.utils.arrow",
                 "omniisaacgymenvs.utils.shape_utils"):
        fm = _FakeModule(name)
        fm.__path__ = []
        sys.modules[name] = fm

    for p in (REFERENCE_ROOT, os.path.join(REFERENCE_ROOT, "rl_games")):
        if p not in sys.path:
            sys.path.insert(0, p)
    _installed = True


def _load_as(modname: str, path: str):
    spec = importlib.util.spec_from_file_location(modname, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[modname] = mod
    spec.loader.exec_module(mod)
    return mod


@contextlib.contextmanager
def quiet():
    """The reference prints on every step; swallow it."""
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        yield


def load_force_modules():
    """Returns (Hydrostatics, Hydrodynamics, ThrusterDynamics) reference modules."""
    install()
    import omniisaacgymenvs.envs.USV.Hydrostatics as hs
    import omniisaacgymenvs.envs.USV.Hydrodynamics as hd
    import omniisaacgymenvs.envs.USV.ThrusterDynamics as td

    return hs, hd, td


def load_disturbances():
    install()
    import omniisaacgymenvs.tasks.USV.USV_disturbances as d

    return d


def load_classic():
    """Alias-load the classic (Variant A) snapshot: returns (core, rewards, capture_xy)."""
    install()
    snap = snapshot_dir()
    saved = {k: sys.modules.get(k) for k in (
        "omniisaacgymenvs.tasks.USV.USV_core",
        "omniisaacgymenvs.tasks.USV.USV_task_rewards",
    )}
    import omniisaacgymenvs.tasks.USV  # noqa: F401  (package must exist first)
    import omniisaacgymenvs.tasks.USV.USV_task_parameters  # noqa: F401

    with quiet():
        core = _load_as("omniisaacgymenvs.tasks.USV.USV_core", os.path.join(snap, "USV_core.py"))
        rew = _load_as("omniisaacgymenvs.tasks.USV.USV_task_rewards", os.path.join(snap, "USV_task_rewards.py"))
        cap = _load_as("usv_classic_capture_xy", os.path.join(snap, "USV_capture_xy.py"))
    # keep private handles, restore whatever was there so the live variant can still load
    for k, v in saved.items():
        if v is not None:
            sys.modules[k] = v
        else:
            sys.modules.pop(k, None)
    return core, rew, cap


def load_live():
    """The live (Variant B) task: CaptureXYTask with static obstacles + BatchedMapGPU; returns (task_module, map_module)."""
    install()
    for k in ("omniisaacgymenvs.tasks.USV.USV_core", "omniisaacgymenvs.tasks.USV.USV_task_rewards"):
        sys.modules.pop(k, None)                 # make sure the LIVE core/rewards are imported, not the snapshot aliases
    with quiet():
        import omniisaacgymenvs.tasks.USV.USV_capture_xy_static_obs as live
        import omniisaacgymenvs.tasks.USV.d_multi_gemini as dmap
    return live, dmap


def live_yaml() -> dict:
    import re
    import yaml

    path = os.path.join(REFERENCE_ROOT, "omniisaacgymenvs", "cfg", "task", "USV", "IROS2024", "USV_Virtual_CaptureXY_SysID-TEST.yaml")
    with open(path) as f:
        txt = f.read()
    txt = re.sub(r"\$\{resolve_default:([^,]+),\$\{[^}]*\}\}", r"\1", txt)
    return yaml.safe_load(txt)


def load_rl_games():
    """Returns the reference rl_games modules used on the PPO path."""
    install()
    from rl_games.common import a2c_common, datasets, common_losses, schedulers
    from rl_games.algos_torch import models, running_mean_std, torch_ext, model_builder, a2c_continuous

    return types.SimpleNamespace(
        a2c_common=a2c_common, datasets=datasets, common_losses=common_losses,
        schedulers=schedulers, models=models, running_mean_std=running_mean_std,
        torch_ext=torch_ext, model_builder=model_builder, a2c_continuous=a2c_continuous,
    )


def classic_yaml() -> dict:
    import yaml

    path = os.path.join(snapshot_dir(), "USV_Virtual_CaptureXY_SysID-TEST.yaml")
    with open(path) as f:
        txt = f.read()
    return yaml.safe_load(txt)
