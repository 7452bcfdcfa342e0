"""TEST INFRASTRUCTURE ONLY -- import shim that lets the *unmodified* reference
hot-path modules (installed under oracle/_ref by oracle/install_reference.py) load here.

habitat-lab's packages cannot be imported as packages here (gym, omegaconf,
hydra, habitat_sim ... are absent, and ``habitat_baselines/__init__.py``
imports every trainer).  The hot-path files themselves contain no arithmetic
outside torch/numpy, so they load verbatim once ``sys.modules`` is pre-seeded
with arithmetic-free stubs (SURVEY.md section 8c).  Nothing in here is product code:
``tests/golden/make_golden.py`` (fixture generation), bench.py's reference
arms and the reference arm's contract test use it.
"""
from __future__ import annotations

import importlib
import importlib.machinery
import logging
import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pick_root() -> str:
    """HB200_REFERENCE_ROOT when set, else the install oracle/install_reference.py made under oracle/_ref/ (git-ignored)."""
    return os.environ.get("HB200_REFERENCE_ROOT") or os.path.join(_REPO, "oracle", "_ref")


REFERENCE_ROOT = _pick_root()
HB = os.path.join(REFERENCE_ROOT, "habitat-baselines", "habitat_baselines")


def reference_available() -> bool:
    return os.path.isdir(HB)


# ----------------------------------------------------------------------------
# gym.spaces stub (shape / dtype / low / high containers only)
# ----------------------------------------------------------------------------
def _make_gym():
    import numpy as np

    gym = types.ModuleType("gym")
    spaces = types.ModuleType("gym.spaces")

    class Space:
        def __init__(self, shape=None, dtype=None):
            self.shape = None if shape is None else tuple(shape)
            self.dtype = None if dtype is None else np.dtype(dtype)

    class Box(Space):
        def __init__(self, low, high, shape=None, dtype=np.float32):
            if shape is None:
                shape = np.asarray(low).shape
            super().__init__(shape, dtype)
            self.low = np.full(self.shape, low, dtype=self.dtype)
            self.high = np.full(self.shape, high, dtype=self.dtype)

    class Discrete(Space):
        def __init__(self, n):
            super().__init__((), np.int64)
            self.n = int(n)

    class MultiDiscrete(Space):
        def __init__(self, nvec):
            self.nvec = np.asarray(nvec, dtype=np.int64)
            super().__init__(self.nvec.shape, np.int64)

    class Dict(Space):
        def __init__(self, spaces=None, **kw):
            super().__init__(None, None)
            import collections

            self.spaces = collections.OrderedDict(spaces or {})
            self.spaces.update(kw)

        def __getitem__(self, k):
            return self.spaces[k]

        def __iter__(self):
            return iter(self.spaces)

        def __contains__(self, k):
            return k in self.spaces

        def keys(self):
            return self.spaces.keys()

        def items(self):
            return self.spaces.items()

        def values(self):
            return self.spaces.values()

        def __len__(self):
            return len(self.spaces)

    class Tuple(Space):
        def __init__(self, spaces):
            super().__init__(None, None)
            self.spaces = tuple(spaces)

    for c in (Space, Box, Discrete, MultiDiscrete, Dict, Tuple):
        setattr(spaces, c.__name__, c)
    gym.spaces = spaces
    gym.Space = Space
    gym.Env = type("Env", (), {})
    gym.Wrapper = type("Wrapper", (), {})
    return gym, spaces


def _ns(name: str, path: str | None = None) -> types.ModuleType:
    """A namespace-style module whose heavy __init__ is skipped."""
    m = types.ModuleType(name)
    m.__path__ = [path] if path else []
    m.__spec__ = importlib.machinery.ModuleSpec(name, None, is_package=True)
    if path:
        m.__spec__.submodule_search_locations = [path]
    sys.modules[name] = m
    return m


def _mod(name: str, **attrs) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    parent, _, leaf = name.rpartition(".")
    if parent and parent in sys.modules:
        setattr(sys.modules[parent], leaf, m)
    return m


_INSTALLED = False


def install() -> None:
    """Seed sys.modules so `import habitat_baselines.rl.ppo.ppo` etc. work."""
    global _INSTALLED
    if _INSTALLED:
        return
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")

    if "gym" not in sys.modules:
        gym, spaces = _make_gym()
        sys.modules["gym"] = gym
        sys.modules["gym.spaces"] = spaces

    # ---- habitat (arithmetic-free stubs) ------------------------------
    habitat = _ns("habitat")
    habitat.logger = logging.getLogger("habitat")
    _ns("habitat.utils")
    _ns("habitat.core")
    _ns("habitat.tasks")
    _ns("habitat.tasks.nav")
    _ns("habitat.utils.visualizations")

    class _RangeContext:
        def __init__(self, *_a, **_k):
            pass

        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

        def __call__(self, fn):  # used as a decorator by utils/common.py:314
            return fn

    noop = lambda *a, **k: None  # noqa: E731
    _mod(
        "habitat.utils.profiling_wrapper",
        range_push=noop,
        range_pop=noop,
        configure=noop,
        on_start_step=noop,
        RangeContext=_RangeContext,
    )

    # same semantics as HL/core/registry.py:43-69 (name -> class dict)
    import collections

    class _Singleton(type):
        _inst: dict = {}

        def __call__(cls, *a, **k):
            if cls not in cls._inst:
                cls._inst[cls] = super().__call__(*a, **k)
            return cls._inst[cls]

    class Registry(metaclass=_Singleton):
        mapping = collections.defaultdict(dict)

        @classmethod
        def _register_impl(cls, _type, to_register, name, assert_type=None):
            def wrap(to_register):
                register_name = to_register.__name__ if name is None else name
                cls.mapping[_type][register_name] = to_register
                return to_register

            if to_register is None:
                return wrap
            return wrap(to_register)

        @classmethod
        def _get_impl(cls, _type, name):
            return cls.mapping[_type].get(name, None)

    _mod("habitat.core.registry", Registry=Registry)
    _mod("habitat.core.utils", Singleton=_Singleton)
    _mod("habitat.core.dataset", Episode=type("Episode", (), {}))
    _mod(
        "habitat.core.spaces",
        EmptySpace=type("EmptySpace", (sys.modules["gym.spaces"].Space,), {}),
        ActionSpace=type("ActionSpace", (sys.modules["gym.spaces"].Dict,), {}),
    )
    _mod("habitat.utils.visualizations.utils", images_to_video=noop)

    def _sensor(uuid):
        return type("S_" + uuid, (), {"cls_uuid": uuid})

    _mod(
        "habitat.tasks.nav.nav",
        EpisodicCompassSensor=_sensor("compass"),
        EpisodicGPSSensor=_sensor("gps"),
        HeadingSensor=_sensor("heading"),
        ImageGoalSensor=_sensor("imagegoal"),
        IntegratedPointGoalGPSAndCompassSensor=_sensor("pointgoal_with_gps_compass"),
        PointGoalSensor=_sensor("pointgoal"),
        ProximitySensor=_sensor("proximity"),
    )
    _mod("habitat.tasks.nav.object_nav_task", ObjectGoalSensor=_sensor("objectgoal"))
    _mod(
        "habitat.tasks.nav.instance_image_nav_task",
        InstanceImageGoalSensor=_sensor("instance_imagegoal"),
    )

    # ---- habitat_baselines as a namespace over the real sources ------
    _ns("habitat_baselines", HB)
    for sub in ("common", "rl", "rl/ddppo", "rl/models", "utils"):
        _ns("habitat_baselines." + sub.replace("/", "."), os.path.join(HB, sub))
    _mod(
        "habitat_baselines.common.tensorboard_utils",
        TensorboardWriter=type("TensorboardWriter", (), {}),
    )
    for opt in ("attr", "cv2", "PIL", "PIL.Image"):
        try:
            importlib.import_module(opt)
        except Exception:  # pragma: no cover
            m = _mod(opt)
            if opt == "attr":
                m.s = lambda *a, **k: (lambda c: c)
                m.ib = lambda *a, **k: None
            if opt == "PIL":
                m.Image = _mod("PIL.Image")

    _INSTALLED = True


def ref():
    """Return a namespace of the reference hot-path classes."""
    install()
    ns = types.SimpleNamespace()
    from habitat_baselines.common.rollout_storage import RolloutStorage
    from habitat_baselines.common.tensor_dict import TensorDict
    from habitat_baselines.rl.ddppo.algo.ddppo import DDPPO
    from habitat_baselines.rl.ddppo.policy.resnet_policy import (
        PointNavResNetNet,
        PointNavResNetPolicy,
        ResNetEncoder,
    )
    from habitat_baselines.rl.ddppo.policy.running_mean_and_var import RunningMeanAndVar
    from habitat_baselines.rl.models.rnn_state_encoder import (
        build_pack_info_from_dones,
        build_rnn_build_seq_info,
        build_rnn_state_encoder,
    )
    from habitat_baselines.rl.ppo.policy import PointNavBaselinePolicy
    from habitat_baselines.rl.ppo.ppo import PPO

    ns.RolloutStorage = RolloutStorage
    ns.TensorDict = TensorDict
    ns.DDPPO = DDPPO
    ns.PPO = PPO
    ns.PointNavResNetPolicy = PointNavResNetPolicy
    ns.PointNavResNetNet = PointNavResNetNet
    ns.ResNetEncoder = ResNetEncoder
    ns.RunningMeanAndVar = RunningMeanAndVar
    ns.PointNavBaselinePolicy = PointNavBaselinePolicy
    ns.build_rnn_state_encoder = build_rnn_state_encoder
    ns.build_pack_info_from_dones = build_pack_info_from_dones
    ns.build_rnn_build_seq_info = build_rnn_build_seq_info
    ns.spaces = sys.modules["gym.spaces"]
    return ns
