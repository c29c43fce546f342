"""Loader for the UNMODIFIED reference (test infrastructure only).

Works only where the environment variable F110_REFERENCE_ROOT names a checkout of the
reference.  It is used by ``make_golden.py`` to generate the committed fixtures and by the
optional differential tests (skipped when F110_REFERENCE_ROOT is unset).

The reference imports ``gymnasium`` and ``pyglet`` at module top
(f110_gymnasium/gym/f110_gym/envs/f110_env.py:27-45, f110_gym/__init__.py:1); neither is
installed here, so tiny in-memory stand-ins are registered in ``sys.modules`` first.  The
reference files themselves are imported as they lie on disk.
"""
import os
import sys
import types

REF_ROOT = os.environ.get("F110_REFERENCE_ROOT", "")
REF_GYM = os.path.join(REF_ROOT, "f110_gymnasium", "gym")
REF_MAPS = os.path.join(REF_ROOT, "rl_training", "maps") + "/"


def reference_available():
    return bool(REF_ROOT) and os.path.isdir(os.path.join(REF_GYM, "f110_gym", "envs"))


def _install_stubs():
    if "gymnasium" not in sys.modules:
        gym = types.ModuleType("gymnasium")

        class Env(object):
            @property
            def unwrapped(self):
                return self

        class Box(object):
            def __init__(self, low, high, shape=None, dtype=None):
                self.low, self.high, self.dtype = low, high, dtype
                self.shape = shape if shape is not None else getattr(low, "shape", None)

        spaces = types.ModuleType("gymnasium.spaces")
        spaces.Box = Box
        error = types.ModuleType("gymnasium.error")
        utils = types.ModuleType("gymnasium.utils")
        envs = types.ModuleType("gymnasium.envs")
        registration = types.ModuleType("gymnasium.envs.registration")
        registration.register = lambda *a, **k: None
        envs.registration = registration
        gym.Env, gym.spaces, gym.error, gym.utils, gym.envs = Env, spaces, error, utils, envs
        sys.modules.update({
            "gymnasium": gym, "gymnasium.spaces": spaces, "gymnasium.error": error,
            "gymnasium.utils": utils, "gymnasium.envs": envs,
            "gymnasium.envs.registration": registration,
        })
    if "pyglet" not in sys.modules:
        pyglet = types.ModuleType("pyglet")
        pyglet.options = {}
        pyglet.gl = types.ModuleType("pyglet.gl")
        sys.modules.update({"pyglet": pyglet, "pyglet.gl": pyglet.gl})


def load_reference():
    """Return a namespace with the reference's own classes / njit kernels."""
    if not REF_ROOT:
        raise SystemExit("set F110_REFERENCE_ROOT to a checkout of the reference (the directory holding f110_gymnasium/ "
                         "and rl_training/)")
    if not reference_available():
        raise SystemExit("F110_REFERENCE_ROOT=%s holds no f110_gymnasium/gym/f110_gym/envs" % REF_ROOT)
    os.environ.setdefault("NUMBA_CACHE_DIR", "/tmp/f110_numba_cache")
    _install_stubs()
    if REF_GYM not in sys.path:
        sys.path.insert(0, REF_GYM)
    # the real renderer subclasses pyglet.window.Window (rendering.py:58); never used on the step path
    if not getattr(sys.modules.get("f110_gym"), "_is_reference", False):
        # the repository's own f110_gym alias package (module id of gym.make) may be loaded: the reference's goes in its place
        for name in [k for k in sys.modules if k == "f110_gym" or k.startswith("f110_gym.")]:
            del sys.modules[name]
    if "f110_gym.envs.rendering" not in sys.modules:
        import importlib.machinery
        pkg = types.ModuleType("f110_gym")
        pkg.__path__ = [os.path.join(REF_GYM, "f110_gym")]
        pkg._is_reference = True
        sub = types.ModuleType("f110_gym.envs")
        sub.__path__ = [os.path.join(REF_GYM, "f110_gym", "envs")]
        rend = types.ModuleType("f110_gym.envs.rendering")
        rend.EnvRenderer = object
        sys.modules["f110_gym"] = pkg
        sys.modules["f110_gym.envs"] = sub
        sys.modules["f110_gym.envs.rendering"] = rend
    ns = types.SimpleNamespace()
    from f110_gym.envs import dynamic_models, laser_models, collision_models, base_classes, f110_env
    ns.dynamic_models, ns.laser_models, ns.collision_models = dynamic_models, laser_models, collision_models
    ns.base_classes, ns.f110_env = base_classes, f110_env
    ns.F110Env, ns.Simulator, ns.RaceCar, ns.Integrator = (
        f110_env.F110Env, base_classes.Simulator, base_classes.RaceCar, base_classes.Integrator)
    return ns


def fresh_statics(ns):
    """RaceCar.scan_simulator & co are class-level statics (base_classes.py:63-67)."""
    ns.RaceCar.scan_simulator = None
    ns.RaceCar.cosines = None
    ns.RaceCar.scan_angles = None
    ns.RaceCar.side_distances = None
