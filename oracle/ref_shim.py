"""Import shim that lets the UNMODIFIED reference (/root/reference, GOPS) be imported in this
container, where gym / ray / matplotlib / ... are not installed.

TEST INFRASTRUCTURE ONLY.  Used by `oracle/make_golden.py` (fixture generation) and by
`oracle/ref_runner.py` (bench.py's reference baselines).  Nothing in `gops_b200/` may import this file.

Technique (SURVEY.md §8(c)): a `sys.meta_path` finder serves permissive stub modules for the
missing third-party packages.  Lower-case attribute -> stub sub-module, Capitalised attribute ->
plain empty class (usable as a base class, e.g. `gym.Env`, `gym.Wrapper`, `spaces.Box`).  The
stubs satisfy *imports only*; nothing on the model/algorithm path calls into them.
"""
import importlib.abc
import importlib.machinery
import os
import sys
import types

def _default_root():
    """/root/reference in the build container; the travelled copy oracle/_ref (oracle/build_ref.py) on the GPU box."""
    if os.path.isdir("/root/reference/gops"):
        return "/root/reference"
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


REFERENCE_ROOT = os.environ.get("GOPS_REFERENCE_ROOT") or _default_root()

_STUBBED = (
    "gym", "gymnasium", "ray", "matplotlib", "seaborn", "pygame", "Box2D", "slxpy",
    "openpyxl", "cyipopt", "casadi", "onnxruntime", "onnx", "mujoco_py",
)


class _Anything:
    """Callable / subscriptable / attribute-tolerant placeholder value."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Anything()

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Anything()

    def __getitem__(self, k):
        return _Anything()

    def __setitem__(self, k, v):
        pass

    def __iter__(self):
        return iter(())


class _StubModule(types.ModuleType):
    def __init__(self, name):
        super().__init__(name)
        self.__path__ = []  # behave like a package so `import a.b.c` resolves
        self.__all__ = []

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        if name[0].isupper():
            # plain `type` class so that `class X(gym.Env, metaclass=ABCMeta)` works
            cls = type(name, (object,), {"__init__": lambda self, *a, **k: None,
                                         "__class_getitem__": classmethod(lambda c, i: c)})
            setattr(self, name, cls)
            return cls
        full = self.__name__ + "." + name
        if full in sys.modules:
            return sys.modules[full]
        if name in ("rcParams",):
            val = {}
        elif name in ("setLevel", "use", "ion", "init", "remote", "get", "put", "wait",
                      "figure", "subplots", "cla", "clf", "seed", "make", "register"):
            val = _Anything()
        else:
            val = _StubModule(full)
            sys.modules[full] = val
        setattr(self, name, val)
        return val

    def __call__(self, *a, **k):
        return _Anything()


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path=None, target=None):
        root = fullname.split(".")[0]
        if root in _STUBBED:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        return _StubModule(spec.name)

    def exec_module(self, module):
        pass


_installed = False


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "gops"))


def install():
    """Make `import gops` resolve to the unmodified reference. Idempotent."""
    global _installed
    if _installed:
        return
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    import numpy as np

    sys.dont_write_bytecode = True  # the reference tree is read-only
    sys.meta_path.insert(0, _StubFinder())
    if not hasattr(np, "float_"):
        np.float_ = np.float64  # reference `common_utils.py:158` (removed in NumPy 2)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _installed = True
