"""`galerkin_transformer` -- the package name the reference's scripts import
(`/root/reference/libs/__init__.py:1-5`: ``from galerkin_transformer.layers import *`` ... ; `libs/model.py:1-6` falls
back to ``from galerkin_transformer.layers import *``), served by the B200 implementation.

With this repository on PYTHONPATH the reference's `examples/*.py` run unchanged:

  * ``galerkin_transformer.layers``  = the reference's `libs/layers.py` namespace with the hot-path operators
    (`SimpleAttention`, `FeedForward`, `SpectralConv1d`, `SpectralConv2d`) rebound to the sm_100a classes of
    `galerkin_transformer_b200`;
  * ``galerkin_transformer.model``   = the reference's `libs/model.py` -- its own model ASSEMBLY code -- over those
    operators, with the fusion units (`SimpleTransformerEncoderLayer`, `SpectralRegressor`, `PointwiseRegressor`) rebound too
    (set GALERKIN_B200_NATIVE_MODELS=1 to also take `FourierTransformer2D` / `SimpleTransformer` / `...2DLite` from
    `galerkin_transformer_b200.model`, which adds the library's scaler convolutions);
  * ``galerkin_transformer.utils / utils_ft / ft`` = the reference's own files (datasets, losses, training loop: out of
    scope here, SURVEY.md section 8).

The reference sources are looked up in $GALERKIN_REFERENCE (the root of a checkout of the reference).  Without them
only the B200 classes are exported.  `torchinfo`, `matplotlib` and `IPython` are optional for the reference's
utilities; minimal stand-ins are registered when they are not installed."""
import importlib.util
import os
import sys
import types


def reference_libs():
    """directory holding the reference's layers.py / model.py / ..., or None"""
    root = os.environ.get("GALERKIN_REFERENCE")
    if root and os.path.isfile(os.path.join(root, "libs", "layers.py")):
        return os.path.join(root, "libs")
    return None


class _Stub(types.ModuleType):
    """Stand-in for an absent plotting / notebook dependency of the reference's utilities: any attribute is a no-op."""
    __path__ = []

    def __getattr__(self, item):
        if item.startswith("__"):
            raise AttributeError(item)
        return lambda *a, **k: None


def _stub_optional_dependencies():
    for name in ("torchinfo", "matplotlib", "matplotlib.pyplot", "IPython", "IPython.display", "seaborn", "h5py"):
        if name in sys.modules:
            continue
        try:
            __import__(name)
        except Exception:
            sys.modules[name] = _Stub(name)


def load_reference_module(name):
    """Execute the reference's libs/<name>.py as `galerkin_transformer._ref_<name>` (once) and return the module."""
    key = f"galerkin_transformer._ref_{name}"
    if key in sys.modules:
        return sys.modules[key]
    libs = reference_libs()
    if libs is None:
        return None
    _stub_optional_dependencies()
    spec = importlib.util.spec_from_file_location(key, os.path.join(libs, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[key] = mod
    try:
        spec.loader.exec_module(mod)
    except Exception:
        del sys.modules[key]
        raise
    return mod


def export(namespace, module):
    """copy a module's public names (its __all__, else everything not underscored) into `namespace`"""
    names = getattr(module, "__all__", None) or [n for n in vars(module) if not n.startswith("_")]
    for n in names:
        namespace[n] = getattr(module, n)
    return names
