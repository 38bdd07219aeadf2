"""Import shim for the *real* reference (chanchanchan97/ICAFusion) -- TEST INFRASTRUCTURE ONLY.

The reference is pure Python/PyTorch but imports a few packages this image lacks
(matplotlib, seaborn, thop, timm, pycocotools).  `load_reference()` installs inert
stand-ins for those in `sys.modules`, puts the reference tree on `sys.path` and returns
its `models.common` / `models.yolo_test` modules.  Nothing in the reference tree is
modified or copied.

Only the `oracle/gen_golden*.py` generators call this; the tests replay what they stored
under tests/golden/ and need no reference tree.
"""
import importlib
import os
import sys
import types

REF_ROOT = os.environ.get("ICAF_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "models", "common.py"))


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []  # behave like a package so `import a.b` works
    sys.modules[name] = m
    return m


def _lenient(mod):
    """Unknown public attributes of a stub resolve to an inert object; dunders do not
    (inspect.getmodule probes `__file__` on every entry of sys.modules)."""
    def _getattr(k):
        if k.startswith("__"):
            raise AttributeError(k)
        return _Anything()
    mod.__getattr__ = _getattr


class _Anything:
    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return self

    def __getattr__(self, k):
        if k.startswith("__"):
            raise AttributeError(k)
        return _Anything()


def _install_stubs():
    class _Unused:
        def __init__(self, *a, **k):
            pass

        def __call__(self, *a, **k):
            return self

        def __getattr__(self, k):
            return _Anything()

    if "matplotlib" not in sys.modules:
        try:
            import matplotlib  # noqa: F401
        except Exception:
            colors = _stub("matplotlib.colors", TABLEAU_COLORS={
                "tab:blue": "#1f77b4", "tab:orange": "#ff7f0e", "tab:green": "#2ca02c",
                "tab:red": "#d62728", "tab:purple": "#9467bd", "tab:brown": "#8c564b",
                "tab:pink": "#e377c2", "tab:gray": "#7f7f7f", "tab:olive": "#bcbd22",
                "tab:cyan": "#17becf"})
            plt = _stub("matplotlib.pyplot")
            _lenient(plt)
            mpl = _stub("matplotlib", colors=colors, pyplot=plt,
                        rc=lambda *a, **k: None, use=lambda *a, **k: None)
            _lenient(mpl)
    for name in ("seaborn", "thop", "pycocotools", "pycocotools.mask"):
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                s = _stub(name)
                _lenient(s)
    try:
        importlib.import_module("timm.models.layers")
    except Exception:
        import torch.nn as nn

        class DropPath(nn.Identity):
            def __init__(self, *a, **k):
                super().__init__()
        _stub("timm")
        _stub("timm.models")
        _stub("timm.models.layers", DropPath=DropPath)


def load_reference():
    """Returns (models.common, models.yolo_test) of the real reference."""
    if not reference_available():
        raise FileNotFoundError(f"reference tree not found at {REF_ROOT}")
    _install_stubs()
    import numpy as np
    if not hasattr(np, "int"):
        np.int = int  # utils/datasets.py:801 uses the removed alias
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    common = importlib.import_module("models.common")
    yolo = importlib.import_module("models.yolo_test")
    return common, yolo
