"""Loader of the compiled autograd node (``csrc/torch_node.cpp`` -> ``_lib/mafed_torch_node*.so``).

The extension is host C++ only: it binds the C ABI of ``libmafed_distill.so`` at run time and turns one
``distill()`` into one call.  It also defines the ``mafed::`` torch.library ops that compiled callers trace
(``mafed_b200.ops``).  Like the library it is built in-tree (``python -m mafed_b200.build``) and there is
nothing to fall back to when it is missing.
"""
from __future__ import annotations

import importlib.util
import os
import sysconfig
import threading

from . import cabi

EXT_NAME = "mafed_torch_node"
EXT_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib",
                        EXT_NAME + (sysconfig.get_config_var("EXT_SUFFIX") or ".so"))

CACHED_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib", "libmafed_cached_step.so")

_ext = None
_lock = threading.Lock()


def load():
    """Import the extension and bind it to the library the ctypes binding uses; raise if either is absent."""
    global _ext
    if _ext is not None:
        return _ext
    with _lock:
        if _ext is not None:
            return _ext
        cabi.load()
        if not os.path.exists(EXT_PATH):
            raise cabi.MafedDistillError(
                f"{EXT_PATH} not found: build it with `python -m mafed_b200.build` "
                "(the distillation path has no CPU / eager fallback)")
        import torch  # noqa: F401  (the extension links against libtorch)
        spec = importlib.util.spec_from_file_location(EXT_NAME, EXT_PATH)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.bind(cabi.LIB_PATH)
        from . import ops
        ops.register()      # fake implementations and autograd of the mafed:: ops the extension defines
        _ext = mod
    return _ext


def load_cached():
    """The extension with ``libmafed_cached_step.so`` bound as well (the step that reads the teacher straight from the
    teacher cache); bound on first use, raise if the library is absent."""
    ext = load()
    if not ext.cached_bound():
        with _lock:
            if not ext.cached_bound():
                if not os.path.exists(CACHED_LIB_PATH):
                    raise cabi.MafedDistillError(f"{CACHED_LIB_PATH} not found: build it with `python -m mafed_b200.build`")
                ext.bind_cached(CACHED_LIB_PATH)
    return ext
