"""Loader for the in-tree native extension ``dist_tuto.pth_b200/_C.so``.

The extension is built by ``build.py`` (nvcc, sm_100a only) and lives in the
package directory so it travels with the repo snapshot.  There is NO silent
PyTorch fallback for the ops it provides: if it cannot be loaded, ``C()`` raises
with the build instruction."""
from __future__ import annotations

import importlib.util
import os
import threading

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SO = os.path.join(_PKG, "_C.so")
_mod = None
_err = None
_lock = threading.Lock()


def so_path() -> str:
    """Path of the in-tree extension (``dist_tuto.pth_b200/_C.so``; built by ``build.py``)."""
    return _SO


def available() -> bool:
    """Whether the native extension can be loaded (building it first if allowed)."""
    try:
        C()
        return True
    except Exception:
        return False


def _build_locked():
    """(Re)build ``_C.so`` if it is missing or stale, serialised ACROSS processes.

    N spawned ranks all land here at once: an ``flock`` on ``csrc/build/.lock`` lets one of them build while the others
    wait and then find an up-to-date library.  ``build.build()`` is content-hashed (no-op when sources, flags and the
    link stamp match) and links to a temporary file that is ``os.replace``d into place, so nobody can import a
    half-written library.  When nvcc is not installed (a deployment box) an existing library is used as is.  An up-to-date
    library is loaded without taking the lock, so a built tree can be used read-only."""
    import fcntl
    import shutil
    from .. import build as _b
    if _b.up_to_date():
        return
    have_nvcc = os.path.exists(os.path.join(_b._cuda_home(), "bin", "nvcc")) or shutil.which("nvcc") is not None
    if not have_nvcc:
        if os.path.isfile(_SO):
            return
        raise ImportError(f"native extension missing and no nvcc to build it: {_SO}")
    os.makedirs(_b.OBJ, exist_ok=True)
    with open(os.path.join(_b.OBJ, ".lock"), "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        try:
            if not os.path.isfile(_SO) or not _b.up_to_date():
                _b.build(verbose=False)
        finally:
            fcntl.flock(lk, fcntl.LOCK_UN)


def C():
    """Return the loaded extension module (loads it on first use)."""
    global _mod, _err
    if _mod is not None:
        return _mod
    with _lock:
        if _mod is not None:
            return _mod
        if os.environ.get("B200DIST_AUTOBUILD", "1") == "1":           # build the real thing (never a PyTorch fallback)
            _build_locked()
        elif not os.path.isfile(_SO):
            raise ImportError(f"native extension missing: {_SO}\n"
                              "build it with:  python -c 'import __graft_entry__ as g; g.build()'")
        import torch  # noqa: F401  (libtorch must be loaded first)
        spec = importlib.util.spec_from_file_location("dist_tuto.pth_b200._C", _SO)
        mod = importlib.util.module_from_spec(spec)
        try:
            spec.loader.exec_module(mod)
        except Exception as e:  # pragma: no cover
            _err = e
            raise ImportError(f"failed to load {_SO}: {e}") from e
        _mod = mod
        return _mod
