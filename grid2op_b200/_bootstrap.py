"""Locate an importable ``grid2op`` (the host framework we plug into; NOT re-implemented here).

Search order: an already importable ``grid2op`` -> ``$GRID2OP_B200_REF`` -> ``<repo>/oracle/_ref`` (the unmodified
reference installed by ``build()``, oracle/reference.py; git-ignored) -> ``<repo>/baseline/_ref`` (the same installed with
``pip install --target``; git-ignored).  Nothing else is searched: a checkout
elsewhere is named through the environment variable (tests/conftest.py does that for the build container).

grid2op imports ``pandapower`` at package-import time (reference:
grid2op/Backend/__init__.py:4 -> grid2op/Backend/pandaPowerBackend.py:18) even when only the
abstract ``Backend`` class is wanted.  When pandapower is not installed an *empty* placeholder
module is registered so that the import of the host framework succeeds; it has no attributes, so
any attempt to actually use PandaPowerBackend fails loudly.  Nothing from the placeholder is ever
used by this package.
"""
from __future__ import annotations

import importlib
import importlib.util
import os
import sys
import types

_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_CANDIDATES = [
    os.environ.get("GRID2OP_B200_REF", ""),
    os.path.join(_REPO, "oracle", "_ref"),
    os.path.join(_REPO, "baseline", "_ref"),
]

_state = {"done": False, "ok": False, "why": ""}


def _ensure_dist_info(root: str) -> None:
    """grid2op/Space/default_var.py:26 calls importlib.metadata.version("grid2op"); a bare source
    checkout has no metadata -> patch the lookup for that one name only."""
    import importlib.metadata as md

    try:
        md.version("grid2op")
        return
    except md.PackageNotFoundError:
        pass
    init = os.path.join(root, "grid2op", "__init__.py")
    ver = "0.0.0"
    try:
        with open(init, "r", encoding="utf-8") as f:
            for line in f:
                if line.strip().startswith("__version__"):
                    ver = line.split("=")[1].strip().strip("'\"")
                    break
    except OSError:
        pass
    orig = md.version

    def version(name):  # pragma: no cover - trivial
        if name == "grid2op":
            return ver
        if name == "pandapower":
            try:
                return orig(name)
            except md.PackageNotFoundError:
                return "0.0.0"
        return orig(name)

    md.version = version


def _ensure_pandapower_placeholder() -> None:
    if importlib.util.find_spec("pandapower") is not None:
        return
    if "pandapower" in sys.modules:
        return
    mod = types.ModuleType("pandapower")
    mod.__doc__ = "placeholder registered by grid2op_b200._bootstrap (pandapower is not installed)"
    mod.__grid2op_b200_placeholder__ = True
    sys.modules["pandapower"] = mod
    import importlib.metadata as md

    orig = md.version

    def version(name):  # pragma: no cover - trivial
        if name == "pandapower":
            try:
                return orig(name)
            except md.PackageNotFoundError:
                return "0.0.0"
        return orig(name)

    md.version = version


def ensure_grid2op() -> bool:
    """Make ``import grid2op`` work if at all possible.  Returns True on success."""
    if _state["done"]:
        return _state["ok"]
    _state["done"] = True
    _ensure_pandapower_placeholder()
    try:
        import warnings

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            importlib.import_module("grid2op")
        _state["ok"] = True
        return True
    except Exception as exc:  # noqa: BLE001
        _state["why"] = repr(exc)
    for root in _CANDIDATES:
        if not root or not os.path.isdir(os.path.join(root, "grid2op")):
            continue
        if root not in sys.path:
            sys.path.insert(0, root)
        _ensure_dist_info(root)
        for k in [k for k in sys.modules if k == "grid2op" or k.startswith("grid2op.")]:
            del sys.modules[k]
        try:
            import warnings

            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                importlib.import_module("grid2op")
            _state["ok"] = True
            return True
        except Exception as exc:  # noqa: BLE001
            _state["why"] = repr(exc)
            if root in sys.path:
                sys.path.remove(root)
    return False


def why_not() -> str:
    return _state["why"]


def grid2op_data_dir() -> str:
    """Directory of the bundled environments (``grid2op/data``) of the located grid2op."""
    import grid2op

    return os.path.join(os.path.dirname(os.path.abspath(grid2op.__file__)), "data")
