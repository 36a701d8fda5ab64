"""Import shim for the UNMODIFIED reference (build container only; TEST INFRASTRUCTURE).

The reference's ``models/common.py:16-18`` imports matplotlib/seaborn through
``utils.plots``/``utils.metrics``; neither is installed.  Four empty ``sys.modules`` stubs
make it importable (SURVEY.md §8c).  Nothing under ``/root/reference`` is modified.
Where the tree itself is absent (the GPU machine) the shim falls back to ``oracle/_ref/`` -- a git-ignored copy of the
tree's ``models/`` and ``utils/`` staged by ``oracle/stage_reference.py`` at build time (SURVEY.md §8c) -- so that the
reference-through-the-boundary tests run on the GPU as well; they skip when neither exists.
"""
import os
import sys
import types

_STAGED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
REF_ROOT = os.environ.get("CFT_REFERENCE_ROOT") or (
    "/root/reference" if os.path.isfile("/root/reference/models/yolo_test.py") else _STAGED)


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "models", "yolo_test.py"))


def import_reference():
    """Returns the reference's ``models.yolo_test`` module."""
    if not available():
        raise RuntimeError(f"reference tree not found at {REF_ROOT}")
    os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")
    sys.dont_write_bytecode = True
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.colors", "seaborn"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    mpl = sys.modules["matplotlib"]
    mpl.pyplot = sys.modules["matplotlib.pyplot"]
    mpl.colors = sys.modules["matplotlib.colors"]
    mpl.use = lambda *a, **k: None
    mpl.rc = lambda *a, **k: None
    if not hasattr(mpl.colors, "TABLEAU_COLORS"):
        mpl.colors.TABLEAU_COLORS = {"tab:blue": "#1f77b4"}
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    import logging
    logging.disable(logging.INFO)
    import models.yolo_test as yt  # noqa: E402
    return yt


def reference_yaml(name: str) -> str:
    return os.path.join(REF_ROOT, "models", "transformer", name + ".yaml")
