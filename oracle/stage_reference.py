"""Stage the UNMODIFIED reference tree for the GPU box (TEST INFRASTRUCTURE; run by ``__graft_entry__.build()``).

The reference tree exists only where the goldens are made.  SURVEY.md section 8c: prefer copying the reference tree at
run time over restating.  This copies the Python files the hot path's tests import -- ``models/``, ``utils/`` (top-level
modules only) and ``global_var.py`` -- into ``oracle/_ref/``, which is git-ignored (never enters the history) and travels
with the built tree like the built ``.so``.  ``oracle/ref_shim.py`` falls back to it when the tree itself is absent, so the
``ref_shim.available()`` tests -- the reference's own ``Model`` / ``forward_once`` running on the B200 kernels through
``install()``, ``attempt_load`` of a checkpoint pickled by the reference, the reference modules as the eager-GPU baseline
and the train step of BASELINE config 4 -- also run on the GPU.  Nothing in the product package imports it."""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("CFT_REFERENCE_SRC", "/root/reference")
DST = os.path.join(ROOT, "oracle", "_ref")


def stage(verbose: bool = False) -> bool:
    if not os.path.isfile(os.path.join(SRC, "models", "yolo_test.py")):
        return False
    ignore = shutil.ignore_patterns("__pycache__", "*.pyc", "aws", "flask_rest_api", "google_app_engine", "wandb_logging")
    for sub in ("models", "utils"):
        dst = os.path.join(DST, sub)
        if os.path.isdir(dst):
            shutil.rmtree(dst)
        shutil.copytree(os.path.join(SRC, sub), dst, ignore=ignore)
    shutil.copy2(os.path.join(SRC, "global_var.py"), os.path.join(DST, "global_var.py"))
    if verbose:
        n = sum(len(f) for _, _, f in os.walk(DST))
        print(f"staged {n} reference files under {DST}")
    return True


if __name__ == "__main__":
    sys.exit(0 if stage(verbose=True) else 1)
