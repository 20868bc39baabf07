"""Runs the reference's UNMODIFIED learning/main.py on top of superpoint_graph_b200:

    python compat/run_main.py [--reference-root DIR] -- <arguments of learning/main.py>

* `superpoint_graph_b200.dropin.install()` registers the sm_100a mirrors under the reference's module
  names (learning.pointnet / graphnet / modules / ecc) before main.py's imports run;
* packages the image lacks (igraph, h5py, torchnet, transforms3d) resolve to the stand-ins in this
  directory — only if the real ones cannot be imported;
* main.py itself is executed with runpy, unmodified: from the checkout given by --reference-root, else
  as the bytecode oracle/build_ref.py compiled from the reference into oracle/_ref/.
"""
import importlib
import os
import runpy
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _use_standins():
    missing = []
    for name in ("igraph", "h5py", "torchnet", "transforms3d"):
        try:
            importlib.import_module(name)
        except Exception:
            missing.append(name)
    if missing and HERE not in sys.path:
        sys.path.insert(0, HERE)
    for name in missing:
        sys.modules.pop(name, None)
        importlib.import_module(name)
    return missing


def main_script(ref):
    """learning/main.py of a checkout, or learning/main.pyc of oracle/_ref; None if there is neither."""
    for name in ("main.py", "main.pyc"):
        path = os.path.join(ref, "learning", name)
        if os.path.exists(path):
            return path
    return None


def reference_root(explicit=None):
    for cand in (explicit, os.path.join(ROOT, "oracle", "_ref")):
        if cand and main_script(cand):
            return cand
    raise RuntimeError("no reference learning/main.py found (pass --reference-root, or build oracle/_ref with "
                       "python -m oracle.build_ref)")


def run(main_args, ref_root=None):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    standins = _use_standins()
    ref = reference_root(ref_root)
    from superpoint_graph_b200 import dropin
    dropin.install(reference_root=ref)
    learning_dir = os.path.join(ref, "learning")
    # `python learning/main.py` puts learning/ first on sys.path (bare `import spg`, `import s3dis_dataset`)
    if learning_dir in sys.path:
        sys.path.remove(learning_dir)
    sys.path.insert(0, learning_dir)
    old_argv = sys.argv
    sys.argv = [main_script(ref)] + list(main_args)
    try:
        print("[run_main] reference: %s  stand-ins: %s" % (ref, ", ".join(standins) or "none"), flush=True)
        runpy.run_path(sys.argv[0], run_name="__main__")
    finally:
        sys.argv = old_argv


if __name__ == "__main__":
    argv = sys.argv[1:]
    ref_root = None
    if argv and argv[0] == "--reference-root":
        ref_root, argv = argv[1], argv[2:]
    if argv and argv[0] == "--":
        argv = argv[1:]
    run(argv, ref_root)
