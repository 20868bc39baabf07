"""Compiles the reference project's learning/ scripts to bytecode under oracle/_ref/ (git-ignored).

    python -m oracle.build_ref

The reference checkout is read from SPG_REFERENCE (default: /root/reference, where the build
environment keeps it).  Only compiled modules are written (sourceless `<name>.pyc`, importable
without their sources), for bench.py's reference arm (baseline/ref_arm.py) and for running the
reference's unmodified learning/main.py (compat/run_main.py).  Their code objects keep the
checkout's file names, so tracebacks show the reference's lines wherever the checkout exists.
Without a checkout nothing is changed: a previously built oracle/_ref/ stays usable.
"""
import os
import py_compile
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
MODULES = [
    # the hot path timed by bench.py --impl reference
    "learning/__init__.py",
    "learning/pointnet.py",
    "learning/graphnet.py",
    "learning/modules.py",
    "learning/metrics.py",
    "learning/ecc/__init__.py",
    "learning/ecc/GraphConvInfo.py",
    "learning/ecc/GraphConvModule.py",
    "learning/ecc/GraphPoolInfo.py",
    "learning/ecc/GraphPoolModule.py",
    "learning/ecc/cuda_kernels.py",
    "learning/ecc/utils.py",
    # the trainer and its data side
    "learning/main.py",
    "learning/spg.py",
    "learning/s3dis_dataset.py",
    "learning/custom_dataset.py",
    "learning/sema3d_dataset.py",
    "learning/vkitti_dataset.py",
]


def reference_checkout():
    return os.environ.get("SPG_REFERENCE", "/root/reference")


def available():
    """True if oracle/_ref/ holds the compiled reference (built here or shipped with the tree)."""
    return os.path.exists(os.path.join(DST, "learning", "main.pyc"))


def build():
    """-> number of modules compiled (0 if the reference checkout is absent)."""
    src_root = reference_checkout()
    if not os.path.isfile(os.path.join(src_root, "learning", "main.py")):
        return 0
    shutil.rmtree(DST, ignore_errors=True)
    for rel in MODULES:
        src = os.path.join(src_root, rel)
        py_compile.compile(src, cfile=os.path.join(DST, rel[:-3] + ".pyc"), dfile=src, doraise=True)
    return len(MODULES)


if __name__ == "__main__":
    print("compiled", build(), "modules ->", DST)
