"""Install the unmodified reference (javieryu/nn_distributed_training) into oracle/_ref/ (git-ignored), the tree that
``bench.py --impl reference``, scripts/precision_parity.py and the reference-arm contract test import.

The reference's setup.py names no packages, so ``pip install`` refuses its flat layout ("Multiple top-level packages
discovered"); what ``pip install -e .`` would have provided is the source tree on ``sys.path``, so its Python packages are
copied verbatim (notebooks, data and trained artefacts skipped).  The source is the checkout named by
``NNDT_REFERENCE_SRC`` (default: /root/reference, where the development environment mounts it).  Without a source
checkout an existing oracle/_ref/ is left as it is.

    python oracle/install_reference.py [SRC]
"""
import os
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
PACKAGES = ("models", "optimizers", "problems", "utils", "floorplans", "experiments")


def install(src=None):
    """Returns the installed tree, or None when neither a source checkout nor an earlier install is there."""
    src = src or os.environ.get("NNDT_REFERENCE_SRC", "/root/reference")
    if not os.path.isdir(os.path.join(src, "optimizers")):
        return DST if os.path.isdir(os.path.join(DST, "optimizers")) else None
    tmp = tempfile.mkdtemp(prefix="_ref.", dir=HERE)
    try:
        keep_py = lambda d, names: [n for n in names if not os.path.isdir(os.path.join(d, n)) and not n.endswith(".py")]
        for p in PACKAGES:
            if os.path.isdir(os.path.join(src, p)):
                shutil.copytree(os.path.join(src, p), os.path.join(tmp, p), ignore=keep_py)
        for f in ("__init__.py", "LICENSE"):
            if os.path.exists(os.path.join(src, f)):
                shutil.copy(os.path.join(src, f), tmp)
        for d, _, _ in os.walk(tmp):            # the source checkout may be read-only
            os.chmod(d, 0o755)
        shutil.rmtree(DST, ignore_errors=True)
        os.rename(tmp, DST)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return DST


if __name__ == "__main__":
    print("reference at", install(sys.argv[1] if len(sys.argv) > 1 else None))
