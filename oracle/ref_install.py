"""Install the unmodified reference (pykg2vec 0.0.52, pure Python) under oracle/_ref/ for the drop-in
tests and the reference arm of bench.py.

The source is a checkout of the reference, taken from $PYKG2VEC_REFERENCE_SRC (default: /root/reference).
Its `pykg2vec` package and the pretrained FB15k TransE checkpoint that its installer does not package
(examples/pretrained/TransE, read through Trainer.load_model, pykg2vec/utils/trainer.py:399-419) are
copied file by file; nothing of them is modified.  oracle/_ref/ is not under version control.  Where no
checkout is readable an existing install is kept, and without one the tests that need it skip.
"""
import os
import shutil

REF_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
CHECKPOINT = os.path.join("examples", "pretrained", "TransE")


def source_dir():
    return os.environ.get("PYKG2VEC_REFERENCE_SRC", "/root/reference")


def installed():
    return os.path.isfile(os.path.join(REF_DIR, "pykg2vec", "__init__.py"))


def _copy_tree(src, dst):
    """plain file copies into writable directories (the checkout may be read-only; its modes are not kept)"""
    for dirpath, dirnames, filenames in os.walk(src):
        dirnames[:] = [d for d in dirnames if d != "__pycache__"]
        out = os.path.join(dst, os.path.relpath(dirpath, src))
        os.makedirs(out, exist_ok=True)
        for name in filenames:
            if not name.endswith(".pyc"):
                shutil.copyfile(os.path.join(dirpath, name), os.path.join(out, name))


def install(force=False):
    """-> REF_DIR when the reference is installed there, else None (no readable checkout)."""
    src = source_dir()
    if installed() and not force:
        return REF_DIR
    if not os.access(os.path.join(src, "pykg2vec", "__init__.py"), os.R_OK):
        return REF_DIR if installed() else None
    tmp = REF_DIR + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    _copy_tree(os.path.join(src, "pykg2vec"), os.path.join(tmp, "pykg2vec"))
    if os.path.isdir(os.path.join(src, CHECKPOINT)):
        _copy_tree(os.path.join(src, CHECKPOINT), os.path.join(tmp, CHECKPOINT))
    shutil.rmtree(REF_DIR, ignore_errors=True)
    os.replace(tmp, REF_DIR)
    return REF_DIR
