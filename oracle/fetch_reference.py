"""Copies the original project's Python modules and driver scripts, unmodified, into the git-ignored oracle/_ref/.

The original (jhbastek/PhysicsInformedDiffusionModels) is a script collection without setup.py, so there is nothing
to install or compile: its whole `src/` tree, `main.py`, `main_toy.py`, `sample.py`, `model.yaml` and `LICENSE` are
copied as they are.  The source is the directory named by PIDM_REFERENCE, else the location the golden-vector
generator and SURVEY.md use (REFERENCE_DEFAULT).  Where it is not readable an existing copy is kept; without any
copy, oracle/ref_arm.py falls back to the oracle port and tests/test_gpu_reference_drivers.py skips.  Nothing in the
product package reads oracle/_ref/.  `__graft_entry__.build()` runs fetch().
"""
import os
import shutil

HERE = os.path.dirname(os.path.abspath(__file__))
DEST = os.path.join(HERE, '_ref')
REFERENCE_DEFAULT = '/root/reference'
FILES = ('main.py', 'sample.py', 'main_toy.py', 'model.yaml', 'LICENSE')


def source_dir():
    return os.environ.get('PIDM_REFERENCE') or REFERENCE_DEFAULT


def _copy_tree(src, dst):
    """File contents only (copyfile, no copystat): the original may be a read-only tree, and its permission bits would
    keep a later build() by an ordinary user from replacing the copy."""
    for d, subdirs, files in os.walk(src):
        subdirs[:] = [s for s in subdirs if s != '__pycache__']
        out = os.path.join(dst, os.path.relpath(d, src))
        os.makedirs(out, exist_ok=True)
        for f in files:
            shutil.copyfile(os.path.join(d, f), os.path.join(out, f))


def fetch():
    """-> True when oracle/_ref/ holds the original's modules afterwards."""
    src = source_dir()
    if os.access(os.path.join(src, 'src'), os.R_OK | os.X_OK):
        shutil.rmtree(DEST, ignore_errors=True)
        _copy_tree(os.path.join(src, 'src'), os.path.join(DEST, 'src'))
        for f in FILES:
            if os.path.exists(os.path.join(src, f)):
                shutil.copyfile(os.path.join(src, f), os.path.join(DEST, f))
    return os.path.isfile(os.path.join(DEST, 'src', 'unet_model.py'))
