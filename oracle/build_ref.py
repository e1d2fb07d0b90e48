"""Installs the reference package (lucidrains/DALLE-pytorch, pure Python: its build is a copy of the package) into oracle/_ref/.

TEST / MEASUREMENT INFRASTRUCTURE ONLY.  oracle/_ref/ is a build product: git-ignored, never imported by the product package,
imported through oracle/ref_import.py by the tests that patch or compare with the reference's own classes and by bench.py's
reference legs.  `__graft_entry__.build()` runs this; by hand:

    python oracle/build_ref.py

The source is the reference checkout found by ref_import.source_root() ($DALLE_REFERENCE_ROOT or the default checkout location).
Where no checkout is readable, an oracle/_ref/ built earlier is kept as it is, so a tree built next to the reference still
carries it to a machine without one.
"""
import os
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_import  # noqa: E402


def _copy_package(src, dst):
    """Copies the files of the package at `src` to `dst` with fresh modes: directories and files are created by this process
    (makedirs / copyfile), not given the checkout's modes, so a read-only checkout still yields a copy the owner can replace."""
    for d, dirs, files in os.walk(src):
        dirs[:] = [x for x in dirs if x != '__pycache__']
        out = os.path.join(dst, os.path.relpath(d, src))
        os.makedirs(out, exist_ok=True)
        for f in files:
            if not f.endswith('.pyc'):
                shutil.copyfile(os.path.join(d, f), os.path.join(out, f))


def _remove_tree(path):
    """rmtree that also removes a tree whose directories are read-only (a copy made before modes were reset)."""
    def writable_and_retry(fn, p, _exc):
        os.chmod(os.path.dirname(p), 0o700)
        if os.path.isdir(p) and not os.path.islink(p):
            os.chmod(p, 0o700)
        fn(p)
    shutil.rmtree(path, **({'onexc': writable_and_retry} if sys.version_info >= (3, 12) else {'onerror': writable_and_retry}))


def build_ref():
    """Returns the directory the reference is imported from afterwards, or None when neither a checkout nor a copy exists."""
    src = ref_import.source_root()
    if src is not None:
        os.makedirs(ref_import.BUILD_ROOT, exist_ok=True)
        tmp = tempfile.mkdtemp(prefix='.dalle_pytorch.', dir=ref_import.BUILD_ROOT)
        try:
            _copy_package(os.path.join(src, 'dalle_pytorch'), os.path.join(tmp, 'dalle_pytorch'))
            dst = os.path.join(ref_import.BUILD_ROOT, 'dalle_pytorch')
            if os.path.isdir(dst):
                _remove_tree(dst)
            os.rename(os.path.join(tmp, 'dalle_pytorch'), dst)
        finally:
            _remove_tree(tmp)
    return ref_import.resolve()


if __name__ == '__main__':
    print('reference:', build_ref())
