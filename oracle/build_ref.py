"""Byte-compile the original IDE-3D project's caller scripts into oracle/_ref/ (git-ignored build output).

tests/test_reference_cli.py runs those scripts (gen_images.py, gen_videos.py, extract_shapes.py, viz/renderer.py) unmodified
against this package.  They are imported from the sourceless .pyc files written here, so the tests need no checkout of the
original project once oracle/_ref/ exists, and nothing of it is committed.  The checkout is read from $IDE3D_REFERENCE, else from
/root/reference (the location baseline/build_ref_plugins.py reads as well); without one there is nothing to build and those
tests skip.  Python bytecode is specific to the interpreter version: run it with the Python that runs the tests.
"""

import os
import py_compile
import shutil
import warnings

REF = os.environ.get('IDE3D_REFERENCE', '/root/reference')
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')
PACKAGES = ('dnnlib', 'inversion', 'training', 'torch_utils', 'metrics', 'gui_utils', 'viz')   # what the scripts import, besides this package


def _sources():
    for name in sorted(os.listdir(REF)):
        if name.endswith('.py'):
            yield name
    for pkg in PACKAGES:
        for dirpath, dirs, files in os.walk(os.path.join(REF, pkg)):
            dirs[:] = sorted(d for d in dirs if d != '__pycache__')
            for f in sorted(files):
                if f.endswith('.py'):
                    yield os.path.relpath(os.path.join(dirpath, f), REF)


def build():
    """-> OUT, or None when no checkout of the original project is readable."""
    if not os.path.isfile(os.path.join(REF, 'gen_images.py')):
        return None
    shutil.rmtree(OUT, ignore_errors=True)
    try:
        with warnings.catch_warnings():
            warnings.simplefilter('ignore', SyntaxWarning)     # the original sources' own style warnings
            for rel in _sources():
                # legacy layout (module.pyc beside where module.py would be): the import system loads it without the source
                py_compile.compile(os.path.join(REF, rel), cfile=os.path.join(OUT, rel + 'c'), dfile=rel, doraise=True,
                                   invalidation_mode=py_compile.PycInvalidationMode.UNCHECKED_HASH)
    except (OSError, py_compile.PyCompileError):             # an unreadable or partial checkout: build nothing rather than half
        shutil.rmtree(OUT, ignore_errors=True)
        return None
    return OUT


if __name__ == '__main__':
    print(build())
