"""Reference products under the git-ignored ``oracle/_ref/`` (test and benchmark infrastructure only).

The reference is pure Python: its product here is the bytecode of the files that the drop-in driver tests
(tests/test_gpu_dropin_driver.py, tests/test_gpu_internet.py) and the CPU arm of ``bench.py`` (oracle/ref_harness.py)
execute, one sourceless ``.pyc`` at the place of each ``.py`` (importable, and runnable with ``runpy.run_path``), plus the
reference's GMM prior data file.  ``__graft_entry__.build()`` makes it from the reference checkout named by
DBOA_REFERENCE_ROOT (default /root/reference) when one is readable; without one an existing ``oracle/_ref/`` is left as it is.
"""
import os
import py_compile
import shutil

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')
SOURCES = ['dynaboa_benchmark.py', 'dynaboa_internet.py', 'base_adaptor.py', 'constants.py', 'config.py', 'model/__init__.py',
           'model/hmr.py', 'model/smpl.py', 'utils/__init__.py', 'utils/geometry.py', 'utils/pose_utils.py', 'utils/dataprocess.py',
           'utils/smplify/__init__.py', 'utils/smplify/prior.py', 'utils/smplify/smplify.py', 'utils/smplify/losses.py',
           'boa_dataset/__init__.py', 'boa_dataset/pw3d.py', 'boa_dataset/internet_data.py']
DATA = ['data/gmm_08.pkl']


def source_root():
    root = os.environ.get('DBOA_REFERENCE_ROOT') or '/root/reference'
    return root if os.path.isfile(os.path.join(root, 'dynaboa_benchmark.py')) else None


def build():
    """Compile the reference files into oracle/_ref/; returns its path, or None when no reference checkout is readable."""
    src = source_root()
    if src is None:
        return None
    for rel in SOURCES + DATA:
        if not os.path.exists(os.path.join(src, rel)):
            raise FileNotFoundError(f'reference checkout {src} lacks {rel}')
    for rel in SOURCES:
        py_compile.compile(os.path.join(src, rel), cfile=os.path.join(OUT, rel[:-3] + '.pyc'), dfile=rel, doraise=True)
    for rel in DATA:
        os.makedirs(os.path.dirname(os.path.join(OUT, rel)), exist_ok=True)
        shutil.copyfile(os.path.join(src, rel), os.path.join(OUT, rel))
    return OUT
