"""Materialise the read-only reference (/root/reference, Dedalus v3.0.5) as an importable,
single-process package under a scratch directory OUTSIDE the repo (default /tmp/dedalus_ref).

TEST INFRASTRUCTURE ONLY.  Used by tests/golden/make_golden.py to generate the committed golden
fixtures.  Nothing in the product (dedalus_b200/), bench.py or the gpu tests imports this: the
reference does not exist on the GPU box.

Recipe (SURVEY.md section 8c): copy the python package, cythonize only tools/linalg.pyx and
libraries/spin_recombination.pyx (no OpenMP), provide 1-rank stand-ins for mpi4py / h5py / numexpr,
replace the FFTW wrapper by a numpy buffer allocator and core/transposes by placeholders (never
instantiated when the process mesh is trivial), and select the reference's own scipy transform classes.
"""
import os, sys, shutil, subprocess, textwrap, pathlib

REF = pathlib.Path(os.environ.get("DEDALUS_REFERENCE", "/root/reference"))
DST = pathlib.Path(os.environ.get("DEDALUS_REF_SHIM", "/tmp/dedalus_ref"))

MPI_STUB = '''
SUM="SUM"; MAX="MAX"; MIN="MIN"; DOUBLE="DOUBLE"; IN_PLACE=object()
class Comm:
    rank=0; size=1; dim=0; coords=[]
    def Create_cart(self, dims, **kw):
        c=Comm(); c.dim=len(dims); c.coords=[0]*len(dims); return c
    def Sub(self, remain): return Comm()
    def Get_coords(self, rank): return list(self.coords)
    def Get_rank(self): return 0
    def Get_size(self): return 1
    def Barrier(self): pass
    def Bcast(self, buf, root=0): pass
    def bcast(self, obj, root=0): return obj
    def allreduce(self, x, op=None): return x
    def reduce(self, x, op=None, root=0): return x
    def Allreduce(self, send, recv, op=None):
        if send is not IN_PLACE: recv[...] = send
    def gather(self, x, root=0): return [x]
    def allgather(self, x): return [x]
    def scatter(self, x, root=0): return x[0]
COMM_WORLD=Comm(); COMM_SELF=Comm()
def Wtime():
    import time; return time.time()
'''

FFTW_STUB = '''
import numpy as np
def fftw_mpi_init(): pass
def create_buffer(n): return np.zeros(int(n), dtype=np.float64)
def create_array(shape, dtype): return np.zeros(shape, dtype=dtype)
def create_copy(a): return np.array(a, copy=True)
class _NoFFTW:
    def __init__(self, *a, **k): raise RuntimeError("FFTW is not available under the oracle shim")
FourierTransform = R2HCTransform = DiscreteCosineTransform = DiscreteSineTransform = _NoFFTW
'''

TRANSPOSES_STUB = '''
class _NoMPI:
    def __init__(self, *a, **k): raise RuntimeError("distributed transposes unavailable under the 1-rank oracle shim")
FFTWTranspose = AlltoallvTranspose = RowDistributor = ColDistributor = _NoMPI
'''


def build(force=False):
    marker = DST / ".built"
    if marker.exists() and not force:
        return DST
    if DST.exists():
        shutil.rmtree(DST)
    DST.mkdir(parents=True)
    shutil.copytree(REF / "dedalus", DST / "dedalus",
                    ignore=shutil.ignore_patterns("tests", "tests_parallel", "__pycache__"))
    for p in [DST / "dedalus", *(DST / "dedalus").rglob("*")]:       # the copy keeps the modes of a read-only checkout
        p.chmod(p.stat().st_mode | 0o200)
    # stand-in modules
    (DST / "mpi4py").mkdir()
    (DST / "mpi4py" / "__init__.py").write_text("def get_include(): return ''\n")
    (DST / "mpi4py" / "MPI.py").write_text(MPI_STUB)
    (DST / "h5py").mkdir()
    (DST / "h5py" / "__init__.py").write_text("class File: pass\n")
    (DST / "numexpr").mkdir()
    (DST / "numexpr" / "__init__.py").write_text(
        "def evaluate(*a, **k): raise NotImplementedError('numexpr stub')\n")
    # fftw wrapper -> numpy allocator
    fdir = DST / "dedalus" / "libraries" / "fftw"
    for f in fdir.iterdir():
        if f.suffix in (".pyx", ".pxd"):
            f.unlink()
    (fdir / "fftw_wrappers.py").write_text(FFTW_STUB)
    (fdir / "__init__.py").write_text("from . import fftw_wrappers\nfftw_wrappers.fftw_mpi_init()\n")
    # transposes -> placeholders
    (DST / "dedalus" / "core" / "transposes.pyx").unlink()
    (DST / "dedalus" / "core" / "transposes.py").write_text(TRANSPOSES_STUB)
    # cythonize the two pure-compute extension modules
    setup = textwrap.dedent('''
        from setuptools import setup, Extension
        from Cython.Build import cythonize
        import numpy as np
        exts = [Extension("dedalus.tools.linalg", ["dedalus/tools/linalg.pyx"], include_dirs=[np.get_include()],
                          extra_compile_args=["-O3", "-Wno-unused-function"]),
                Extension("dedalus.libraries.spin_recombination", ["dedalus/libraries/spin_recombination.pyx"],
                          include_dirs=[np.get_include()], extra_compile_args=["-O3"])]
        setup(name="ref_ext", ext_modules=cythonize(exts, language_level=3), script_args=["build_ext", "--inplace"])
    ''')
    (DST / "_build_ext.py").write_text(setup)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    subprocess.run([sys.executable, "_build_ext.py"], cwd=DST, check=True, env=env,
                   stdout=subprocess.DEVNULL)
    marker.write_text("ok\n")
    return DST


def activate():
    """Build if needed, put the shim first on sys.path, import dedalus with scipy transforms selected."""
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    root = build()
    if str(root) not in sys.path:
        sys.path.insert(0, str(root))
    import logging
    logging.disable(logging.INFO)
    import dedalus.public as d3
    from dedalus.core import basis
    basis.FourierBase.default_library = "scipy"
    basis.Jacobi.default_dct = "scipy_dct"
    return d3


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
