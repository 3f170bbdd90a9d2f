"""Materialise the UNMODIFIED reference (Dedalus v3.0.5, from a read-only checkout located by build() below) as a single-process
importable package under oracle/_ref/ (git-ignored build product) so that `bench.py --impl reference` and the `cpu_baseline`
leg can time the reference's own solver.step on the host cores.  TEST / BENCH INFRASTRUCTURE.

    python -m oracle.build_ref          (where the reference checkout exists; elsewhere an existing oracle/_ref is kept)

Recipe = tests/golden/ref_shim.py (SURVEY.md section 8c): the reference's python package is copied as it is; only
tools/linalg.pyx and libraries/spin_recombination.pyx are cythonized (no OpenMP); mpi4py / h5py / numexpr get 1-rank
stand-in modules; the FFTW wrapper is replaced by a numpy buffer allocator and the reference's OWN scipy transform classes
(core/transforms.py:270-289, 512-534, 893-896) are selected; core/transposes is a placeholder (never instantiated on a trivial
mesh).  No reference source enters the repository's history."""
import os, sys, pathlib
ROOT = pathlib.Path(__file__).resolve().parents[1]
DST = ROOT / "oracle" / "_ref"


def build(force=False):
    if not pathlib.Path(os.environ.get("DEDALUS_REFERENCE", "/root/reference")).exists():
        return DST if (DST / ".built").exists() else None
    os.environ["DEDALUS_REF_SHIM"] = str(DST)
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    import importlib
    import ref_shim
    importlib.reload(ref_shim)
    return ref_shim.build(force=force)


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
