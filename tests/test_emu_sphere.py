"""Sphere (S2) path -- SphereBasis, spin recombination, SWSH transforms, per-m banded pencil systems, RHS plan -- executed
on the CPU through the test-only kernel emulation against reference data; GPU versions: tests/test_gpu_t2_sphere.py."""
import ctypes as C
import numpy as np, pytest
from emu import emu_lib as E
import sphere_cases as S


@pytest.fixture(autouse=True)
def emulation():
    E.install()
    yield
    E.uninstall()


@pytest.mark.parametrize("tag", ["a", "b"])
def test_sphere_field_transforms(golden, tag):
    S.check_field_transforms(golden("sphere.npz"), tag)


def test_sphere_pencil_matrices(golden):
    S.check_pencil_matrices(golden("sphere.npz"))


@pytest.mark.parametrize("tag,scheme", [("sw16", "RK222"), ("sw32", "RK222"), ("sw32sbdf2", "SBDF2")])
def test_shallow_water_matches_reference(golden, tag, scheme):
    sw, solver = S.check_shallow_water(golden("sphere.npz"), tag, scheme)
    assert solver.bset.last_verify < 1e-12


def test_balanced_shallow_water_matches_reference(golden):
    """The stock shallow-water problem start to finish at 32 x 16: LBVP with a gauge constant and an average condition, MulCosine
    on its right-hand side, then 3 RK222 steps of the IVP (GPU version: tests/test_gpu_t7_sphere_lbvp.py)."""
    S.check_balanced_shallow_water(golden("sphere_lbvp.npz"), "bal32")


def test_shallow_water_rk443_with_timestep_changes_matches_oracle():
    dt = 1 / 12
    S.check_against_oracle(16, 8, "RK443", [dt, dt, dt / 2, dt / 2, dt])


def test_shallow_water_with_shifted_packing_matches_oracle():
    """Ntheta > Nphi / 2: the folded triangular packing has shift > 0 and wavenumber Nphi/2 - 1 lives in the extra columns of pair 0."""
    dt = 1 / 12
    solver = S.check_against_oracle(16, 12, "RK222", [dt, dt / 2])
    assert solver.bset.nsys == 8


def test_analysis_tasks_with_operator_expressions(golden):
    S.check_analysis_tasks(golden("sphere.npz"))


def test_cfl_on_sphere_and_shell_matches_reference(golden):
    S.check_cfl_curvilinear(golden("cfl_curvilinear.npz"))


class _EmuArrays:
    """numpy arrays + the emulated library, behind the small interface sphere_cases.check_banded_* use."""
    lib = property(lambda self: E.emu())
    stream = None

    def dev(self, a):
        return np.ascontiguousarray(a)

    def ptr(self, a):
        return E.ptr(a)

    def host(self, a):
        return a


def test_banded_kernels_against_dense_solves():
    S.check_banded_kernels(_EmuArrays())


def test_banded_factor_flags_singular_system():
    S.check_banded_singular(_EmuArrays())
