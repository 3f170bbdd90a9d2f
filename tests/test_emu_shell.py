"""Spherical-shell field transforms (T6) through the CPU emulation of the kernels, against reference vectors
(tests/golden/shell.npz); GPU version: tests/test_gpu_t6_shell.py."""
import pytest
from emu import emu_lib as E
import shell_cases as SC


@pytest.fixture(autouse=True)
def emulation():
    E.install()
    yield
    E.uninstall()


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_shell_field_transforms(golden, tag):
    SC.check_shell_field_transforms({**golden("shell.npz"), **golden("shell_rank2.npz")}, tag)


def test_intertwiner_orthogonal():
    SC.check_intertwiner_orthogonal()


def test_shell_pencil_matrices(golden):
    SC.check_shell_pencil_matrices(golden("shell_ivp.npz"))


@pytest.mark.parametrize("tag,scheme", [("a_sbdf2", "SBDF2"), ("a_rk222", "RK222"), ("b_sbdf2", "SBDF2")])
def test_shell_convection_matches_reference(golden, tag, scheme):
    solver = SC.check_shell_convection(golden("shell_ivp.npz"), tag, scheme)
    assert solver.bset.last_verify < 1e-12


@pytest.mark.parametrize("smem", ["1", "0"])
def test_dense_kernels_against_numpy(smem, monkeypatch):
    """smem = 0: the solve variant that keeps the columns in global memory (systems too large for shared memory)."""
    from test_emu_sphere import _EmuArrays
    monkeypatch.setenv("DB_DENSE_SOLVE_SMEM", smem)
    SC.check_dense_kernels(_EmuArrays())


def test_shell_output_tasks_match_reference(golden):
    SC.check_shell_tasks(golden("shell_tasks.npz"))


def test_shell_convection_with_strong_flow_matches_reference(golden):
    SC.check_shell_convection_strong(golden("shell_strong.npz"))


def test_shell_convection_with_grid_function_forcing_matches_reference(golden):
    SC.check_shell_convection_forced(golden("shell_strong.npz"))
