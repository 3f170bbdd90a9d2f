"""Spherical shell on the GPU: field transforms (T6: radial Jacobi transform + regularity recombination on top of the sphere
chain) against reference vectors (tests/golden/shell.npz), the dense per-l pencil kernels, and the shell-convection IVP of
BASELINE config 5 against reference states (tests/golden/shell_ivp.npz)."""
import pytest
import shell_cases as SC

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_shell_field_transforms(golden, tag):
    SC.check_shell_field_transforms({**golden("shell.npz"), **golden("shell_rank2.npz")}, tag)


@pytest.mark.parametrize("smem", ["1", "0"])
def test_dense_kernels_against_numpy(smem, monkeypatch):
    from test_gpu_t2_sphere import _CudaArrays
    monkeypatch.setenv("DB_DENSE_SOLVE_SMEM", smem)
    SC.check_dense_kernels(_CudaArrays())


def test_shell_pencil_matrices(golden):
    SC.check_shell_pencil_matrices(golden("shell_ivp.npz"))


@pytest.mark.parametrize("tag,scheme", [("a_sbdf2", "SBDF2"), ("a_rk222", "RK222"), ("b_sbdf2", "SBDF2")])
def test_shell_convection_matches_reference(golden, tag, scheme):
    """BASELINE config 5's problem (shell convection) at 16 x 8 x 6 and 32 x 16 x 12 against the reference."""
    solver = SC.check_shell_convection(golden("shell_ivp.npz"), tag, scheme)
    assert solver.bset.last_verify < 1e-12


@pytest.mark.parametrize("which", ["sphere:sw16", "sphere:sw32", "shell:a_sbdf2", "shell:b_sbdf2", "tasks:cartesian", "tasks:shell",
                                   "plugin:transpose", "strong3d", "shell:forced", "staged2d"])
def test_two_gpu_curvilinear_matches_reference(which):
    """Sphere / shell problems on 2 GPUs over NCCL (coefficients distributed over the azimuthal pairs, grid over colatitude)
    against the single-rank reference states."""
    import torch, subprocess, sys, os, socket, pathlib
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = pathlib.Path(__file__).resolve().parents[1]
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(root / "tests" / "dist_worker.py"), which]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, DB_DIST_BACKEND="nccl"))
    assert "DIST_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]


def test_sphere_analysis_tasks_with_operator_expressions(golden):
    import sphere_cases as S
    S.check_analysis_tasks(golden("sphere.npz"))


def test_cfl_on_sphere_and_shell_matches_reference(golden):
    import sphere_cases as S
    S.check_cfl_curvilinear(golden("cfl_curvilinear.npz"))


def test_shell_output_tasks_match_reference(golden):
    """Tasks and flow property of the stock shell-convection script (radial / azimuthal interpolation of a flux, np.sqrt(u@u)/nu)."""
    import shell_cases as SC
    SC.check_shell_tasks(golden("shell_tasks.npz"))


def test_shell_convection_with_strong_flow_matches_reference(golden):
    import shell_cases as SC
    SC.check_shell_convection_strong(golden("shell_strong.npz"))


def test_shell_convection_with_grid_function_forcing_matches_reference(golden):
    import shell_cases as SC
    SC.check_shell_convection_forced(golden("shell_strong.npz"))


def test_shell_convection_64x32x24_matches_reference(golden):
    """A larger shell with a real flow (passes under emulation in 2 minutes, so it is a GPU-suite case only)."""
    import shell_cases as SC
    solver = SC.check_shell_convection_big(golden("shell_strong.npz"))
    assert solver.bset.last_verify < 1e-12
