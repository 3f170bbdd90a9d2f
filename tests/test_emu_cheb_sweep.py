"""Chebyshev transforms at every basis order and fused derivative through the CPU emulation of the kernels, against the
high-precision reference of cheb_sweep_cases.py.  The same body runs on the GPU in test_gpu_u1_cheb_sweep.py."""
import pytest
from emu import emu_lib as E
import cheb_sweep_cases as S


@pytest.fixture(autouse=True)
def emulation():
    E.install()
    yield
    E.uninstall()


def test_reference_pins_fixtures(golden):
    S.check_reference_pins_fixtures(golden("transforms.npz"))


# M < N, M = N, M > N; odd N and N with factors 7, 11, 13; the register-kernel lengths 48 and 96
@pytest.mark.parametrize("path,M,N", [
    ("strided", 32, 48), ("strided", 15, 22), ("strided", 24, 16), ("strided", 21, 21), ("strided", 26, 39),
    ("lines", 32, 48), ("lines", 64, 96), ("lines", 15, 22), ("lines", 21, 21), ("lines", 20, 26),
    ("lines", 24, 16), ("lines", 17, 16),
    ("offset", 32, 48), ("offset", 15, 22),
    ("complex", 32, 48), ("complex", 24, 16)])
def test_backward_every_order_and_derivative(path, M, N):
    S.sweep_backward(path, M, N)


@pytest.mark.parametrize("path,M,N", [("strided", 32, 48), ("strided", 24, 16), ("lines", 15, 22), ("lines", 32, 48), ("lines", 64, 96)])
def test_forward_every_order(path, M, N):
    S.sweep_forward(path, M, N)


def test_fused_scan_option():
    S.check_fused_scan()


def test_fields_on_derivative_bases():
    S.check_fields_on_derivative_bases()


def test_fused_derivative_expressions():
    S.check_fused_derivative_expressions()
