"""Chebyshev transforms at every basis order and fused derivative on the GPU, against the high-precision reference of
cheb_sweep_cases.py (the body test_emu_cheb_sweep.py runs through the emulation), plus the 192 and 384 register lengths."""
import pytest
import cheb_sweep_cases as S

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("path,M,N", [
    ("strided", 32, 48), ("strided", 15, 22), ("strided", 24, 16), ("strided", 21, 21), ("strided", 26, 39),
    ("lines", 32, 48), ("lines", 64, 96), ("lines", 15, 22), ("lines", 21, 21), ("lines", 20, 26),
    ("lines", 24, 16), ("lines", 17, 16),
    ("offset", 32, 48), ("offset", 15, 22),
    ("complex", 32, 48), ("complex", 24, 16)])
def test_backward_every_order_and_derivative(path, M, N):
    S.sweep_backward(path, M, N)


# rounding in the back-substitution grows with M (cheb_sweep_cases.TOL): up to 9 diagonals at these lengths
@pytest.mark.parametrize("path,M,N", [("strided", 128, 192), ("lines", 128, 192), ("lines", 256, 384), ("strided", 200, 384)])
def test_backward_register_lengths(path, M, N):
    S.sweep_backward(path, M, N, pairs=S.PAIRS_LOW)


@pytest.mark.parametrize("path,M,N", [("strided", 32, 48), ("strided", 24, 16), ("lines", 15, 22), ("lines", 32, 48),
                                      ("lines", 64, 96), ("lines", 128, 192)])
def test_forward_every_order(path, M, N):
    S.sweep_forward(path, M, N)


def test_fused_scan_option():
    S.check_fused_scan()


def test_fields_on_derivative_bases():
    S.check_fields_on_derivative_bases()


def test_fused_derivative_expressions():
    S.check_fused_derivative_expressions()
