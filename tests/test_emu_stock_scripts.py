"""The reference's stock example scripts, restated at reduced sizes (tests/stock_cases.py, bc_cases.py), executed through the CPU
emulation of the kernels against the unmodified reference executing its own scripts (tests/golden/stock_scripts.npz).  The sphere
script is covered in tests/test_emu_sphere.py."""
import pytest
import dedalus_b200 as d3
from emu import emu_lib as E
import bc_cases
import stock_cases


@pytest.fixture(autouse=True)
def emulation():
    E.install()
    yield
    E.uninstall()


@pytest.mark.parametrize("tag", ["kdv", "poisson", "rb2d", "shear", "shell"])
def test_stock_script_matches_reference(golden, tag, tmp_path):
    g = golden("stock_scripts.npz")
    if tag == "kdv":
        stock_cases.check_kdv_burgers(g)
    elif tag == "poisson":
        bc_cases.check_poisson_lbvp(d3, g)
    else:
        stock_cases.check_stock_ivp(g, tag, tmp_path)
