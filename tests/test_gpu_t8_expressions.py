"""Stand-alone expression evaluation on the GPU (analysis tasks / flow properties of the stock Rayleigh-Benard script: vorticity,
np.sqrt(u@u)/nu, ...) against the unmodified reference (tests/golden/expressions.npz)."""
import pytest
import expression_cases as X

pytestmark = pytest.mark.gpu


def test_task_expressions_match_reference(golden):
    X.check_expressions(golden("expressions.npz"))


def test_flow_property_reductions_of_expressions(golden):
    X.check_flow_property_reductions(golden("expressions.npz"))


def test_boundary_conditions_with_data_match_reference(golden):
    import bc_cases, dedalus_b200 as d3
    bc_cases.check_bc_data(d3, golden("bc_data.npz"))


def test_right_hand_side_factors_without_a_basis_along_some_axis(golden):
    import bc_cases, dedalus_b200 as d3
    bc_cases.check_background(d3, golden("bc_data.npz"))


def test_left_hand_side_coefficients_varying_along_the_coupled_axis(golden):
    import bc_cases, dedalus_b200 as d3
    bc_cases.check_ncc(d3, golden("bc_data.npz"))


def test_right_hand_sides_with_grid_functions_and_derivatives_of_products(golden):
    import bc_cases, dedalus_b200 as d3
    bc_cases.check_conservative(d3, golden("bc_data.npz"))


def test_field_filters_norms_and_global_data(golden):
    X.check_field_helpers(golden("expressions.npz"))


def test_cartesian_lbvp_poisson_matches_reference(golden):
    import bc_cases, dedalus_b200 as d3
    bc_cases.check_poisson_lbvp(d3, golden("stock_scripts.npz"))


@pytest.mark.parametrize("tag", ["kdv", "rb2d", "shear", "shell"])
def test_stock_script_matches_reference(golden, tag, tmp_path):
    """The restated stock scripts (tests/stock_cases.py) with their CFL / flow-property main loops on the GPU."""
    import stock_cases
    g = golden("stock_scripts.npz")
    if tag == "kdv":
        stock_cases.check_kdv_burgers(g)
    else:
        stock_cases.check_stock_ivp(g, tag, tmp_path)


def test_rayleigh_benard_with_strong_flow_matches_reference(golden):
    import bc_cases, dedalus_b200 as d3
    bc_cases.check_strong(d3, golden("bc_data.npz"))


def test_3d_rayleigh_benard_with_strong_flow_matches_reference(golden):
    import bc_cases, dedalus_b200 as d3
    bc_cases.check_strong_3d(d3, golden("bc_data.npz"))


def test_sphere_right_hand_side_with_grid_function_and_forcing(golden):
    import bc_cases, dedalus_b200 as d3
    bc_cases.check_shallow_water_forced(d3, golden("bc_data.npz"))
