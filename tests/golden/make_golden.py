"""Generate the committed golden fixtures by running the UNMODIFIED reference (Dedalus v3.0.5,
/root/reference) single-process under tests/golden/ref_shim.py.

Run here (the build container), never on the GPU box:   python tests/golden/make_golden.py
Outputs: tests/golden/*.npz (small; committed).  Each fixture stores the inputs, the reference outputs and the
reference call that produced them, so tests can replay the same inputs through oracle/ and through the CUDA path.
"""
import sys, pathlib
import numpy as np
HERE = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(HERE))
import ref_shim
d3 = ref_shim.activate()
from scipy import sparse
from dedalus.core import transforms as rtr
from dedalus.core import basis as rbasis
from dedalus.core import timesteppers as rts


def natural_matrices(sp):
    """Reference pencil matrices expanded back to natural (field-major, un-permuted) ordering."""
    out = {}
    for name in ("M", "L"):
        mat = (sp.pre_left.T @ getattr(sp, name + "_min") @ sp.pre_right.T).tocoo()
        out[name] = mat
    return out


# ----------------------------------------------------------------------------------------------------------
# 1. Transform vectors (reference classes: ScipyRealFFT / RealFourierMMT / ScipyComplexFFT / ScipyFastChebyshev / JacobiMMT)
# ----------------------------------------------------------------------------------------------------------
def gen_transforms():
    rng = np.random.default_rng(1234)
    out = {}
    # Real Fourier: reference tests use N=16, dealias in {0.5, 1, 1.5} (tests/test_transforms.py:18-57); add odd and 3-D shapes
    for (M, N) in [(16, 8), (16, 16), (16, 24), (16, 21), (32, 48), (12, 18), (10, 15)]:
        for lib in ("scipy", "matrix"):
            plan = rbasis.RealFourier.transforms[lib](N, M)
            c = rng.standard_normal((3, M, 2))
            g = np.zeros((3, N, 2))
            plan.backward(c.copy(), g, 1)
            gg = rng.standard_normal((3, N, 2))
            cc = np.zeros((3, M, 2))
            plan.forward(gg.copy(), cc, 1)
            out[f"rf_{lib}_{M}_{N}_cin"] = c; out[f"rf_{lib}_{M}_{N}_gout"] = g
            out[f"rf_{lib}_{M}_{N}_gin"] = gg; out[f"rf_{lib}_{M}_{N}_cout"] = cc
    # Complex Fourier
    for (M, N) in [(16, 8), (16, 16), (16, 24), (15, 22), (12, 18)]:
        for lib in ("scipy", "matrix"):
            plan = rbasis.ComplexFourier.transforms[lib](N, M)
            c = rng.standard_normal((2, M, 3)) + 1j * rng.standard_normal((2, M, 3))
            g = np.zeros((2, N, 3), dtype=complex)
            plan.backward(c.copy(), g, 1)
            gg = rng.standard_normal((2, N, 3)) + 1j * rng.standard_normal((2, N, 3))
            cc = np.zeros((2, M, 3), dtype=complex)
            plan.forward(gg.copy(), cc, 1)
            out[f"cf_{lib}_{M}_{N}_cin"] = c; out[f"cf_{lib}_{M}_{N}_gout"] = g
            out[f"cf_{lib}_{M}_{N}_gin"] = gg; out[f"cf_{lib}_{M}_{N}_cout"] = cc
    # Chebyshev / ultraspherical with Chebyshev grid (tests/test_transforms.py:117-158: N in {15,16}, alpha in {0,1,2})
    for (M, N) in [(16, 8), (16, 16), (16, 24), (15, 22), (15, 15), (32, 48)]:
        for alpha in (0, 1, 2):
            a = b = alpha - 0.5
            for lib in ("scipy_dct", "matrix"):
                plan = rbasis.Jacobi.transforms[lib](N, M, a, b, -0.5, -0.5)
                c = rng.standard_normal((2, 3, M))
                g = np.zeros((2, 3, N))
                plan.backward(c.copy(), g, 2)
                gg = rng.standard_normal((2, 3, N))
                cc = np.zeros((2, 3, M))
                plan.forward(gg.copy(), cc, 2)
                key = f"ch_{lib}_{M}_{N}_{alpha}"
                out[key + "_cin"] = c; out[key + "_gout"] = g; out[key + "_gin"] = gg; out[key + "_cout"] = cc
    # Non-Chebyshev Jacobi (dense MMT, T4): Legendre and (a,b)=(1,0.5) on their own Gauss grids
    for (M, N) in [(16, 24), (12, 12)]:
        for (a, b) in [(0.0, 0.0), (1.0, 0.5)]:
            plan = rbasis.Jacobi.transforms["matrix"](N, M, a, b, a, b)
            out[f"jac_{M}_{N}_{a}_{b}_fwdmat"] = plan.forward_matrix
            out[f"jac_{M}_{N}_{a}_{b}_bwdmat"] = plan.backward_matrix
    # Jacobi helper quantities used in host matrix assembly
    from dedalus.tools import jacobi as tj
    for (a, b) in [(-0.5, -0.5), (0.5, 0.5), (1.5, 1.5), (0.0, 0.0)]:
        N = 12
        out[f"jop_D_{a}_{b}"] = tj.differentiation_matrix(N, a, b).toarray()
        out[f"jop_C_{a}_{b}"] = tj.conversion_matrix(N, a, b, a + 1, b + 1).toarray()
        out[f"jop_Z_{a}_{b}"] = tj.jacobi_matrix(N, a, b).toarray()
        out[f"jop_int_{a}_{b}"] = tj.integration_vector(N, a, b)
        out[f"jop_grid_{a}_{b}"] = tj.build_grid(N, a, b)
        out[f"jop_wts_{a}_{b}"] = tj.build_weights(N, a, b)
        out[f"jop_pm1_{a}_{b}"] = tj.build_polynomials(N, a, b, np.array([-1.0, 0.3, 1.0]))
    np.savez_compressed(HERE / "transforms.npz", **out)
    print("transforms.npz", len(out), "arrays")


# ----------------------------------------------------------------------------------------------------------
# 2. IVPs: KdV-Burgers (cfg 1), 2-D RB (cfg 2), 3-D RB (cfg 3) at oracle-friendly sizes
# ----------------------------------------------------------------------------------------------------------
def kdv(N=64, steps=20, tstep=2e-3, scheme="SBDF2"):
    # examples/ivp_1d_kdv_burgers/kdv_burgers.py:22-54
    Lx = 10; a = 1e-4; b = 2e-4
    xcoord = d3.Coordinate('x')
    dist = d3.Distributor(xcoord, dtype=np.float64)
    xbasis = d3.RealFourier(xcoord, size=N, bounds=(0, Lx), dealias=3/2)
    u = dist.Field(name='u', bases=xbasis)
    dx = lambda A: d3.Differentiate(A, xcoord)
    problem = d3.IVP([u], namespace=locals())
    problem.add_equation("dt(u) - a*dx(dx(u)) - b*dx(dx(dx(u))) = - u*dx(u)")
    x = dist.local_grid(xbasis)
    n = 20
    u['g'] = np.log(1 + np.cosh(n)**2/np.cosh(n*(x-0.2*Lx))**2) / (2*n)
    solver = problem.build_solver(getattr(d3, scheme))
    u0 = u['c'].copy()
    for i in range(steps):
        solver.step(tstep)
    return dict(u0_c=u0, u_c=u['c'].copy(), u_g=u['g'].copy(), N=N, steps=steps, dt=tstep, scheme=scheme)


def rb(dim, Nh, Nz, steps, tstep, Ra, scheme="RK222", dump_pencils=(), return_solver=False):
    # examples/ivp_2d_rayleigh_benard/rayleigh_benard.py:33-89 (2-D) and SURVEY.md Appendix C (3-D)
    Lx = Ly = 4; Lz = 1; Pr = 1
    names = ('x', 'z') if dim == 2 else ('x', 'y', 'z')
    coords = d3.CartesianCoordinates(*names)
    dist = d3.Distributor(coords, dtype=np.float64)
    hb = [d3.RealFourier(coords[n], size=Nh, bounds=(0, Lx), dealias=3/2) for n in names[:-1]]
    zb = d3.ChebyshevT(coords['z'], size=Nz, bounds=(0, Lz), dealias=3/2)
    bases = tuple(hb) + (zb,)
    p = dist.Field(name='p', bases=bases); b = dist.Field(name='b', bases=bases)
    u = dist.VectorField(coords, name='u', bases=bases)
    tau_p = dist.Field(name='tau_p')
    tau_b1 = dist.Field(name='tau_b1', bases=tuple(hb)); tau_b2 = dist.Field(name='tau_b2', bases=tuple(hb))
    tau_u1 = dist.VectorField(coords, name='tau_u1', bases=tuple(hb)); tau_u2 = dist.VectorField(coords, name='tau_u2', bases=tuple(hb))
    kappa = (Ra * Pr)**(-1/2); nu = (Ra / Pr)**(-1/2)
    grids = dist.local_grids(*bases); z = grids[-1]
    ez = coords.unit_vector_fields(dist)[-1]
    lift_basis = zb.derivative_basis(1)
    lift = lambda A: d3.Lift(A, lift_basis, -1)
    grad_u = d3.grad(u) + ez*lift(tau_u1); grad_b = d3.grad(b) + ez*lift(tau_b1)
    problem = d3.IVP([p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2], namespace=locals())
    problem.add_equation("trace(grad_u) + tau_p = 0")
    problem.add_equation("dt(b) - kappa*div(grad_b) + lift(tau_b2) = - u@grad(b)")
    problem.add_equation("dt(u) - nu*div(grad_u) + grad(p) - b*ez + lift(tau_u2) = - u@grad(u)")
    problem.add_equation("b(z=0) = Lz"); problem.add_equation("u(z=0) = 0")
    problem.add_equation("b(z=Lz) = 0"); problem.add_equation("u(z=Lz) = 0")
    problem.add_equation("integ(p) = 0")
    solver = problem.build_solver(getattr(d3, scheme))
    b.fill_random('g', seed=42, distribution='normal', scale=1e-3)
    b['g'] *= z * (Lz - z); b['g'] += Lz - z
    out = dict(dim=dim, Nh=Nh, Nz=Nz, steps=steps, dt=tstep, Ra=Ra, scheme=scheme)
    out['b0_c'] = b['c'].copy()
    out['b0_g1'] = b['g'].copy()     # dealias-scale grid values? (scales=1 after fill_random + item access)
    # pencil matrices in natural ordering
    for grp in dump_pencils:
        sp = [s for s in solver.subproblems if tuple(g for g in s.group if g is not None) == tuple(grp)][0]
        nat = natural_matrices(sp)
        tag = "pen_" + "_".join(str(g) for g in grp)
        for name, mat in nat.items():
            out[f"{tag}_{name}_row"] = mat.row.astype(np.int32); out[f"{tag}_{name}_col"] = mat.col.astype(np.int32)
            out[f"{tag}_{name}_val"] = mat.data; out[f"{tag}_{name}_shape"] = np.array(mat.shape)
        out[f"{tag}_valid_rows"] = np.asarray(sp.pre_left.sum(axis=0)).ravel().astype(bool)
        out[f"{tag}_valid_cols"] = np.asarray(sp.pre_right.sum(axis=1)).ravel().astype(bool)
    # F evaluation at the initial state (stage-1 RHS fields), after one evaluate of the F group
    solver.evaluator.evaluate_group('F')
    for i, F in enumerate(solver.F):
        F.change_layout('c') if hasattr(F, 'change_layout') else None
        out[f"F0_{i}"] = np.array(F['c']) if hasattr(F, '__getitem__') else np.array(F)
    state_hist = []
    for i in range(steps):
        solver.step(tstep)
        if i == 0:
            for f in (p, b, u):
                out[f"{f.name}_c_step1"] = f['c'].copy()
    for f in (p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2):
        out[f"{f.name}_c"] = f['c'].copy()
    out['checks'] = np.array([np.sum(b['c']**2), np.sum(p['c']**2), np.sum(u['c']**2)])
    if return_solver:
        return out, solver
    return out


def heat(scheme, N=8, steps=20):
    # tests/test_ivp.py:20-49 (complex Fourier heat equation, every timestepper)
    xcoord = d3.Coordinate('x')
    dist = d3.Distributor(xcoord, dtype=np.complex128)
    xbasis = d3.ComplexFourier(xcoord, size=N, bounds=(0, 2*np.pi))
    u = dist.Field(name='u', bases=xbasis); F = dist.Field(name='F', bases=xbasis)
    x = dist.local_grid(xbasis)
    F['g'] = -np.sin(x)
    dx = lambda A: d3.Differentiate(A, xcoord)
    problem = d3.IVP([u], namespace=locals())
    problem.add_equation("-dt(u) + dx(dx(u)) = F")
    solver = problem.build_solver(scheme)
    for i in range(steps):
        solver.step(1e-5)
    return u['c'].copy()


def gen_ivps():
    out = {}
    for k, v in kdv().items(): out["kdv_" + k] = v
    for k, v in kdv(N=32, steps=8, tstep=1e-3, scheme="RK443").items(): out["kdv443_" + k] = v
    np.savez_compressed(HERE / "kdv.npz", **out)
    r2 = rb(2, 16, 16, steps=5, tstep=0.01, Ra=2e6, dump_pencils=[(0,), (1,), (5,)])
    np.savez_compressed(HERE / "rb2d_16x16.npz", **r2)
    r3 = rb(3, 8, 8, steps=5, tstep=0.01, Ra=1e6, dump_pencils=[(0, 0), (0, 2), (3, 0), (1, 2)])
    np.savez_compressed(HERE / "rb3d_8.npz", **r3)
    r3s = rb(3, 8, 12, steps=3, tstep=0.02, Ra=1e5, scheme="SBDF2")
    np.savez_compressed(HERE / "rb3d_8x8x12_sbdf2.npz", **{k: v for k, v in r3s.items() if not k.startswith('pen_')})
    # Known-answer checksums at larger sizes (SURVEY.md section 8c): only the three sums are stored
    chk = {}
    c2 = rb(2, 256, 128, steps=10, tstep=0.01, Ra=2e6)
    chk['rb2d_256x128_10steps'] = c2['checks']
    c3 = rb(3, 32, 32, steps=10, tstep=0.01, Ra=1e6)
    chk['rb3d_32_10steps'] = c3['checks']
    k = kdv(N=1024, steps=200, tstep=2e-3)
    chk['kdv_1024_200steps_maxabs'] = np.array([np.max(np.abs(k['u_g']))])
    heat_out = {}
    for name, scheme in rts.schemes.items():
        heat_out['heat_' + name] = heat(scheme)
    np.savez_compressed(HERE / "checks.npz", **chk, **heat_out)
    print({k: v for k, v in chk.items()})


def gen_transforms_bench():
    """Reference transform outputs AT THE BENCHMARK LINE LENGTHS (256 -> 384 and 128 -> 192, dealias 3/2) in layouts the
    register-resident kernels take: real Fourier on a strided axis with 16 lines, Chebyshev on contiguous lines (alpha 0 and 2)."""
    rng = np.random.default_rng(4321)
    out = {}
    for (M, N) in [(256, 384), (128, 192)]:
        plan = rbasis.RealFourier.transforms["scipy"](N, M)
        c = rng.standard_normal((1, M, 16)); c[:, 1, :] = 0
        g = np.zeros((1, N, 16)); plan.backward(c.copy(), g, 1)
        gg = rng.standard_normal((1, N, 16)); cc = np.zeros((1, M, 16)); plan.forward(gg.copy(), cc, 1)
        out[f"rf_{M}_{N}_cin"] = c; out[f"rf_{M}_{N}_gout"] = g; out[f"rf_{M}_{N}_gin"] = gg; out[f"rf_{M}_{N}_cout"] = cc
        for alpha in ((0, 2) if M == 256 else (2,)):
            a = alpha - 0.5
            plan = rbasis.Jacobi.transforms["scipy_dct"](N, M, a, a, -0.5, -0.5)
            c = rng.standard_normal((17, M)); g = np.zeros((17, N)); plan.backward(c.copy(), g, 1)
            gg = rng.standard_normal((17, N)); cc = np.zeros((17, M)); plan.forward(gg.copy(), cc, 1)
            key = f"ch_{M}_{N}_{alpha}"
            out[key + "_cin"] = c; out[key + "_gout"] = g; out[key + "_gin"] = gg; out[key + "_cout"] = cc
    np.savez_compressed(HERE / "transforms_bench.npz", **out)
    print("transforms_bench.npz", len(out), "arrays")


def gen_rb3d_16():
    """16^3 (24-point dealiased lines: the smallest size at which the register-resident FFT / Chebyshev kernels run)."""
    r = rb(3, 16, 16, steps=3, tstep=0.01, Ra=1e6)
    np.savez_compressed(HERE / "rb3d_16.npz", **{k: v for k, v in r.items() if not k.startswith('pen_')})


if __name__ == "__main__" and ("rb3d_16" in sys.argv[1:] or "transforms_bench" in sys.argv[1:]):
    if "rb3d_16" in sys.argv[1:]: gen_rb3d_16()
    if "transforms_bench" in sys.argv[1:]: gen_transforms_bench()
    sys.exit(0)

if __name__ == "__main__":
    which = sys.argv[1:] or ["transforms", "ivps"]
    if "transforms" in which: gen_transforms()
    if "ivps" in which: gen_ivps()


def gen_cfl():
    """2-D RB with the reference CFL controller (extras/flow_tools.py:139-233): dt sequence and final state."""
    Lx, Lz, Ra, Pr, Nh, Nz = 4, 1, 2e6, 1, 32, 16
    coords = d3.CartesianCoordinates('x', 'z')
    dist = d3.Distributor(coords, dtype=np.float64)
    xb = d3.RealFourier(coords['x'], size=Nh, bounds=(0, Lx), dealias=3/2)
    zb = d3.ChebyshevT(coords['z'], size=Nz, bounds=(0, Lz), dealias=3/2)
    p = dist.Field(name='p', bases=(xb, zb)); b = dist.Field(name='b', bases=(xb, zb)); u = dist.VectorField(coords, name='u', bases=(xb, zb))
    tau_p = dist.Field(name='tau_p'); tau_b1 = dist.Field(name='tau_b1', bases=xb); tau_b2 = dist.Field(name='tau_b2', bases=xb)
    tau_u1 = dist.VectorField(coords, name='tau_u1', bases=xb); tau_u2 = dist.VectorField(coords, name='tau_u2', bases=xb)
    kappa = (Ra * Pr)**(-1/2); nu = (Ra / Pr)**(-1/2)
    x, z = dist.local_grids(xb, zb); ex, ez = coords.unit_vector_fields(dist)
    lift_basis = zb.derivative_basis(1); lift = lambda A: d3.Lift(A, lift_basis, -1)
    grad_u = d3.grad(u) + ez*lift(tau_u1); grad_b = d3.grad(b) + ez*lift(tau_b1)
    problem = d3.IVP([p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2], namespace=locals())
    problem.add_equation("trace(grad_u) + tau_p = 0")
    problem.add_equation("dt(b) - kappa*div(grad_b) + lift(tau_b2) = - u@grad(b)")
    problem.add_equation("dt(u) - nu*div(grad_u) + grad(p) - b*ez + lift(tau_u2) = - u@grad(u)")
    problem.add_equation("b(z=0) = Lz"); problem.add_equation("u(z=0) = 0"); problem.add_equation("b(z=Lz) = 0"); problem.add_equation("u(z=Lz) = 0")
    problem.add_equation("integ(p) = 0")
    solver = problem.build_solver(d3.RK222)
    b.fill_random('g', seed=42, distribution='normal', scale=1e-3); b['g'] *= z * (Lz - z); b['g'] += Lz - z
    u['g'][0] = 3.0 * np.sin(2 * np.pi * x / Lx) * z * (Lz - z) * 4
    u['g'][1] = 1.0 * np.cos(2 * np.pi * x / Lx) * np.sin(np.pi * z / Lz)
    CFL = d3.CFL(solver, initial_dt=0.01, cadence=2, safety=0.5, threshold=0.05, max_change=1.5, min_change=0.5, max_dt=0.05)
    CFL.add_velocity(u)
    out = dict(b0_c=b['c'].copy(), u0_c=u['c'].copy())
    dts = []
    for i in range(12):
        tstep = CFL.compute_timestep()
        dts.append(tstep)
        solver.step(tstep)
    out['dts'] = np.array(dts)
    out['b_c'] = b['c'].copy(); out['u_c'] = u['c'].copy()
    np.savez_compressed(HERE / "rb2d_cfl.npz", **out)
    print("cfl dts", dts)


if __name__ == "__main__" and "cfl" in sys.argv[1:]:
    gen_cfl()


def gen_swsh():
    """SWSH colatitude transform (reference core/transforms.py:1251-1340, matrices from libraries/dedalus_sphere/sphere.py:43-64
    x Gauss weights): the reference's own plan objects on its own m_maps (real dtype: cos / -sin pairs per m, folded
    triangular coefficient packing, core/basis.py:2800-2809, 2940-2970), forward and backward, spin weights -2 .. 2, with and
    without 3/2 dealiasing.  Stored: the m_maps as integer rows (m, mg0, mg1, mc0, mc1, ell_start, ell_stop_or_-1, ell_step),
    inputs, outputs and two of the matrices."""
    rng = np.random.default_rng(77)
    out = {}
    for tag, (Nphi, Ntheta, dealias) in dict(a=(16, 12, 1), b=(32, 16, 1.5)).items():
        coords = d3.S2Coordinates('phi', 'theta')
        dist = d3.Distributor(coords, dtype=np.float64)
        basis = d3.SphereBasis(coords, (Nphi, Ntheta), radius=1, dealias=(dealias, dealias), dtype=np.float64)
        f = dist.Field(bases=basis)
        f.preset_scales(dealias)
        gshape = tuple(int(n) for n in basis.grid_shape((dealias, dealias)))
        mm = basis.m_maps(dist)
        rows = []
        for m, mg, mc, ell in mm:
            rows.append((int(m), int(mg.start), int(mg.stop), int(mc.start), int(mc.stop), int(ell.start),
                         -1 if ell.stop is None else int(ell.stop), -1 if ell.step == -1 else 1))
        cshape = tuple(int(n) for n in f['c'].shape)
        out[f"{tag}_m_maps"] = np.array(rows, dtype=np.int64)
        out[f"{tag}_meta"] = np.array([Nphi, Ntheta, basis.Lmax, gshape[0], gshape[1], cshape[0], cshape[1]], dtype=np.int64)
        for s in (0, 1, -1, 2, -2):
            plan = basis.transform_plan(dist, gshape[1], s)
            # arrays as the reference passes them for a rank-|s| component: (1, Nphi_cg, Ntheta_g) <-> (1, Nphi_c, Nell)
            g = rng.standard_normal((2, gshape[0], gshape[1]))
            c = np.zeros((2,) + cshape)
            plan.forward(g.copy(), c, 2)
            cc = rng.standard_normal((2,) + cshape)
            gg = np.full((2, gshape[0], gshape[1]), np.nan)
            plan.backward(cc.copy(), gg, 2)
            out[f"{tag}_s{s}_gin"] = g; out[f"{tag}_s{s}_cout"] = c
            out[f"{tag}_s{s}_cin"] = cc; out[f"{tag}_s{s}_gout"] = gg
            if s in (0, 2):
                for m in (0, 3):
                    out[f"{tag}_s{s}_m{m}_fwdmat"] = np.array(plan._forward_SWSH_matrices[m])
                    out[f"{tag}_s{s}_m{m}_bwdmat"] = np.array(plan._backward_SWSH_matrices[m])
    np.savez_compressed(HERE / "swsh.npz", **out)
    print({k: v.shape for k, v in out.items() if k.endswith("m_maps") or k.endswith("meta")})


if __name__ == "__main__" and "swsh" in sys.argv[1:]:
    gen_swsh()


# ----------------------------------------------------------------------------------------------------------
# Sphere (S2) fields and the shallow-water IVP of examples/ivp_sphere_shallow_water (config 4)
# ----------------------------------------------------------------------------------------------------------
def shallow_water(Nphi, Ntheta, steps, scheme="RK222", dump_mats=(), dealias=3/2):
    """The stock script's problem (examples/ivp_sphere_shallow_water/shallow_water.py:25-86) with the zonal-jet + height
    perturbation initial condition evaluated analytically (the LBVP for the balanced height is not part of the IVP path)."""
    meter = 1 / 6.37122e6; hour = 1; second = hour / 3600
    R = 6.37122e6 * meter; Omega = 7.292e-5 / second; nu = 1e5 * meter**2 / second / 32**2
    g = 9.80616 * meter / second**2; H = 1e4 * meter; timestep = 600 * second * min(1.0, 128 / Ntheta)
    coords = d3.S2Coordinates('phi', 'theta')
    dist = d3.Distributor(coords, dtype=np.float64)
    basis = d3.SphereBasis(coords, (Nphi, Ntheta), radius=R, dealias=dealias, dtype=np.float64)
    u = dist.VectorField(coords, name='u', bases=basis)
    h = dist.Field(name='h', bases=basis)
    zcross = lambda A: d3.MulCosine(d3.skew(A))
    phi, theta = dist.local_grids(basis)
    lat = np.pi / 2 - theta + 0*phi
    umax = 80 * meter / second
    lat0 = np.pi / 7; lat1 = np.pi / 2 - lat0
    en = np.exp(-4 / (lat1 - lat0)**2)
    jet = (lat0 <= lat) * (lat <= lat1)
    u_jet = umax / en * np.exp(1 / (lat[jet] - lat0) / (lat[jet] - lat1))
    u['g'][0][jet] = u_jet
    lat2 = np.pi / 4; hpert = 120 * meter; alpha = 1 / 3; beta = 1 / 15
    h['g'] += hpert * np.cos(lat) * np.exp(-(phi/alpha)**2) * np.exp(-((lat2-lat)/beta)**2)
    out = dict(u0=u['c'].copy(), h0=h['c'].copy(), meta=np.array([Nphi, Ntheta, dealias, steps, timestep]))
    problem = d3.IVP([u, h], namespace=locals())
    problem.add_equation("dt(u) + nu*lap(lap(u)) + g*grad(h) + 2*Omega*zcross(u) = - u@grad(u)")
    problem.add_equation("dt(h) + nu*lap(lap(h)) + H*div(u) = - div(h*u)")
    solver = problem.build_solver(getattr(d3, scheme))
    for sp in solver.subproblems:
        m = sp.group[0]
        if m in dump_mats:
            nat = natural_matrices(sp)
            for name in ("M", "L"):
                out[f"m{m}_{name}"] = nat[name].toarray()
    for i in range(steps):
        solver.step(timestep)
    out.update(u1=u['c'].copy(), h1=h['c'].copy())
    # analysis tasks of the stock script (lines 90-92): vorticity, and a Laplacian, evaluated on the final state
    v = (-d3.div(d3.skew(u))).evaluate(); v.change_layout('c')
    l = d3.lap(h).evaluate(); l.change_layout('c')
    out.update(vort1=v.data.copy(), laph1=l.data.copy())
    return out


def gen_sphere():
    """(1) random grid data of scalar / vector / rank-2 fields -> coefficients -> grid through the reference's own transform
    chain (azimuthal FFT, spin recombination, SWSH colatitude transform) incl. the folded triangular packing with shift > 0;
    (2) shallow-water states after K steps at 16 x 8 (RK222, with three pencil matrices), 32 x 16 (RK222 and SBDF2);
    (3) config 4's size (512 x 256, Lmax = 254): checksums and one m-line of the state after 3 RK222 steps."""
    out = {}
    for tag, (Nphi, Ntheta, dealias) in dict(a=(16, 8, 1.5), b=(32, 24, 1.0)).items():
        coords = d3.S2Coordinates('phi', 'theta')
        dist = d3.Distributor(coords, dtype=np.float64)
        basis = d3.SphereBasis(coords, (Nphi, Ntheta), radius=1.7, dealias=dealias, dtype=np.float64)
        phi, theta = dist.local_grids(basis, scales=(dealias, dealias))
        out[f"f{tag}_meta"] = np.array([Nphi, Ntheta, dealias])
        out[f"f{tag}_phi"] = phi.ravel(); out[f"f{tag}_theta"] = theta.ravel()
        rng = np.random.default_rng(5)
        for name, f in (("s", dist.Field(bases=basis)), ("v", dist.VectorField(coords, bases=basis)),
                        ("t", dist.TensorField((coords, coords), bases=basis))):
            f.preset_scales(dealias)
            g = rng.standard_normal(f['g'].shape)
            f['g'] = g
            c = f['c'].copy()
            g2 = f['g'].copy()
            out[f"f{tag}_{name}_gin"] = g; out[f"f{tag}_{name}_c"] = c; out[f"f{tag}_{name}_g2"] = g2
    for tag, kw in dict(sw16=dict(Nphi=16, Ntheta=8, steps=3, dump_mats=(0, 1, 5)), sw32=dict(Nphi=32, Ntheta=16, steps=5),
                        sw32sbdf2=dict(Nphi=32, Ntheta=16, steps=6, scheme="SBDF2")).items():
        for k, v in shallow_water(**kw).items():
            out[f"{tag}_{k}"] = v
    big = shallow_water(512, 256, 3)
    out["sw512_meta"] = big["meta"]
    for name in ("u", "h"):
        a = big[name + "1"]
        out[f"sw512_{name}1_sumsq"] = np.array(np.sum(a.astype(np.longdouble)**2), dtype=np.float64)
        out[f"sw512_{name}1_absmax"] = np.abs(a).max()
        out[f"sw512_{name}1_rows"] = a[..., 20:24, :].copy()        # m = 10, 11 (and the folded partners 245, 244)
    np.savez_compressed(HERE / "sphere.npz", **out)
    print({k: getattr(v, 'shape', v) for k, v in out.items() if 'meta' in k or 'sumsq' in k})


if __name__ == "__main__" and "sphere" in sys.argv[1:]:
    gen_sphere()


def shallow_water_balanced(Nphi, Ntheta, steps, dealias=3/2):
    """The stock script start to finish (examples/ivp_sphere_shallow_water/shallow_water.py:45-86): zonal jet, the LBVP for the
    balanced height with its gauge constant, the height perturbation, then `steps` RK222 steps."""
    meter = 1 / 6.37122e6; hour = 1; second = hour / 3600
    R = 6.37122e6 * meter; Omega = 7.292e-5 / second; nu = 1e5 * meter**2 / second / 32**2
    g = 9.80616 * meter / second**2; H = 1e4 * meter; timestep = 600 * second * min(1.0, 128 / Ntheta)
    coords = d3.S2Coordinates('phi', 'theta')
    dist = d3.Distributor(coords, dtype=np.float64)
    basis = d3.SphereBasis(coords, (Nphi, Ntheta), radius=R, dealias=dealias, dtype=np.float64)
    u = dist.VectorField(coords, name='u', bases=basis)
    h = dist.Field(name='h', bases=basis)
    zcross = lambda A: d3.MulCosine(d3.skew(A))
    phi, theta = dist.local_grids(basis)
    lat = np.pi / 2 - theta + 0*phi
    umax = 80 * meter / second
    lat0 = np.pi / 7; lat1 = np.pi / 2 - lat0
    en = np.exp(-4 / (lat1 - lat0)**2)
    jet = (lat0 <= lat) * (lat <= lat1)
    u_jet = umax / en * np.exp(1 / (lat[jet] - lat0) / (lat[jet] - lat1))
    u['g'][0][jet] = u_jet
    c = dist.Field(name='c')
    problem = d3.LBVP([h, c], namespace=locals())
    problem.add_equation("g*lap(h) + c = - div(u@grad(u) + 2*Omega*zcross(u))")
    problem.add_equation("ave(h) = 0")
    solver = problem.build_solver()
    solver.solve()
    out = dict(meta=np.array([Nphi, Ntheta, dealias, steps, timestep]), h_bal=h['c'].copy(), c_bal=c['c'].copy(), u_bal=u['c'].copy())
    lat2 = np.pi / 4; hpert = 120 * meter; alpha = 1 / 3; beta = 1 / 15
    h.change_scales(1); u.change_scales(1)
    h['g'] += hpert * np.cos(lat) * np.exp(-(phi/alpha)**2) * np.exp(-((lat2-lat)/beta)**2)
    problem = d3.IVP([u, h], namespace=locals())
    problem.add_equation("dt(u) + nu*lap(lap(u)) + g*grad(h) + 2*Omega*zcross(u) = - u@grad(u)")
    problem.add_equation("dt(h) + nu*lap(lap(h)) + H*div(u) = - div(h*u)")
    solver = problem.build_solver(d3.RK222)
    out.update(u0=u['c'].copy(), h0=h['c'].copy())
    for i in range(steps):
        solver.step(timestep)
    out.update(u1=u['c'].copy(), h1=h['c'].copy())
    return out


def gen_sphere_lbvp():
    out = {}
    for tag, kw in dict(bal32=dict(Nphi=32, Ntheta=16, steps=3), bal64=dict(Nphi=64, Ntheta=32, steps=2)).items():
        for k, v in shallow_water_balanced(**kw).items():
            out[f"{tag}_{k}"] = v
    np.savez_compressed(HERE / "sphere_lbvp.npz", **out)
    print({k: (v.shape, float(np.abs(v).max())) for k, v in out.items()})


if __name__ == "__main__" and "sphere_lbvp" in sys.argv[1:]:
    gen_sphere_lbvp()


# ----------------------------------------------------------------------------------------------------------
# Complex-dtype pencil path (T3): ComplexFourier x ChebyshevT in complex128, complex LHS coefficients, cubic RHS
# ----------------------------------------------------------------------------------------------------------
def complex_cgl(scheme, steps, tstep=1e-3, Nx=16, Nz=12):
    coords = d3.CartesianCoordinates('x', 'z')
    dist = d3.Distributor(coords, dtype=np.complex128)
    xb = d3.ComplexFourier(coords['x'], size=Nx, bounds=(0, 2 * np.pi), dealias=3/2)
    zb = d3.ChebyshevT(coords['z'], size=Nz, bounds=(0, 1), dealias=3/2)
    u = dist.Field(name='u', bases=(xb, zb))
    tau1 = dist.Field(name='tau1', bases=xb)
    tau2 = dist.Field(name='tau2', bases=xb)
    lift_basis = zb.derivative_basis(2)
    lift = lambda A, n: d3.Lift(A, lift_basis, n)
    dx = lambda A: d3.Differentiate(A, coords['x'])
    c1, c2 = 0.3 + 0.2j, 1.0 - 0.5j
    x, z = dist.local_grids(xb, zb)
    u.fill_random('g', seed=3, distribution='normal', scale=0.1)
    u['g'] *= z * (1 - z)
    out = dict(u0=u['c'].copy(), meta=np.array([Nx, Nz, steps, tstep]))
    problem = d3.IVP([u, tau1, tau2], namespace=locals())
    problem.add_equation("dt(u) - c1*lap(u) + (0.5j)*dx(u) + lift(tau1,-1) + lift(tau2,-2) = - c2*u*dx(u) + u*u*u")
    problem.add_equation("u(z=0) = 0")
    problem.add_equation("u(z=1) = 0")
    solver = problem.build_solver(getattr(d3, scheme))
    for i in range(steps):
        solver.step(tstep)
    out.update(u1=u['c'].copy(), tau1=tau1['c'].copy(), tau2=tau2['c'].copy())
    return out


def gen_complex():
    out = {}
    for tag, (scheme, steps) in dict(rk222=("RK222", 5), sbdf2=("SBDF2", 6)).items():
        for k, v in complex_cgl(scheme, steps).items():
            out[f"{tag}_{k}"] = v
    np.savez_compressed(HERE / "complex_cgl.npz", **out)
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__" and "complex" in sys.argv[1:]:
    gen_complex()


# ----------------------------------------------------------------------------------------------------------
# Spherical-shell field transforms (T6: core/basis.py:4474-4508 on top of the sphere chain)
# ----------------------------------------------------------------------------------------------------------
def gen_shell():
    """Random grid data of scalar / vector / rank-2 fields on a ShellBasis -> coefficients -> grid through the reference.
    Case b has the folded (m, l) packing with shift > 0 and an ODD Lmax: for even Lmax and shift > 0 the reference's ell_maps merge
    the m = 0 row and the folded rows of l = Lmax / 2 into one slice that also covers the rows of another degree, which then get
    two regularity recombinations (a reference oddity, not reproduced).  Case c: a k = 1 (derivative) basis."""
    out = {}
    for tag, (shape, dealias, k) in dict(a=((16, 8, 6), 1.5, 0), b=((32, 23, 8), 1.0, 0), c=((16, 8, 6), 1.5, 1)).items():
        coords = d3.SphericalCoordinates('phi', 'theta', 'r')
        dist = d3.Distributor(coords, dtype=np.float64)
        shell = d3.ShellBasis(coords, shape=shape, radii=(1.2, 2.7), dealias=dealias, dtype=np.float64, k=k)
        phi, theta, r = dist.local_grids(shell, scales=(dealias,) * 3)
        out[f"{tag}_meta"] = np.array(list(shape) + [dealias, k])
        out[f"{tag}_phi"] = phi.ravel(); out[f"{tag}_theta"] = theta.ravel(); out[f"{tag}_r"] = r.ravel()
        rng = np.random.default_rng(11)
        for name, f in (("s", dist.Field(bases=shell)), ("v", dist.VectorField(coords, bases=shell)),
                        ("t", dist.TensorField((coords, coords), bases=shell))):
            f.preset_scales(dealias)
            g = rng.standard_normal(f['g'].shape)
            f['g'] = g
            c = f['c'].copy()
            g2 = f['g'].copy()
            out[f"{tag}_{name}_c"] = c; out[f"{tag}_{name}_g2"] = g2        # the input g is regenerated from the seed by the test
    # the rank-2 field of case b in a file of its own: each file stays under 1 MB
    np.savez_compressed(HERE / "shell.npz", **{k: v for k, v in out.items() if not k.startswith("b_t_")})
    np.savez_compressed(HERE / "shell_rank2.npz", **{k: v for k, v in out.items() if k.startswith("b_t_")})
    print({k: v.shape for k, v in out.items() if k.endswith("_c")})


if __name__ == "__main__" and "shell" in sys.argv[1:]:
    gen_shell()


# ----------------------------------------------------------------------------------------------------------
# Shell convection IVP (BASELINE config 5: examples/ivp_shell_convection/shell_convection.py)
# ----------------------------------------------------------------------------------------------------------
def shell_convection(shape, steps, scheme="SBDF2", tstep=0.05, dump=()):
    Ri, Ro = 14, 15
    Nphi, Ntheta, Nr = shape
    Rayleigh = 3500; Prandtl = 1; dealias = 3/2
    coords = d3.SphericalCoordinates('phi', 'theta', 'r')
    dist = d3.Distributor(coords, dtype=np.float64)
    shell = d3.ShellBasis(coords, shape=(Nphi, Ntheta, Nr), radii=(Ri, Ro), dealias=dealias, dtype=np.float64)
    sphere = shell.outer_surface
    p = dist.Field(name='p', bases=shell); b = dist.Field(name='b', bases=shell)
    u = dist.VectorField(coords, name='u', bases=shell)
    tau_p = dist.Field(name='tau_p')
    tau_b1 = dist.Field(name='tau_b1', bases=sphere); tau_b2 = dist.Field(name='tau_b2', bases=sphere)
    tau_u1 = dist.VectorField(coords, name='tau_u1', bases=sphere); tau_u2 = dist.VectorField(coords, name='tau_u2', bases=sphere)
    kappa = (Rayleigh * Prandtl)**(-1/2); nu = (Rayleigh / Prandtl)**(-1/2)
    phi, theta, r = dist.local_grids(shell)
    er = dist.VectorField(coords, bases=shell.radial_basis); er['g'][2] = 1
    rvec = dist.VectorField(coords, bases=shell.radial_basis); rvec['g'][2] = r
    lift_basis = shell.derivative_basis(1)
    lift = lambda A: d3.Lift(A, lift_basis, -1)
    grad_u = d3.grad(u) + rvec*lift(tau_u1)
    grad_b = d3.grad(b) + rvec*lift(tau_b1)
    problem = d3.IVP([p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2], namespace=locals())
    problem.add_equation("trace(grad_u) + tau_p = 0")
    problem.add_equation("dt(b) - kappa*div(grad_b) + lift(tau_b2) = - u@grad(b)")
    problem.add_equation("dt(u) - nu*div(grad_u) + grad(p) - b*er + lift(tau_u2) = - u@grad(u)")
    problem.add_equation("b(r=Ri) = 1"); problem.add_equation("u(r=Ri) = 0")
    problem.add_equation("b(r=Ro) = 0"); problem.add_equation("u(r=Ro) = 0")
    problem.add_equation("integ(p) = 0")
    solver = problem.build_solver(getattr(d3, scheme))
    b.fill_random('g', seed=42, distribution='normal', scale=1e-3)
    b['g'] *= (r - Ri) * (Ro - r)
    b['g'] += (Ri - Ri*Ro/r) / (Ri - Ro)
    out = dict(b0=b['c'].copy(), meta=np.array(list(shape) + [steps, tstep]))
    for sp in solver.subproblems:
        ell = sp.group[1]
        if ell in dump:
            nat = natural_matrices(sp)
            for name in ("M", "L"):
                out[f"l{ell}_{name}"] = nat[name].toarray()
    for i in range(steps):
        solver.step(tstep)
    for f in (p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2):
        out[f.name + "1"] = f['c'].copy()
    return out


def shell_convection_strong(shape=(16, 8, 6), steps=3, tstep=0.02, forced=False):
    """Shell convection started from the state of tests/golden/shell_tasks.npz with the velocity amplified to O(0.1): the advection
    terms are then as large as the linear ones, which exposes the order of truncations in the right-hand side (the fixtures above
    start from noise and keep |u| ~ 1e-6 |b|)."""
    g = np.load(HERE / "shell_tasks.npz")
    Ri, Ro = 14, 15
    Nphi, Ntheta, Nr = shape
    Rayleigh = 3500; Prandtl = 1; dealias = 3/2
    coords = d3.SphericalCoordinates('phi', 'theta', 'r')
    dist = d3.Distributor(coords, dtype=np.float64)
    shell = d3.ShellBasis(coords, shape=(Nphi, Ntheta, Nr), radii=(Ri, Ro), dealias=dealias, dtype=np.float64)
    sphere = shell.outer_surface
    p = dist.Field(name='p', bases=shell); b = dist.Field(name='b', bases=shell)
    u = dist.VectorField(coords, name='u', bases=shell)
    tau_p = dist.Field(name='tau_p')
    tau_b1 = dist.Field(name='tau_b1', bases=sphere); tau_b2 = dist.Field(name='tau_b2', bases=sphere)
    tau_u1 = dist.VectorField(coords, name='tau_u1', bases=sphere); tau_u2 = dist.VectorField(coords, name='tau_u2', bases=sphere)
    kappa = (Rayleigh * Prandtl)**(-1/2); nu = (Rayleigh / Prandtl)**(-1/2)
    phi, theta, r = dist.local_grids(shell)
    er = dist.VectorField(coords, bases=shell.radial_basis); er['g'][2] = 1
    rvec = dist.VectorField(coords, bases=shell.radial_basis); rvec['g'][2] = r
    lift_basis = shell.derivative_basis(1)
    lift = lambda A: d3.Lift(A, lift_basis, -1)
    grad_u = d3.grad(u) + rvec*lift(tau_u1)
    grad_b = d3.grad(b) + rvec*lift(tau_b1)
    problem = d3.IVP([p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2], namespace=locals())
    problem.add_equation("trace(grad_u) + tau_p = 0")
    if forced:
        problem.add_equation("dt(b) - kappa*div(grad_b) + lift(tau_b2) = - u@grad(b) + 0.05*sin(3*b)")
    else:
        problem.add_equation("dt(b) - kappa*div(grad_b) + lift(tau_b2) = - u@grad(b)")
    problem.add_equation("dt(u) - nu*div(grad_u) + grad(p) - b*er + lift(tau_u2) = - u@grad(u)")
    problem.add_equation("b(r=Ri) = 1"); problem.add_equation("u(r=Ri) = 0")
    problem.add_equation("b(r=Ro) = 0"); problem.add_equation("u(r=Ro) = 0")
    problem.add_equation("integ(p) = 0")
    solver = problem.build_solver(d3.SBDF2)
    b['c'] = g['b_c']; u['c'] = g['u_c'] * 100
    out = dict(b0=b['c'].copy(), u0=u['c'].copy(), meta=np.array(list(shape) + [steps, tstep]))
    for i in range(steps):
        solver.step(tstep)
    for f in (p, b, u):
        out[f.name + "1"] = f['c'].copy()
    return out


def shell_convection_big(shape=(64, 32, 24), steps=2, tstep=0.02):
    """A larger shell (Lmax = 30, 24 radial modes: dense systems of 128 unknowns, up to 62 columns each) with an O(0.05) flow."""
    Ri, Ro = 14, 15
    Nphi, Ntheta, Nr = shape
    Rayleigh = 3500; Prandtl = 1; dealias = 3/2
    coords = d3.SphericalCoordinates('phi', 'theta', 'r')
    dist = d3.Distributor(coords, dtype=np.float64)
    shell = d3.ShellBasis(coords, shape=(Nphi, Ntheta, Nr), radii=(Ri, Ro), dealias=dealias, dtype=np.float64)
    sphere = shell.outer_surface
    p = dist.Field(name='p', bases=shell); b = dist.Field(name='b', bases=shell)
    u = dist.VectorField(coords, name='u', bases=shell)
    tau_p = dist.Field(name='tau_p')
    tau_b1 = dist.Field(name='tau_b1', bases=sphere); tau_b2 = dist.Field(name='tau_b2', bases=sphere)
    tau_u1 = dist.VectorField(coords, name='tau_u1', bases=sphere); tau_u2 = dist.VectorField(coords, name='tau_u2', bases=sphere)
    kappa = (Rayleigh * Prandtl)**(-1/2); nu = (Rayleigh / Prandtl)**(-1/2)
    phi, theta, r = dist.local_grids(shell)
    er = dist.VectorField(coords, bases=shell.radial_basis); er['g'][2] = 1
    rvec = dist.VectorField(coords, bases=shell.radial_basis); rvec['g'][2] = r
    lift_basis = shell.derivative_basis(1)
    lift = lambda A: d3.Lift(A, lift_basis, -1)
    grad_u = d3.grad(u) + rvec*lift(tau_u1)
    grad_b = d3.grad(b) + rvec*lift(tau_b1)
    problem = d3.IVP([p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2], namespace=locals())
    problem.add_equation("trace(grad_u) + tau_p = 0")
    problem.add_equation("dt(b) - kappa*div(grad_b) + lift(tau_b2) = - u@grad(b)")
    problem.add_equation("dt(u) - nu*div(grad_u) + grad(p) - b*er + lift(tau_u2) = - u@grad(u)")
    problem.add_equation("b(r=Ri) = 1"); problem.add_equation("u(r=Ri) = 0")
    problem.add_equation("b(r=Ro) = 0"); problem.add_equation("u(r=Ro) = 0")
    problem.add_equation("integ(p) = 0")
    solver = problem.build_solver(d3.SBDF2)
    b.fill_random('g', seed=42, distribution='normal', scale=1e-3)
    b['g'] *= (r - Ri) * (Ro - r)
    b['g'] += (Ri - Ri*Ro/r) / (Ri - Ro)
    u.fill_random('g', seed=7, distribution='normal', scale=0.5)
    u.low_pass_filter(scales=0.5)
    u['g'] *= (r - Ri) * (Ro - r)
    out = dict(b0=b['c'].copy(), u0=u['c'].copy(), meta=np.array(list(shape) + [steps, tstep]))
    for i in range(steps):
        solver.step(tstep)
    for f in (p, b, u):
        out[f.name + "1"] = f['c'].copy()
    return out


def gen_shell_strong():
    out = {f"strong_{k}": v for k, v in shell_convection_strong().items()}
    out.update({f"forced_{k}": v for k, v in shell_convection_strong(forced=True).items() if k.endswith("1")})
    out.update({f"big_{k}": v for k, v in shell_convection_big().items() if k not in ("b0", "u0")})    # initial state: rebuilt by the test
    np.savez_compressed(HERE / "shell_strong.npz", **out)
    print({k: (v.shape, float(np.abs(v).max())) for k, v in out.items()})


if __name__ == "__main__" and "shell_strong" in sys.argv[1:]:
    gen_shell_strong()


def gen_shell_ivp():
    """Shell convection: three per-l pencil matrices (natural ordering) and states after K steps, 16 x 8 x 6 (SBDF2, RK222) and
    32 x 16 x 12 (SBDF2)."""
    out = {}
    for tag, kw in dict(a_sbdf2=dict(shape=(16, 8, 6), steps=3, dump=(0, 1, 3)), a_rk222=dict(shape=(16, 8, 6), steps=3, scheme="RK222"),
                        b_sbdf2=dict(shape=(32, 16, 12), steps=3)).items():
        for k, v in shell_convection(**kw).items():
            out[f"{tag}_{k}"] = v
    np.savez_compressed(HERE / "shell_ivp.npz", **out)
    print({k: v.shape for k, v in out.items() if k.endswith("b1") or "_l" in k})


if __name__ == "__main__" and "shell_ivp" in sys.argv[1:]:
    gen_shell_ivp()


# ----------------------------------------------------------------------------------------------------------
# Advective CFL frequency on the sphere and in the shell (core/basis.py:6156-6212)
# ----------------------------------------------------------------------------------------------------------
def gen_cfl_curvilinear():
    """Grid maximum of the reference's AdvectiveCFL operator for random velocities (the quantity extras/flow_tools.CFL reduces)."""
    out = {}
    c = d3.S2Coordinates('phi', 'theta'); d = d3.Distributor(c, dtype=np.float64)
    b = d3.SphereBasis(c, (32, 16), radius=2.5, dealias=1.5, dtype=np.float64)
    u = d.VectorField(c, bases=b); u.fill_random(layout='g', seed=3)
    uc = u['c'].copy()
    f = d3.AdvectiveCFL(u, c).evaluate(); f.change_scales(1.5)
    out['sphere_u_c'] = uc; out['sphere_fmax'] = np.max(f['g'])
    c3 = d3.SphericalCoordinates('phi', 'theta', 'r'); d = d3.Distributor(c3, dtype=np.float64)
    b = d3.ShellBasis(c3, (32, 16, 12), radii=(14, 15), dealias=1.5, dtype=np.float64)
    u = d.VectorField(c3, bases=b); u.fill_random(layout='g', seed=4)
    uc = u['c'].copy()
    f = d3.AdvectiveCFL(u, c3).evaluate(); f.change_scales(1.5)
    out['shell_u_c'] = uc; out['shell_fmax'] = np.max(f['g'])
    np.savez_compressed(HERE / "cfl_curvilinear.npz", **out)
    print({k: (v.shape if getattr(v, 'shape', ()) else float(v)) for k, v in out.items()})


if __name__ == "__main__" and "cfl_curvilinear" in sys.argv[1:]:
    gen_cfl_curvilinear()


# ----------------------------------------------------------------------------------------------------------
# Stand-alone expression evaluation (analysis tasks / flow properties of the stock Rayleigh-Benard script)
# ----------------------------------------------------------------------------------------------------------
def gen_expressions():
    """Output-task expressions of examples/ivp_2d_rayleigh_benard/rayleigh_benard.py:93-103 (vorticity, Reynolds number) and a
    few more grid-function expressions, evaluated by the reference on seeded random fields (RealFourier x ChebyshevT, dealias 3/2):
    coefficient data and grid data at scale 1, as the reference's handlers deliver them."""
    out = {}
    Nx, Nz = 32, 16
    coords = d3.CartesianCoordinates('x', 'z')
    dist = d3.Distributor(coords, dtype=np.float64)
    xb = d3.RealFourier(coords['x'], size=Nx, bounds=(0, 4), dealias=3/2)
    zb = d3.ChebyshevT(coords['z'], size=Nz, bounds=(0, 1), dealias=3/2)
    u = dist.VectorField(coords, name='u', bases=(xb, zb))
    b = dist.Field(name='b', bases=(xb, zb))
    u.fill_random('g', seed=11, distribution='normal', scale=1.0); u.low_pass_filter(scales=0.75)
    b.fill_random('g', seed=12, distribution='normal', scale=1.0); b.low_pass_filter(scales=0.75)
    out['u_c'] = u['c'].copy(); out['b_c'] = b['c'].copy(); out['meta'] = np.array([Nx, Nz])
    out['norms'] = np.array([b.allreduce_L2_norm(), b.allreduce_L2_norm(normalize_volume=False), u.allreduce_L2_norm(),
                             b.allreduce_data_norm('c', 2), b.allreduce_data_max('g')])
    hp = b.copy(); hp.high_pass_filter(shape=(16, 8)); out['b_highpass_c'] = hp['c'].copy()
    nu = 0.37
    tasks = dict(vorticity=-d3.div(d3.skew(u)), Re=np.sqrt(u@u)/nu, ke=0.5*(u@u), sinb_b=np.sin(b)*b + b,
                 grad_mag=np.sqrt(d3.grad(b)@d3.grad(b)), absdiv=np.abs(d3.div(u)) * 2.0)
    for name, op in tasks.items():
        f = op.evaluate()
        f.change_scales(1)
        out[f"{name}_g"] = f['g'].copy()
        out[f"{name}_c"] = f['c'].copy()
    # reductions: integrals, averages, interpolation (profiles, mid-plane values, volume integrals)
    x, z = coords['x'], coords['z']
    reductions = dict(int_bb=d3.Integrate(d3.Integrate(b*b, x), z), prof_b=d3.Average(b, x), mid_uu=(u@u)(z=0.3),
                      avg_speed=2.0*d3.Average(np.sqrt(u@u), x), point=b(x=1.3)(z=0.6), vol_avg=d3.Average(d3.Average(b, z), x),
                      int_dzb=d3.Integrate(d3.Differentiate(b, z), z))
    for name, op in reductions.items():
        f = op.evaluate()
        f.change_scales(1)
        out[f"red_{name}_g"] = f['g'].copy()
    np.savez_compressed(HERE / "expressions.npz", **out)
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__" and "expressions" in sys.argv[1:]:
    gen_expressions()


# ----------------------------------------------------------------------------------------------------------
# Stock example scripts, executed by the reference with reduced sizes (the test executes the same source with the import changed)
# ----------------------------------------------------------------------------------------------------------
STOCK = {
    "rb2d": ("examples/ivp_2d_rayleigh_benard/rayleigh_benard.py",
             [("Nx, Nz = 256, 64", "Nx, Nz = 32, 16"), ("stop_sim_time = 50", "stop_sim_time = 2")], ("b", "u", "p")),
    "shell": ("examples/ivp_shell_convection/shell_convection.py",
              [("Nphi, Ntheta, Nr = 192, 96, 6", "Nphi, Ntheta, Nr = 16, 8, 6"), ("stop_sim_time = 2000", "stop_sim_time = 11")],
              ("p", "b", "u")),
    "shear": ("examples/ivp_2d_shear_flow/shear_flow.py",
              [("Nx, Nz = 128, 256", "Nx, Nz = 16, 32"), ("stop_sim_time = 20", "stop_sim_time = 0.12")], ("u", "s", "p")),
    "poisson": ("examples/lbvp_2d_poisson/poisson.py",
                [("Nx, Ny = 256, 128", "Nx, Ny = 32, 16"), ("f.low_pass_filter(shape=(64, 32))", "f.low_pass_filter(shape=(16, 8))")],
                ("u", "tau_1", "tau_2")),
    "kdv": ("examples/ivp_1d_kdv_burgers/kdv_burgers.py",
            [("Nx = 1024", "Nx = 64"), ("stop_sim_time = 10", "stop_sim_time = 0.05")], ("u",)),
}


def run_stock(tag):
    """Execute a stock script of the reference with the substitutions above; output handlers need h5py, which the shim does not
    have, so the lines creating file handlers are dropped for the reference run only."""
    import re
    rel, subs, names = STOCK[tag]
    src = (pathlib.Path("/root/reference") / rel).read_text()
    for old, new in subs:
        assert src.count(old) == 1, old
        src = src.replace(old, new)
    src = "\n".join(l for l in src.splitlines() if not re.match(r"\s*snapshots(\.| =)", l))
    src = src.replace("import matplotlib.pyplot as plt", "plt = None").split("# Plot")[0]
    ns = {"__name__": "__main__"}
    exec(compile(src, rel, "exec"), ns)
    out = {f"{tag}_{n}": ns[n]['c'].copy() for n in names}
    out[f"{tag}_iteration"] = np.array(ns['solver'].iteration)
    out[f"{tag}_sim_time"] = np.array(getattr(ns['solver'], 'sim_time', 0.0))
    for extra in ("max_Re", "max_w", "timestep"):
        if extra in ns:
            out[f"{tag}_{extra}"] = np.array(float(ns[extra]))
    return out


def gen_stock():
    out = {}
    for tag in STOCK:
        out.update(run_stock(tag))
    np.savez_compressed(HERE / "stock_scripts.npz", **out)
    print({k: (v.shape, float(np.abs(v).max())) for k, v in out.items()})


if __name__ == "__main__" and "stock" in sys.argv[1:]:
    gen_stock()


def gen_shell_tasks():
    """Output tasks and the flow property of examples/ivp_shell_convection/shell_convection.py:82-109 -- radial interpolation of a
    field and of a flux built from a radial unit vector, a gradient and a product; azimuthal interpolation; np.sqrt(u@u)/nu --
    evaluated by the reference on a state a few steps into the run (16 x 8 x 6, dealias 3/2), at the scales the script asks for."""
    res = shell_convection((16, 8, 6), 4)
    Ri, Ro = 14, 15
    Rayleigh = 3500; Prandtl = 1; dealias = 3/2
    coords = d3.SphericalCoordinates('phi', 'theta', 'r')
    dist = d3.Distributor(coords, dtype=np.float64)
    shell = d3.ShellBasis(coords, shape=(16, 8, 6), radii=(Ri, Ro), dealias=dealias, dtype=np.float64)
    b = dist.Field(name='b', bases=shell); u = dist.VectorField(coords, name='u', bases=shell)
    b['c'] = res['b1']; u['c'] = res['u1'] * 1e3          # amplified: the velocity is still tiny after four steps
    kappa = (Rayleigh * Prandtl)**(-1/2); nu = (Rayleigh / Prandtl)**(-1/2)
    er = dist.VectorField(coords, bases=shell.radial_basis); er['g'][2] = 1
    flux = er @ (-kappa*d3.grad(b) + u*b)
    out = dict(b_c=b['c'].copy(), u_c=u['c'].copy())
    tasks = dict(bmid=(b(r=(Ri+Ro)/2), dealias), flux_r_outer=(flux(r=Ro), dealias), flux_r_inner=(flux(r=Ri), dealias),
                 flux_phi_start=(flux(phi=0), dealias), flux_phi_end=(flux(phi=3*np.pi/2), dealias), Re=(np.sqrt(u@u)/nu, 1),
                 flux=(flux, 1))
    # evaluated the way the script's file handler evaluates them: scheduled, not forced -- the evaluator walks all tasks from
    # coefficient space to the grid and back, so sums that contain a product are formed on the grid (a forced .evaluate() adds in
    # the layout of the first operand instead, core/arithmetic.py:240-244)
    problem = d3.IVP([b, u], namespace=locals())
    problem.add_equation("dt(b) = 0"); problem.add_equation("dt(u) = 0")
    solver = problem.build_solver(d3.SBDF1)
    handler = solver.evaluator.add_dictionary_handler(iter=1)
    for name, (op, scales) in tasks.items():
        handler.add_task(op, layout='g', name=name, scales=scales)
    solver.evaluator.evaluate_handlers([handler], iteration=0, wall_time=0, sim_time=0, timestep=1)
    for name in tasks:
        out[f"{name}_g"] = handler.fields[name]['g'].copy()
    np.savez_compressed(HERE / "shell_tasks.npz", **out)
    print({k: (v.shape, float(np.abs(v).max())) for k, v in out.items()})


if __name__ == "__main__" and "shell_tasks" in sys.argv[1:]:
    gen_shell_tasks()


# ----------------------------------------------------------------------------------------------------------
# Boundary conditions with data: lower-dimensional equations whose right-hand side is a field
# ----------------------------------------------------------------------------------------------------------
sys.path.insert(0, str(HERE.parent))
from bc_cases import rb2d_bc_data, rb2d_background, rb2d_ncc, rb2d_conservative, rb2d_strong, rb3d_strong, shallow_water_forced


def gen_bc_data():
    res = rb2d_bc_data(d3)
    out = {k: v['c'].copy() for k, v in res.items()}
    out.update({"bg_" + k: v['c'].copy() for k, v in rb2d_background(d3).items()})
    out.update({"ncc_" + k: v['c'].copy() for k, v in rb2d_ncc(d3).items()})
    out.update({"cons_" + k: v['c'].copy() for k, v in rb2d_conservative(d3).items()})
    strong, init = rb2d_strong(d3)
    out.update({"strong_" + k: v['c'].copy() for k, v in strong.items()})
    out.update({"strong_" + k: v for k, v in init.items()})
    out.update({"swf_" + k: v['c'].copy() for k, v in shallow_water_forced(d3)[0].items()})
    strong, init = rb3d_strong(d3)
    out.update({"strong3d_" + k: v['c'].copy() for k, v in strong.items()})
    out.update({"strong3d_" + k: v for k, v in init.items()})
    np.savez_compressed(HERE / "bc_data.npz", **out)
    print({k: (v.shape, float(np.abs(v).max())) for k, v in out.items()})


if __name__ == "__main__" and "bc_data" in sys.argv[1:]:
    gen_bc_data()
