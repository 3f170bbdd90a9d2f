"""The reference's stock example scripts restated at reduced sizes: 2-D Rayleigh-Benard, shell convection, 2-D shear flow and
KdV-Burgers, each set up and stepped through the public API as the script does it, main loop included: the CFL time step,
the flow property logged every 10 iterations and a snapshot file handler.  Shared by the emulated tests
(tests/test_emu_stock_scripts.py) and the GPU tests (tests/test_gpu_t8_expressions.py).  Expected values:
tests/golden/stock_scripts.npz (make_golden.py run_stock, the unmodified reference executing its own scripts at these
sizes).  The Poisson LBVP and the shallow-water script are restated in bc_cases.py and sphere_cases.py."""
import numpy as np
import dedalus_b200 as d3


def _rayleigh_benard_2d():
    """examples/ivp_2d_rayleigh_benard/rayleigh_benard.py at 32 x 16 up to t = 2."""
    Lx, Lz = 4, 1
    kappa = nu = 2e6 ** (-1/2)                                       # Rayleigh 2e6, Prandtl 1
    coords = d3.CartesianCoordinates('x', 'z')
    dist = d3.Distributor(coords, dtype=np.float64)
    xbasis = d3.RealFourier(coords['x'], size=32, bounds=(0, Lx), dealias=3/2)
    zbasis = d3.ChebyshevT(coords['z'], size=16, bounds=(0, Lz), dealias=3/2)
    p = dist.Field(name='p', bases=(xbasis, zbasis))
    b = dist.Field(name='b', bases=(xbasis, zbasis))
    u = dist.VectorField(coords, name='u', bases=(xbasis, zbasis))
    tau_p = dist.Field(name='tau_p')
    tau_b1, tau_b2 = (dist.Field(name=n, bases=xbasis) for n in ('tau_b1', 'tau_b2'))
    tau_u1, tau_u2 = (dist.VectorField(coords, name=n, bases=xbasis) for n in ('tau_u1', 'tau_u2'))
    x, z = dist.local_grids(xbasis, zbasis)
    ex, ez = coords.unit_vector_fields(dist)
    lift_basis = zbasis.derivative_basis(1)
    lift = lambda A: d3.Lift(A, lift_basis, -1)
    ns = dict(p=p, b=b, u=u, tau_p=tau_p, tau_b2=tau_b2, tau_u2=tau_u2, kappa=kappa, nu=nu, ez=ez, Lz=Lz, lift=lift,
              grad_u=d3.grad(u) + ez*lift(tau_u1), grad_b=d3.grad(b) + ez*lift(tau_b1))
    problem = d3.IVP([p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2], namespace=ns)
    problem.add_equation("trace(grad_u) + tau_p = 0")
    problem.add_equation("dt(b) - kappa*div(grad_b) + lift(tau_b2) = - u@grad(b)")
    problem.add_equation("dt(u) - nu*div(grad_u) + grad(p) - b*ez + lift(tau_u2) = - u@grad(u)")
    problem.add_equation("b(z=0) = Lz")
    problem.add_equation("u(z=0) = 0")
    problem.add_equation("b(z=Lz) = 0")
    problem.add_equation("u(z=Lz) = 0")
    problem.add_equation("integ(p) = 0")
    solver = problem.build_solver(d3.RK222)
    solver.stop_sim_time = 2
    b.fill_random('g', seed=42, distribution='normal', scale=1e-3)
    b['g'] *= z * (Lz - z)
    b['g'] += Lz - z
    tasks = dict(buoyancy=b, vorticity=-d3.div(d3.skew(u)))
    return solver, dict(p=p, b=b, u=u), tasks, dict(sim_dt=0.25, max_writes=50), \
        dict(initial_dt=0.125, cadence=10, safety=0.5, threshold=0.05, max_change=1.5, min_change=0.5, max_dt=0.125), \
        ('max_Re', np.sqrt(u@u)/nu)


def _shell_convection():
    """examples/ivp_shell_convection/shell_convection.py at 16 x 8 x 6 up to t = 11."""
    Ri, Ro = 14, 15
    kappa = nu = 3500 ** (-1/2)                                      # Rayleigh 3500, Prandtl 1
    coords = d3.SphericalCoordinates('phi', 'theta', 'r')
    dist = d3.Distributor(coords, dtype=np.float64)
    shell = d3.ShellBasis(coords, shape=(16, 8, 6), radii=(Ri, Ro), dealias=3/2, dtype=np.float64)
    sphere = shell.outer_surface
    p = dist.Field(name='p', bases=shell)
    b = dist.Field(name='b', bases=shell)
    u = dist.VectorField(coords, name='u', bases=shell)
    tau_p = dist.Field(name='tau_p')
    tau_b1, tau_b2 = (dist.Field(name=n, bases=sphere) for n in ('tau_b1', 'tau_b2'))
    tau_u1, tau_u2 = (dist.VectorField(coords, name=n, bases=sphere) for n in ('tau_u1', 'tau_u2'))
    phi, theta, r = dist.local_grids(shell)
    er = dist.VectorField(coords, bases=shell.radial_basis)
    er['g'][2] = 1
    rvec = dist.VectorField(coords, bases=shell.radial_basis)
    rvec['g'][2] = r
    lift_basis = shell.derivative_basis(1)
    lift = lambda A: d3.Lift(A, lift_basis, -1)
    ns = dict(p=p, b=b, u=u, tau_p=tau_p, tau_b2=tau_b2, tau_u2=tau_u2, kappa=kappa, nu=nu, er=er, Ri=Ri, Ro=Ro, lift=lift,
              grad_u=d3.grad(u) + rvec*lift(tau_u1), grad_b=d3.grad(b) + rvec*lift(tau_b1))
    problem = d3.IVP([p, b, u, tau_p, tau_b1, tau_b2, tau_u1, tau_u2], namespace=ns)
    problem.add_equation("trace(grad_u) + tau_p = 0")
    problem.add_equation("dt(b) - kappa*div(grad_b) + lift(tau_b2) = - u@grad(b)")
    problem.add_equation("dt(u) - nu*div(grad_u) + grad(p) - b*er + lift(tau_u2) = - u@grad(u)")
    problem.add_equation("b(r=Ri) = 1")
    problem.add_equation("u(r=Ri) = 0")
    problem.add_equation("b(r=Ro) = 0")
    problem.add_equation("u(r=Ro) = 0")
    problem.add_equation("integ(p) = 0")
    solver = problem.build_solver(d3.SBDF2)
    solver.stop_sim_time = 11
    b.fill_random('g', seed=42, distribution='normal', scale=1e-3)
    b['g'] *= (r - Ri) * (Ro - r)
    b['g'] += (Ri - Ri*Ro/r) / (Ri - Ro)
    flux = er @ (-kappa*d3.grad(b) + u*b)
    tasks = dict(bmid=b(r=(Ri+Ro)/2), flux_r_outer=flux(r=Ro), flux_r_inner=flux(r=Ri), flux_phi_start=flux(phi=0),
                 flux_phi_end=flux(phi=3*np.pi/2))
    return solver, dict(p=p, b=b, u=u), tasks, dict(sim_dt=10, max_writes=10, scales=3/2), \
        dict(initial_dt=1, cadence=10, safety=2, threshold=0.1, max_change=1.5, min_change=0.5, max_dt=1), \
        ('max_Re', np.sqrt(u@u)/nu)


def _shear_flow():
    """examples/ivp_2d_shear_flow/shear_flow.py at 16 x 32 up to t = 0.12: doubly periodic, a passive tracer, pressure gauge
    through tau_p and integ(p)."""
    Lx, Lz = 1, 2
    nu = D = 1 / 5e4                                                 # Reynolds 5e4, Schmidt 1
    coords = d3.CartesianCoordinates('x', 'z')
    dist = d3.Distributor(coords, dtype=np.float64)
    xbasis = d3.RealFourier(coords['x'], size=16, bounds=(0, Lx), dealias=3/2)
    zbasis = d3.RealFourier(coords['z'], size=32, bounds=(-Lz/2, Lz/2), dealias=3/2)
    p = dist.Field(name='p', bases=(xbasis, zbasis))
    s = dist.Field(name='s', bases=(xbasis, zbasis))
    u = dist.VectorField(coords, name='u', bases=(xbasis, zbasis))
    tau_p = dist.Field(name='tau_p')
    x, z = dist.local_grids(xbasis, zbasis)
    ex, ez = coords.unit_vector_fields(dist)
    problem = d3.IVP([u, s, p, tau_p], namespace=dict(u=u, s=s, p=p, tau_p=tau_p, nu=nu, D=D))
    problem.add_equation("dt(u) + grad(p) - nu*lap(u) = - u@grad(u)")
    problem.add_equation("dt(s) - D*lap(s) = - u@grad(s)")
    problem.add_equation("div(u) + tau_p = 0")
    problem.add_equation("integ(p) = 0")
    solver = problem.build_solver(d3.RK222)
    solver.stop_sim_time = 0.12
    u['g'][0] = 1/2 + 1/2 * (np.tanh((z-0.5)/0.1) - np.tanh((z+0.5)/0.1))
    s['g'] = u['g'][0]
    for z0 in (0.5, -0.5):
        u['g'][1] += 0.1 * np.sin(2*np.pi*x/Lx) * np.exp(-(z-z0)**2/0.01)
    tasks = dict(tracer=s, pressure=p, vorticity=-d3.div(d3.skew(u)))
    return solver, dict(u=u, s=s, p=p), tasks, dict(sim_dt=0.1, max_writes=10), \
        dict(initial_dt=1e-2, cadence=10, safety=0.2, threshold=0.1, max_change=1.5, min_change=0.5, max_dt=1e-2), \
        ('max_w', (u@ez)**2)                                           # the script logs sqrt(max w^2)


def _run_cfl_loop(solver, u, tasks, handler, cfl_args, prop, outdir):
    """The scripts' main loop: CFL time step, and the flow property taken every 10 iterations (after iteration 1, 11, ...)."""
    snapshots = solver.evaluator.add_file_handler(str(outdir / 'snapshots'), **{k: v for k, v in handler.items() if k != 'scales'})
    for name, task in tasks.items():
        snapshots.add_task(task, name=name, **({'scales': handler['scales']} if 'scales' in handler else {}))
    cfl = d3.CFL(solver, **cfl_args)
    cfl.add_velocity(u)
    prop_name, prop_expr = prop
    flow = d3.GlobalFlowProperty(solver, cadence=10)
    flow.add_property(prop_expr, name=prop_name)
    logged = dict()
    while solver.proceed:
        timestep = cfl.compute_timestep()
        solver.step(timestep)
        if (solver.iteration - 1) % 10 == 0:
            logged[prop_name] = flow.max(prop_name)
    logged['timestep'] = timestep
    return logged


def _compare(g, tag, solver, fields, logged, outdir=None):
    assert solver.iteration == int(g[f"{tag}_iteration"])
    assert np.isclose(solver.sim_time, float(g[f"{tag}_sim_time"]), rtol=1e-13)
    for n, f in fields.items():
        ref = g[f"{tag}_{n}"]
        atol = 1e-11 * np.abs(ref).max() if tag != "shell" else 1e-10 * np.abs(g[f"{tag}_b"]).max()    # shell: u ~ 1e-6 b
        got = f['c']
        assert np.allclose(got, ref, rtol=1e-8, atol=atol), (tag, n, np.abs(got - ref).max(), np.abs(ref).max())
    for name, value in logged.items():
        assert np.isclose(float(value), float(g[f"{tag}_{name}"]), rtol=1e-9), (tag, name)
    if outdir is not None:
        assert list((outdir / "snapshots").iterdir())


CASES = dict(rb2d=_rayleigh_benard_2d, shell=_shell_convection, shear=_shear_flow)


def check_stock_ivp(g, tag, outdir):
    """Set up the restated script `tag`, run its main loop to its stop time, compare with the reference's end state, the
    last CFL time step and the last logged flow property."""
    solver, fields, tasks, handler, cfl_args, prop = CASES[tag]()
    logged = _run_cfl_loop(solver, fields['u'], tasks, handler, cfl_args, prop, outdir)
    if prop[0] == 'max_w':
        logged['max_w'] = np.sqrt(logged['max_w'])
    _compare(g, tag, solver, fields, logged, outdir)


def check_kdv_burgers(g):
    """examples/ivp_1d_kdv_burgers/kdv_burgers.py at Nx = 64 up to t = 0.05 (fixed step, SBDF2), including its sampling of the
    grid data at scale 1 every 25 iterations."""
    Lx, a, b, n = 10, 1e-4, 2e-4, 20
    xcoord = d3.Coordinate('x')
    dist = d3.Distributor(xcoord, dtype=np.float64)
    xbasis = d3.RealFourier(xcoord, size=64, bounds=(0, Lx), dealias=3/2)
    u = dist.Field(name='u', bases=xbasis)
    dx = lambda A: d3.Differentiate(A, xcoord)
    problem = d3.IVP([u], namespace=dict(u=u, a=a, b=b, dx=dx))
    problem.add_equation("dt(u) - a*dx(dx(u)) - b*dx(dx(dx(u))) = - u*dx(u)")
    x = dist.local_grid(xbasis)
    u['g'] = np.log(1 + np.cosh(n)**2/np.cosh(n*(x-0.2*Lx))**2) / (2*n)
    solver = problem.build_solver(d3.SBDF2)
    solver.stop_sim_time = 0.05
    timestep = 2e-3
    samples = [u['g', 1].copy()]
    while solver.proceed:
        solver.step(timestep)
        if solver.iteration % 25 == 0:
            samples.append(u['g', 1].copy())
    _compare(g, "kdv", solver, dict(u=u), dict(timestep=timestep))
