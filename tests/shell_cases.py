"""Shared body of the spherical-shell transform tests (emulation: tests/test_emu_shell.py, GPU: tests/test_gpu_t6_shell.py)."""
import numpy as np
import dedalus_b200 as d3
import pytest


def check_shell_field_transforms(g, tag):
    """Scalar / vector / rank-2 fields on a ShellBasis: grid -> coefficients (regularity components, reference packing) -> grid,
    vs the reference chain (core/basis.py:4474-4508: radial factor, regularity recombination Q(l), radial Jacobi transform; plus
    the sphere chain of core/basis.py:3062-3138 with three spin components)."""
    *shape, dealias, k = g[f"{tag}_meta"]
    shape = tuple(int(v) for v in shape)
    coords = d3.SphericalCoordinates('phi', 'theta', 'r')
    dist = d3.Distributor(coords, dtype=np.float64)
    shell = d3.ShellBasis(coords, shape=shape, radii=(1.2, 2.7), dealias=float(dealias), dtype=np.float64, k=int(k))
    grids = dist.local_grids(shell, scales=(dealias,) * 3)
    for got, name in zip(grids, ("phi", "theta", "r")):
        assert np.allclose(got.ravel(), g[f"{tag}_{name}"], rtol=0, atol=1e-14), name
    rng = np.random.default_rng(11)          # the grid data the reference transformed (make_golden.py gen_shell)
    for name, f in (("s", dist.Field(bases=shell)), ("v", dist.VectorField(coords, bases=shell)),
                    ("t", dist.TensorField((coords, coords), bases=shell))):
        f.preset_scales(dealias)
        f['g'] = rng.standard_normal(f['g'].shape)
        c = f['c'].copy()
        assert c.shape == g[f"{tag}_{name}_c"].shape
        assert np.allclose(c, g[f"{tag}_{name}_c"], rtol=1e-12, atol=1e-13), (tag, name, "forward", np.abs(c - g[f"{tag}_{name}_c"]).max())
        assert np.allclose(f['g'], g[f"{tag}_{name}_g2"], rtol=1e-12, atol=1e-12), (tag, name, "backward")


def check_intertwiner_orthogonal():
    """Q(l) is orthogonal on the allowed components and zero on the forbidden ones (l < rank)."""
    from dedalus_b200.shell import Intertwiner
    for rank in (1, 2):
        for ell in range(0, 12):
            Q = Intertwiner(ell).matrix(rank)
            G = Q.T @ Q
            d = np.diag(G)
            assert np.allclose(G, np.diag(d), atol=1e-13)
            assert np.all((np.abs(d - 1) < 1e-13) | (np.abs(d) < 1e-13))
            if ell >= rank:
                assert np.allclose(d, 1)


def _shell_problem(g, tag):
    from dedalus_b200 import examples
    Nphi, Ntheta, Nr, steps, dt = g[f"{tag}_meta"]
    sc = examples.shell_convection(int(Nphi), int(Ntheta), int(Nr))
    return sc, int(steps), float(dt)


def check_shell_pencil_matrices(g, tag="a_sbdf2"):
    """M and L of the shell-convection pencils of degree l = 0, 1, 3 against the reference's subproblem matrices in natural
    ordering (variable, component, (cos | -sin), radial mode; core/subsystems.py:497-602): every operator of the problem --
    gradient, divergence, trace, radial-NCC products, lift, interpolation, integration, conversions."""
    from dedalus_b200 import shell_ivp
    sc, steps, dt = _shell_problem(g, tag)
    problem = sc['problem']
    low = shell_ivp.ShellLowering(problem)
    for ell in (0, 1, 3):
        M, L, rows, cols = shell_ivp.assemble(low, ell)

        def ref_index(layout, kinds):
            idx, off = [], 0
            for c, kd in zip(layout, kinds):
                if kd == 'const' and ell > 0:            # constants only exist in the l = 0 subproblem
                    idx += [-1]
                    continue
                idx += list(range(off, off + c['n']))    # the cos part; the -sin part follows it in the reference ordering
                off += c['n'] * (1 if kd == 'const' else 2)
            return np.array(idx)
        ci = ref_index(cols, [low.kind_of(low.variables[c['item']])[0] for c in cols])
        ri = ref_index(rows, [low.kind_of(problem.equations[r['item']]['LHS'])[0] for r in rows])
        vr = np.array([r['valid'] for r in rows for _ in range(r['n'])])
        vc = np.array([c['valid'] for c in cols for _ in range(c['n'])])
        for name, mine in (("M", M), ("L", L)):
            R = g[f"{tag}_l{ell}_{name}"]
            Rp = np.zeros((R.shape[0] + 1, R.shape[1] + 1)); Rp[:-1, :-1] = R
            ref = Rp[np.ix_(ri, ci)]
            got = mine * np.outer(vr, vc)
            assert np.allclose(got, ref, rtol=1e-11, atol=1e-12 * np.abs(ref).max()), (ell, name, np.abs(got - ref).max())


def check_shell_convection(g, tag, scheme):
    """K steps of shell convection vs the reference.  b, p, u: rtol 1e-8 with atol 1e-10 max|field| + 1e-13 max|b| (after a
    few steps from noise the velocity is 1e-6 of the buoyancy it is coupled to in the same pencil systems, so its error floor is
    rounding relative to b); the tau fields (the unknowns most sensitive to the conditioning of the tau systems, which the
    reference solves with another pivot order): atol 1e-4 max|tau|."""
    from dedalus_b200 import examples
    sc, steps, dt = _shell_problem(g, tag)
    solver = sc['problem'].build_solver(getattr(d3, scheme))
    examples.shell_convection_initial_condition(sc['b'], sc['shell'], sc['Ri'], sc['Ro'])
    assert np.allclose(sc['b']['c'], g[f"{tag}_b0"], rtol=1e-11, atol=1e-13)
    for _ in range(steps):
        solver.step(dt)
    floor = 1e-13 * np.abs(g[f"{tag}_b1"]).max()
    for name in ('p', 'b', 'u'):
        ref = g[f"{tag}_{name}1"]
        got = sc[name]['c']
        assert np.allclose(got, ref, rtol=1e-8, atol=1e-10 * np.abs(ref).max() + floor), (name, np.abs(got - ref).max(), np.abs(ref).max())
    for name, f in sc['taus'].items():
        ref = g[f"{tag}_{name}1"]
        got = f['c']
        assert np.allclose(got, ref, rtol=1e-6, atol=1e-4 * max(np.abs(ref).max(), 1e-300) + 1e-20), (name, np.abs(got - ref).max(), np.abs(ref).max())
    return solver


def check_dense_kernels(B):
    """db_dense_combine / factor / solve / matvec (ragged column counts, pivoting forced) against numpy; B: array backend."""
    import ctypes as C
    from dedalus_b200 import lib as dlib
    rng = np.random.default_rng(1)
    n, nsys = 23, 4
    ncols = [1, 5, 40, 33]
    A = rng.standard_normal((nsys, n, n)); Bm = rng.standard_normal((nsys, n, n))
    A[2, 0, 0] = 0
    sysarr = (dlib.DenseSys * nsys)(); off = 0
    for i, nc in enumerate(ncols):
        sysarr[i].ncols = nc; sysarr[i].vec_off = off; off += n * nc
    a0, b0 = 1.0, 0.3
    P = B.ptr
    sysb = B.dev(np.frombuffer(bytes(sysarr), dtype=np.uint8).copy())
    Ad, Bd = B.dev(A), B.dev(Bm)
    lu, ipiv, info = B.dev(np.zeros_like(A)), B.dev(np.zeros((nsys, n), dtype=np.int32)), B.dev(np.full(nsys, -1, dtype=np.int32))
    B.lib.call("db_dense_combine", nsys, n, a0, P(Ad), b0, P(Bd), P(lu), B.stream)
    B.lib.call("db_dense_factor", nsys, n, P(lu), P(ipiv), P(info), B.stream)
    assert not B.host(info).any()
    v1h, v2h = rng.standard_normal(off), rng.standard_normal(off)
    v1, v2, x, ya, yb = B.dev(v1h), B.dev(v2h), B.dev(np.zeros(off)), B.dev(np.zeros(off)), B.dev(np.zeros(off))
    vc = dlib.VecComb(); vc.nvec = 2
    vc.vec[0], vc.vec[1] = P(v1).value, P(v2).value
    vc.coef[0], vc.coef[1] = 2.0, -0.5
    B.lib.call("db_dense_solve", P(sysb), nsys, n, max(ncols), P(lu), P(ipiv), C.byref(vc), P(x), B.stream)
    B.lib.call("db_dense_matvec", P(sysb), nsys, n, P(Ad), P(Bd), P(x), P(ya), P(yb), B.stream)
    # the same products with the operators in CSR (one of them made sparse)
    As = A * (rng.random(A.shape) < 0.2)
    def csr(Mx):
        nz = Mx != 0
        counts = nz.sum(axis=2)
        ptr = np.zeros((nsys, n + 1), dtype=np.int64); ptr[:, 1:] = np.cumsum(counts, axis=1)
        ptr += np.concatenate([[0], np.cumsum(counts.sum(axis=1))[:-1]])[:, None]
        s_, r_, c_ = np.nonzero(nz)
        return B.dev(ptr), B.dev(c_.astype(np.int32)), B.dev(Mx[s_, r_, c_])
    (ap, ac, av), (bp, bc, bv) = csr(As), csr(Bm)
    za, zb = B.dev(np.zeros(off)), B.dev(np.zeros(off))
    B.lib.call("db_csr_matvec", P(sysb), nsys, n, P(ap), P(ac), P(av), P(bp), P(bc), P(bv), P(x), P(za), P(zb), B.stream)
    zah, zbh = B.host(za), B.host(zb)
    xh, yah, ybh = B.host(x), B.host(ya), B.host(yb)
    for i, nc in enumerate(ncols):
        o = sysarr[i].vec_off
        assert np.allclose(zah[o:o + n * nc].reshape(n, nc), As[i] @ xh[o:o + n * nc].reshape(n, nc), rtol=1e-12, atol=1e-12)
        assert np.allclose(zbh[o:o + n * nc].reshape(n, nc), Bm[i] @ xh[o:o + n * nc].reshape(n, nc), rtol=1e-12, atol=1e-12)
        b = (2 * v1h[o:o + n * nc] - 0.5 * v2h[o:o + n * nc]).reshape(n, nc)
        xr = np.linalg.solve(a0 * A[i] + b0 * Bm[i], b)
        xg = xh[o:o + n * nc].reshape(n, nc)
        assert np.abs(xg - xr).max() <= 1e-10 * np.abs(xr).max(), (i, np.abs(xg - xr).max())
        assert np.allclose(yah[o:o + n * nc].reshape(n, nc), A[i] @ xg, rtol=1e-12, atol=1e-12)
        assert np.allclose(ybh[o:o + n * nc].reshape(n, nc), Bm[i] @ xg, rtol=1e-12, atol=1e-12)


def check_shell_tasks(g):
    """Output tasks and the flow property of the stock shell-convection script (shell_convection.py:82-109) on a stored state:
    radial interpolations, the flux built from a radial unit vector, a gradient and a product, azimuthal interpolation (a field
    locked to the grid) and np.sqrt(u@u)/nu, against the unmodified reference (tests/golden/shell_tasks.npz)."""
    Ri, Ro = 14, 15
    Rayleigh = 3500; Prandtl = 1; dealias = 3/2
    coords = d3.SphericalCoordinates('phi', 'theta', 'r')
    dist = d3.Distributor(coords, dtype=np.float64)
    shell = d3.ShellBasis(coords, shape=(16, 8, 6), radii=(Ri, Ro), dealias=dealias, dtype=np.float64)
    b = dist.Field(name='b', bases=shell); u = dist.VectorField(coords, name='u', bases=shell)
    b['c'] = g['b_c']; u['c'] = g['u_c']
    kappa = (Rayleigh * Prandtl)**(-1/2); nu = (Rayleigh / Prandtl)**(-1/2)
    er = dist.VectorField(coords, bases=shell.radial_basis); er['g'][2] = 1
    flux = er @ (-kappa*d3.grad(b) + u*b)
    tasks = dict(bmid=(b(r=(Ri+Ro)/2), dealias), flux_r_outer=(flux(r=Ro), dealias), flux_r_inner=(flux(r=Ri), dealias),
                 flux_phi_start=(flux(phi=0), dealias), flux_phi_end=(flux(phi=3*np.pi/2), dealias), Re=(np.sqrt(u@u)/nu, 1),
                 flux=(flux, 1))
    for name, (op, scales) in tasks.items():
        f = op.evaluate()
        f.change_scales(scales)
        got, ref = np.asarray(f['g']), g[f"{name}_g"]
        assert got.shape == ref.shape, (name, got.shape, ref.shape)
        assert np.allclose(got, ref, rtol=1e-9, atol=1e-11 * np.abs(ref).max()), (name, np.abs(got - ref).max(), np.abs(ref).max())
    with pytest.raises(ValueError):
        f = flux(phi=0).evaluate(); f['c']


def check_shell_convection_strong(g):
    """Shell convection with O(0.1) velocities (advection as large as the linear terms): 3 SBDF2 steps against the reference.  The
    noise-started fixtures keep |u| ~ 1e-6 |b| and cannot see the order of truncations in the right-hand side; this one can."""
    from dedalus_b200 import examples
    Nphi, Ntheta, Nr, steps, dt = g["strong_meta"]
    sc = examples.shell_convection(int(Nphi), int(Ntheta), int(Nr))
    solver = sc['problem'].build_solver(d3.SBDF2)
    sc['b']['c'] = g["strong_b0"]; sc['u']['c'] = g["strong_u0"]
    for _ in range(int(steps)):
        solver.step(float(dt))
    for name in ('p', 'b', 'u'):
        ref = g[f"strong_{name}1"]
        got = sc[name]['c']
        assert np.allclose(got, ref, rtol=1e-8, atol=1e-10 * np.abs(ref).max()), (name, np.abs(got - ref).max(), np.abs(ref).max())


def check_shell_convection_forced(g):
    """The same start with a grid function on the right-hand side of the buoyancy equation (0.05 sin(3 b)): outside the fused shell
    plan, carried by the general curvilinear evaluator."""
    from dedalus_b200 import examples
    Nphi, Ntheta, Nr, steps, dt = g["strong_meta"]
    sc = examples.shell_convection(int(Nphi), int(Ntheta), int(Nr), rhs_b_extra="0.05*sin(3*b)")
    solver = sc['problem'].build_solver(d3.SBDF2)
    sc['b']['c'] = g["strong_b0"]; sc['u']['c'] = g["strong_u0"]
    for _ in range(int(steps)):
        solver.step(float(dt))
    assert type(solver.rhs_plan).__name__ == "GenericCurvilinearRHS"
    for name in ('p', 'b', 'u'):
        ref = g[f"forced_{name}1"]
        got = sc[name]['c']
        assert np.allclose(got, ref, rtol=1e-8, atol=1e-10 * np.abs(ref).max()), (name, np.abs(got - ref).max(), np.abs(ref).max())


def check_shell_convection_big(g):
    """64 x 32 x 24 (Lmax = 30, 24 radial modes, up to 62 right-hand-side columns per degree) from an O(0.05) flow: 2 SBDF2 steps."""
    from dedalus_b200 import examples
    Nphi, Ntheta, Nr, steps, dt = g["big_meta"]
    sc = examples.shell_convection(int(Nphi), int(Ntheta), int(Nr))
    solver = sc['problem'].build_solver(d3.SBDF2)
    Ri, Ro, b, u = sc['Ri'], sc['Ro'], sc['b'], sc['u']
    phi, theta, r = sc['dist'].local_grids(sc['shell'])
    b.fill_random('g', seed=42, distribution='normal', scale=1e-3)          # the initial state of make_golden.py shell_convection_big
    b['g'] *= (r - Ri) * (Ro - r)
    b['g'] += (Ri - Ri*Ro/r) / (Ri - Ro)
    u.fill_random('g', seed=7, distribution='normal', scale=0.5)
    u.low_pass_filter(scales=0.5)
    u['g'] *= (r - Ri) * (Ro - r)
    for _ in range(int(steps)):
        solver.step(float(dt))
    for name in ('p', 'b', 'u'):
        ref = g[f"big_{name}1"]
        got = sc[name]['c']
        assert np.allclose(got, ref, rtol=1e-8, atol=1e-10 * np.abs(ref).max()), (name, np.abs(got - ref).max(), np.abs(ref).max())
    return solver
