"""Timed CPU arm: the UNMODIFIED reference (Dedalus v3.0.5 under oracle/_ref, built by oracle/build_ref.py) stepping the
benchmark problem through its own public API -- d3.IVP / problem.build_solver(d3.RK222) / solver.step(dt), the stock code
path of core/solvers.py:683-711 and core/timesteppers.py:552-644 -- on the GPU box's host cores.
TEST / BENCH INFRASTRUCTURE (bench.py `--impl reference` and `cpu_baseline` only).

Bounded sample.  The full 256^3 problem needs ~1 h of per-pencil matrix assembly and ~100 s per step on one core (SURVEY.md
section 8d), and the reference has no threading: its parallelism is MPI ranks, each owning a block of (kx, ky) pencils
(core/distributor.py:357-385).  mpi4py / MPI are not installed, so C ranks are emulated by C CONCURRENT single-rank
instances, each stepping a Fourier x Fourier x Chebyshev problem of shape (nx_s, ny_s, Nz): the FULL pencil height Nz (the
same 5 Nz + 8 unknowns per parity component as at 256^3) and 1/f of the (N/2)^2 pencils, f = N^2 / (nx_s ny_s).  One timed
"step" is one solver.step of every instance (started together behind a barrier, the slowest instance counts); the full-size
estimate is   t_full = t_sample * f / C   (C f-th parts run at once).  What the sample leaves out favours the reference:
no inter-rank transposes (MPI Alltoallv absent), and the x / y FFT lines are nx_s, ny_s instead of N points long (smaller
log factor).  Memory-bandwidth contention between the C instances is inside the measurement.
"""
import json, os, sys, time, pathlib

ROOT = pathlib.Path(__file__).resolve().parents[1]
REF = ROOT / "oracle" / "_ref"


def available():
    return (REF / ".built").exists()


_BARRIER = None          # multiprocessing.Barrier, inherited by the forked instances


def _instance(args):
    shape, tstep, warmup, steps, seed = args        # (not `dt`: the equations' namespace is locals())
    barrier = _BARRIER
    os.environ["OMP_NUM_THREADS"] = "1"            # the reference mandates it (dedalus/__init__.py:17-19)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    sys.path.insert(0, str(REF))
    import logging
    logging.disable(logging.INFO)
    import numpy as np
    import dedalus.public as d3
    from dedalus.core import basis
    basis.FourierBase.default_library = "scipy"      # the reference's own scipy transform classes (FFTW is not installed)
    basis.Jacobi.default_dct = "scipy_dct"
    Nx, Ny, Nz = shape
    Lx = Ly = 4.0; Lz = 1.0; Rayleigh = 1e6; Prandtl = 1.0
    t0 = time.perf_counter()
    # SURVEY.md Appendix C (examples/ivp_2d_rayleigh_benard/rayleigh_benard.py:33-89 with a y axis)
    coords = d3.CartesianCoordinates('x', 'y', 'z')
    dist = d3.Distributor(coords, dtype=np.float64)
    xb = d3.RealFourier(coords['x'], size=Nx, bounds=(0, Lx), dealias=3/2)
    yb = d3.RealFourier(coords['y'], size=Ny, bounds=(0, Ly), dealias=3/2)
    zb = d3.ChebyshevT(coords['z'], size=Nz, bounds=(0, Lz), dealias=3/2)
    p = dist.Field(name='p', bases=(xb, yb, zb)); b = dist.Field(name='b', bases=(xb, yb, zb))
    u = dist.VectorField(coords, name='u', bases=(xb, yb, zb))
    tau_p = dist.Field(name='tau_p')
    tau_b1 = dist.Field(name='tau_b1', bases=(xb, yb)); tau_b2 = dist.Field(name='tau_b2', bases=(xb, yb))
    tau_u1 = dist.VectorField(coords, name='tau_u1', bases=(xb, yb)); tau_u2 = dist.VectorField(coords, name='tau_u2', bases=(xb, yb))
    kappa = (Rayleigh * Prandtl)**(-1/2); nu = (Rayleigh / Prandtl)**(-1/2)
    x, y, z = dist.local_grids(xb, yb, zb)
    ex, ey, ez = coords.unit_vector_fields(dist)
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
    solver = problem.build_solver(d3.RK222)
    b.fill_random('g', seed=seed, distribution='normal', scale=1e-3)
    b['g'] *= z * (Lz - z); b['g'] += Lz - z
    setup = time.perf_counter() - t0
    barrier.wait()
    for _ in range(warmup):                          # first step factorises every pencil (timesteppers.py:632-639): untimed
        solver.step(tstep)
    times = []
    for _ in range(steps):
        barrier.wait()
        t1 = time.perf_counter()
        solver.step(tstep)
        times.append(time.perf_counter() - t1)
    chk = float(np.sum(b['c']**2))
    return dict(setup=setup, times=times, pencils=len(solver.subproblems), n=int(max(sp.LHS.shape[0] for sp in solver.subproblems)) if hasattr(solver.subproblems[0], 'LHS') else None,
                check=chk)


def sample_shape(N, instances, max_pencils=256):
    """(nx_s, ny_s) of one instance: 32 x 32 (256 pencils) unless that would make instances * fraction exceed the whole
    (or max_pencils asks for a cheaper set-up: the per-pencil matrix assembly dominates the arm's wall time)."""
    nx = ny = min(32, N)
    while (instances * nx * ny > N * N or (nx // 2) * (ny // 2) > max_pencils) and ny > 4:
        if nx >= ny and nx > 4: nx //= 2
        else: ny //= 2
    return nx, ny


def run(N=256, dt=0.0025, warmup=1, steps=5, instances=None, max_pencils=256):
    """Returns dict(steps_per_sec (median, scaled to N^3), list, spread, cores, sample, ...)."""
    import multiprocessing as mp
    import numpy as np
    if not available():
        raise RuntimeError("oracle/_ref is missing: run `python -m oracle.build_ref` where the reference checkout exists")
    cores = os.cpu_count() or 1
    C = instances or cores
    nx, ny = sample_shape(N, C, max_pencils)
    f = (N * N) / (nx * ny)
    C = int(min(C, f))
    ctx = mp.get_context("fork")
    global _BARRIER
    _BARRIER = ctx.Barrier(C)
    t0 = time.time()
    with ctx.Pool(C) as pool:
        res = pool.map(_instance, [((nx, ny, N), dt, warmup, steps, 42 + i) for i in range(C)], chunksize=1)
    wall = time.time() - t0
    t_sample = np.max(np.array([r['times'] for r in res]), axis=0)         # slowest instance, per step
    t_full = t_sample * f / C
    sps = 1.0 / t_full
    med = float(np.median(sps))
    return dict(steps_per_sec=med, steps_per_sec_list=[float(v) for v in sps], spread=float((sps.max() - sps.min()) / med),
                cores=C, host_cores=cores, sample_shape=[nx, ny, N], fraction_per_instance=1.0 / f, instances=C,
                sample_step_seconds=float(np.median(t_sample)), setup_seconds=float(max(r['setup'] for r in res)), wall_seconds=wall,
                pencils_per_instance=res[0]['pencils'],
                sample=(f"UNMODIFIED reference (Dedalus v3.0.5, scipy transforms, SuperLU), {C} concurrent single-rank instances "
                        f"(1 thread each; {cores} host cores) of RB3D {nx}x{ny}x{N}: full pencil height, {res[0]['pencils']} of "
                        f"{(N // 2)**2} pencils each (1/{f:g} of the {N}^3 step); {steps} timed solver.step calls after {warmup} warm-up, "
                        f"slowest instance per step, scaled by {f:g}/{C}; no inter-rank transposes (MPI absent): upper bound for "
                        f"an MPI run on {C} cores"))


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=256); ap.add_argument("--dt", type=float, default=None)
    ap.add_argument("--steps", type=int, default=5); ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--instances", type=int, default=None)
    a = ap.parse_args()
    print(json.dumps(run(a.size, a.dt or 1e-2 * 64.0 / a.size, a.warmup, a.steps, a.instances)))
