"""Chebyshev-grid transforms of every basis order and fused derivative against an independent high-precision reference.

Shared body of tests/test_emu_cheb_sweep.py (CPU emulation of the kernels) and tests/test_gpu_u1_cheb_sweep.py (B200).

The reference evaluates the unit-normalised Jacobi polynomials p_n^(a,a), a = alpha - 1/2, in mpmath at 30 digits by their
three-term recurrence, with p_n = P_n / sqrt(h_n) and h_n = int (1-z)^a (1+z)^a P_n^2 dz (DLMF 18.3), on the Chebyshev grid
z_j = -cos(pi (2j+1) / 2N).  Derivatives use d/dz P_n^(a,b) = (n+a+b+1)/2 P_{n-1}^(a+1,b+1) (DLMF 18.9.15), divided by the
interval stretch per order.  With more coefficients than grid points (M > N) all M coefficients are differentiated and the
result, in the derivative basis, keeps its modes below N: the derivative followed by that basis's backward transform.  The
forward reference is Gauss-Chebyshev quadrature of the Chebyshev-T coefficients below min(M, N), converted to p^(a,a) by the
inner products <p_m^(a,a), p_n^(-1/2,-1/2)>, themselves computed by an exact Gauss-Chebyshev rule.  Nothing here imports the
product's Jacobi algebra or oracle/; check_reference_pins_fixtures ties the conventions to the reference's own outputs.

Errors are measured per line, relative to sum_n |c_n| max_j |B_jn| (backward) or sum_j |g_j| max_m |F_mj| (forward), where B
and F are the reference matrices: the size of the largest term the line can contain, so the bound does not depend on how
smooth the random data happen to be.
"""
import contextlib
import functools
import os
import subprocess
import sys

import mpmath as mp
import numpy as np

DPS = 30
# Tolerances on the per-line error ratio, calibrated through the emulation.  Backward: worst observed 8.2e-10 (alpha = 4,
# deriv = 4, M = 64, N = 96).  It is float64 rounding amplified by the back-substitution of the conversion, as in the
# reference's own banded solve (scipy's solve_banded gives the same size); it grows with M and with alpha + deriv (1e-13 for
# M <= 26, 8e-12 at M = 32, ~1e-5 at M = 256, alpha + deriv = 8), so the large GPU lengths run alpha + deriv <= 4.
# Forward: worst observed 1.1e-14.  Fields and evaluated expressions: worst observed 2.0e-14.
TOL = 5e-9
TOL_FORWARD = 1e-13
TOL_FIELD = 2e-13
REG_LENGTHS = (24, 48, 96, 192, 384, 768)          # grid sizes with a register-resident Chebyshev kernel (csrc/rfft_regs.cu)
PAIRS = [(alpha, d) for alpha in range(7) for d in range(5) if alpha + d <= 8]        # 2 (alpha + d) + 1 <= 17 diagonals
PAIRS_LOW = [(alpha, d) for alpha, d in PAIRS if alpha + d <= 4]                     # up to 9 diagonals


def stretch_of(alpha, d):
    """Both interval stretches run at every derivative order: 1 when alpha + d is even, 0.5 when it is odd."""
    return 0.5 if (alpha + d) % 2 else 1.0


# ------------------------------------------------------------------------------------------------------------------
# reference
# ------------------------------------------------------------------------------------------------------------------
def _jacobi_table(nmax, c, zs):
    """P_n^(c,c)(z) for n < nmax, z in zs (mpf), by the three-term recurrence (DLMF 18.9.1-2)."""
    rows = []
    if nmax > 0:
        rows.append([mp.mpf(1)] * len(zs))
    if nmax > 1:
        rows.append([(c + 1) * z for z in zs])
    for n in range(2, nmax):
        s = 2 * n + 2 * c
        A = (s - 1) * s * (s - 2)
        Bc = 2 * (n + c - 1) ** 2 * s
        den = 2 * n * (n + 2 * c) * (s - 2)
        p1, p2 = rows[-1], rows[-2]
        rows.append([(A * z * u - Bc * v) / den for z, u, v in zip(zs, p1, p2)])
    return rows


def _norm(n, c):
    """h_n^(c,c) = int_{-1}^{1} (1 - z^2)^c P_n^(c,c)(z)^2 dz."""
    if n == 0:
        return mp.power(2, 2 * c + 1) * mp.gamma(c + 1) ** 2 / mp.gamma(2 * c + 2)
    return mp.power(2, 2 * c + 1) * mp.gamma(n + c + 1) ** 2 / ((2 * n + 2 * c + 1) * mp.gamma(n + 2 * c + 1) * mp.factorial(n))


def _grid(N):
    return [-mp.cos(mp.pi * (2 * j + 1) / (2 * N)) for j in range(N)]


@functools.lru_cache(maxsize=None)
def backward_matrix(N, M, alpha, k):
    """(N, M): grid values of d^k/dz^k p_n^(a,a) at stretch 1, a = alpha - 1/2, with the derivative-basis truncation of M > N."""
    with mp.workdps(DPS):
        c = mp.mpf(alpha) - mp.mpf(1) / 2
        z = _grid(N)
        K = min(M, N)
        P = _jacobi_table(M - k, c + k, z)
        B = np.zeros((N, M))
        for n in range(k, M):
            if n - k >= K:
                continue
            fac = mp.rf(n + 2 * c + 1, k) / mp.power(2, k) / mp.sqrt(_norm(n, c))
            B[:, n] = [float(fac * v) for v in P[n - k]]
    B.setflags(write=False)
    return B


def backward_ref(N, M, alpha, k, stretch):
    return backward_matrix(N, M, alpha, k) / stretch ** k


@functools.lru_cache(maxsize=None)
def forward_matrix(N, M, alpha):
    """(M, N): p^(a,a) coefficients from grid values; Chebyshev-T modes below min(M, N), then converted."""
    with mp.workdps(DPS):
        K = min(M, N)
        half = mp.mpf(1) / 2
        z = _grid(N)
        T = [[mp.pi / N * v / mp.sqrt(_norm(n, -half)) for v in row] for n, row in enumerate(_jacobi_table(K, -half, z))]
        F = np.zeros((M, N))
        if alpha == 0:
            for n in range(K):
                F[n] = [float(v) for v in T[n]]
        else:
            c = mp.mpf(alpha) - half
            Q = M + K + alpha + 2              # integrand degree < 2Q: the Gauss-Chebyshev rule is exact
            x = [mp.cos(mp.pi * (2 * i + 1) / (2 * Q)) for i in range(Q)]
            pa = [[v / mp.sqrt(_norm(m, c)) for v in row] for m, row in enumerate(_jacobi_table(M, c, x))]
            pt = [[v / mp.sqrt(_norm(n, -half)) for v in row] for n, row in enumerate(_jacobi_table(K, -half, x))]
            env = [(1 - xi * xi) ** alpha * mp.pi / Q for xi in x]
            for m in range(M):
                acc = [mp.mpf(0)] * N
                for n in range(m, min(K, m + 2 * alpha + 1)):       # p_n^T has p_m^(a,a) components for n - 2 alpha <= m <= n
                    g = mp.fsum(e * u * v for e, u, v in zip(env, pa[m], pt[n]))
                    acc = [s + g * t for s, t in zip(acc, T[n])]
                F[m] = [float(v) for v in acc]
    F.setflags(write=False)
    return F


def line_errors(out, ref, data, mat, axis=1):
    """Per-line max |out - ref| over the size of the largest term: data (lines, n_in), mat (n_out, n_in)."""
    scale = np.abs(data) @ np.abs(mat).max(axis=0)
    return np.abs(out - ref).max(axis=axis) / scale


def check_reference_pins_fixtures(g):
    """The reference reproduces the reference implementation's own Chebyshev transforms (tests/golden/transforms.npz, ch_*):
    backward and forward, alpha = 0, 1, 2, M below, at and above N; and the recurrence agrees with mpmath.jacobi."""
    with mp.workdps(DPS):
        for c in (mp.mpf(-1) / 2, mp.mpf(13) / 2):
            z = [mp.mpf('-0.83'), mp.mpf('0.31')]
            for n, row in enumerate(_jacobi_table(12, c, z)):
                for zz, v in zip(z, row):
                    assert abs(v - mp.jacobi(n, c, c, zz)) <= mp.mpf(10) ** (-25) * max(1, abs(v)), (c, n)
    keys = sorted({k.rsplit('_', 1)[0] for k in g.files if k.startswith('ch_')})
    assert len(keys) == 36
    for key in keys:
        M, N, alpha = (int(v) for v in key.split('_')[-3:])
        cin, gout, gin, cout = (g[f"{key}_{s}"] for s in ("cin", "gout", "gin", "cout"))
        ref = np.einsum('jn,abn->abj', backward_matrix(N, M, alpha, 0), cin)
        assert np.abs(ref - gout).max() <= 1e-12 * max(1.0, np.abs(gout).max()), (key, "backward", np.abs(ref - gout).max())
        ref = np.einsum('mj,abj->abm', forward_matrix(N, M, alpha), gin)
        assert np.abs(ref - cout).max() <= 1e-12 * max(1.0, np.abs(cout).max()), (key, "forward", np.abs(ref - cout).max())


# ------------------------------------------------------------------------------------------------------------------
# the product's transform plans, with the entry points they reach recorded
# ------------------------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def recorded_entries():
    """Names of the C-ABI entries the library runs inside the block (db_band_lines with its diagonal stride), and the
    register-kernel launch count, read from the same library object the transforms call."""
    from dedalus_b200.lib import get_lib
    lib = get_lib()
    names = []
    call, call_optional = lib.call, lib.call_optional

    def tag(name, args):
        return f"{name}/{args[8]}" if name == "db_band_lines" else name

    def rec_call(name, *args):
        names.append(tag(name, args))
        return call(name, *args)

    def rec_optional(name, *args):
        ok = call_optional(name, *args)
        if ok:
            names.append(tag(name, args))
        return ok

    lib.call, lib.call_optional = rec_call, rec_optional
    rec = dict(names=names, regs0=lib.rfft_regs_launches())
    try:
        yield rec
    finally:
        del lib.call, lib.call_optional
        rec['regs'] = lib.rfft_regs_launches() - rec['regs0']


def _plan(N, M, alpha, stretch):
    from dedalus_b200.transforms import FastChebyshevTransform
    a = alpha - 0.5
    return FastChebyshevTransform(N, M, a, a, -0.5, -0.5, stretch=stretch)


LINES = 7
BACKWARD_PATHS = ("strided", "lines", "offset", "complex")


def _expected_backward(path, M, N, alpha, d):
    """(entry names, register launches) FastChebyshevTransform.backward takes for this case."""
    reg = N in REG_LENGTHS and M % 2 == 0 and M <= N
    if path in ("strided", "complex"):              # complex data: view_as_real puts the real / imaginary pairs innermost
        return ["db_cheb_backward"], 0
    if alpha + d == 0:                              # nothing banded: the plain transform
        return ["db_cheb_backward"], int(reg and path == "lines")
    if M > N:                                       # in-kernel derivative, truncation and back-substitution
        return ["db_cheb_backward"], 0
    compact = alpha + d == 1 and M % 2 == 0 and path == "lines"     # parity-structured, 16-byte aligned lines
    return [f"db_band_lines/{2 if compact else 1}", "db_cheb_backward"], int(reg)


def _layout(path, M, rng, torch, dev):
    """Random coefficients (lines, M) and the tensor handed to the transform, whose transformed axis is `axis`."""
    if path == "strided":
        c = rng.standard_normal((2, M, 5))
        return np.moveaxis(c, 1, -1).reshape(-1, M), torch.from_numpy(c).to(dev), 1
    if path == "complex":
        c = rng.standard_normal((LINES, M)) + 1j * rng.standard_normal((LINES, M))
        return np.concatenate([c.real, c.imag]), torch.from_numpy(c).to(dev), 1
    c = rng.standard_normal((LINES, M))
    if path == "offset":                            # a view one double past an aligned allocation
        base = torch.zeros(LINES * M + 1, dtype=torch.float64, device=dev)
        t = base[1:].view(LINES, M)
        t.copy_(torch.from_numpy(c))
        assert t.data_ptr() % 16 == 8
        return c, t, 1
    return c, torch.from_numpy(c).to(dev), 1


def _lines_of(path, out, N):
    o = out.cpu()
    if path == "strided":
        return np.moveaxis(o.numpy(), 1, -1).reshape(-1, N)
    if path == "complex":
        o = o.numpy()
        return np.concatenate([o.real, o.imag])
    return o.numpy()


def sweep_backward(path, M, N, pairs=PAIRS, tol=TOL):
    """FastChebyshevTransform.backward(deriv=d) from p^(alpha - 1/2) coefficients at every (alpha, d) in `pairs`, on one
    dispatch path, against the reference.  Returns the worst per-line error ratio; fails listing every failing cell."""
    import torch
    from dedalus_b200.lib import compute_device
    dev = compute_device()
    bad, worst = [], 0.0
    for alpha, d in pairs:
        stretch = stretch_of(alpha, d)
        rng = np.random.default_rng(1000 * M + 10 * N + 7 * alpha + d)
        lines, c, axis = _layout(path, M, rng, torch, dev)
        shp = list(c.shape); shp[axis] = N
        out = torch.full(shp, float('nan'), dtype=c.dtype, device=dev)
        plan = _plan(N, M, alpha, stretch)
        with recorded_entries() as rec:
            plan.backward(c, out, axis, deriv=d)
        names, regs = _expected_backward(path, M, N, alpha, d)
        assert (rec['names'], rec['regs']) == (names, regs), (path, M, N, alpha, d, rec['names'], rec['regs'], names, regs)
        B = backward_ref(N, M, alpha, d, stretch)
        err = line_errors(_lines_of(path, out, N), lines @ B.T, lines, B).max()
        worst = max(worst, float(np.nan_to_num(err, nan=np.inf)))
        if not err <= tol:
            bad.append((alpha, d, float(err)))
    assert not bad, f"{path} M={M} N={N}: (alpha, deriv, error / tolerance {tol}) {bad}"
    return worst


def sweep_forward(path, M, N, alphas=range(7), tol=TOL_FORWARD):
    """FastChebyshevTransform.forward into p^(alpha - 1/2) coefficients, alpha = 0..6: conversions of up to 13 diagonals,
    on the generic kernel (strided axis, or a length without register kernel) or the register-resident one."""
    import torch
    from dedalus_b200.lib import compute_device
    dev = compute_device()
    bad, worst = [], 0.0
    reg = path == "lines" and N in REG_LENGTHS and M % 2 == 0 and M <= N
    for alpha in alphas:
        rng = np.random.default_rng(2000 * M + 10 * N + alpha)
        if path == "strided":
            g = rng.standard_normal((2, N, 5))
            gl = np.moveaxis(g, 1, -1).reshape(-1, N)
        else:
            g = rng.standard_normal((LINES, N))
            gl = g
        gt = torch.from_numpy(g).to(dev)
        shp = list(g.shape); shp[1] = M
        out = torch.full(shp, float('nan'), dtype=torch.float64, device=dev)
        with recorded_entries() as rec:
            _plan(N, M, alpha, 1.0).forward(gt, out, 1)
        assert (rec['names'], rec['regs']) == (["db_cheb_forward"], int(reg)), (path, M, N, alpha, rec)
        o = out.cpu().numpy()
        ol = np.moveaxis(o, 1, -1).reshape(-1, M) if path == "strided" else o
        F = forward_matrix(N, M, alpha)
        err = line_errors(ol, gl @ F.T, gl, F).max()
        worst = max(worst, float(np.nan_to_num(err, nan=np.inf)))
        if not err <= tol:
            bad.append((alpha, float(err)))
    assert not bad, f"forward {path} M={M} N={N}: (alpha, error / tolerance {tol}) {bad}"
    return worst


# ------------------------------------------------------------------------------------------------------------------
# DB_CHEB_FUSED_SCAN=1 (read when dedalus_b200.transforms is imported): derivative + back-conversion + transform in one
# kernel where the register kernels cover the length, the stride-2 scan kernel + transform elsewhere.  Runs in a child process.
# ------------------------------------------------------------------------------------------------------------------
FUSED_CASES = [(32, 48), (64, 96), (22, 33)]


def _fused_scan_child():
    if os.environ.get("DB_SWEEP_EMULATED") == "1":
        from emu import emu_lib as E
        E.install()
    import torch
    from dedalus_b200 import transforms
    from dedalus_b200.lib import compute_device
    assert transforms._FUSED_SCAN
    dev = compute_device()
    worst = 0.0
    for M, N in FUSED_CASES:
        for alpha, d in ((1, 0), (0, 1)):
            stretch = 0.5
            rng = np.random.default_rng(M + N + alpha)
            c = rng.standard_normal((LINES, M))
            out = torch.full((LINES, N), float('nan'), dtype=torch.float64, device=dev)
            with recorded_entries() as rec:
                _plan(N, M, alpha, stretch).backward(torch.from_numpy(c).to(dev), out, 1, deriv=d)
            want = (["db_cheb_backward_scan"], 1) if N in REG_LENGTHS else (["db_band_lines/2", "db_cheb_backward"], 0)
            assert (rec['names'], rec['regs']) == want, (M, N, alpha, d, rec)
            B = backward_ref(N, M, alpha, d, stretch)
            err = line_errors(out.cpu().numpy(), c @ B.T, c, B).max()
            assert err <= TOL, (M, N, alpha, d, err)
            worst = max(worst, float(err))
    print(f"fused-scan worst {worst:.3g}")


def check_fused_scan():
    """The opt-in fused scan path, in a child process with DB_CHEB_FUSED_SCAN=1 and the same backend as this process."""
    from dedalus_b200 import lib as dlib
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, DB_CHEB_FUSED_SCAN="1",
               DB_SWEEP_EMULATED="0" if isinstance(dlib._BACKEND, dlib.CudaBackend) else "1",
               PYTHONPATH=os.pathsep.join([here, os.path.dirname(here)] + [p for p in [os.environ.get("PYTHONPATH")] if p]))
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", "import cheb_sweep_cases as S; S._fused_scan_child()"], env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


# ------------------------------------------------------------------------------------------------------------------
# user level: fields on derivative bases, and evaluated expressions whose derivatives the evaluator folds into transforms
# ------------------------------------------------------------------------------------------------------------------
NX, NZ, LX = 8, 16, 4.0


def _fourier_backward(Ng, q):
    """(Ng, NX) grid values of d^q/dx^q of the real Fourier modes [cos 0x, -sin 0x, cos kx, -sin kx, ...] on [0, LX)."""
    x = np.arange(Ng) * LX / Ng
    B = np.zeros((Ng, NX))
    for k in range(NX // 2):
        w = 2 * np.pi * k / LX
        B[:, 2 * k] = w ** q * np.cos(w * x + q * np.pi / 2)
        if k:
            B[:, 2 * k + 1] = -w ** q * np.sin(w * x + q * np.pi / 2)
    return B


def _fourier_forward(Ng):
    x = np.arange(Ng) * LX / Ng
    F = np.zeros((NX, Ng))
    F[0] = 1.0 / Ng
    for k in range(1, NX // 2):
        w = 2 * np.pi * k / LX
        F[2 * k] = 2.0 / Ng * np.cos(w * x)
        F[2 * k + 1] = -2.0 / Ng * np.sin(w * x)
    return F


def _domain():
    import dedalus_b200 as d3
    coords = d3.CartesianCoordinates('x', 'z')
    dist = d3.Distributor(coords, dtype=np.float64)
    xb = d3.RealFourier(coords['x'], size=NX, bounds=(0, LX), dealias=3/2)
    zb = d3.ChebyshevT(coords['z'], size=NZ, bounds=(0, 1), dealias=3/2)
    return d3, coords, dist, xb, zb


def _random_coeffs(rng):
    c = rng.standard_normal((NX, NZ))
    c[1] = 0.0                                       # -sin 0x
    return c


def _rel(got, ref):
    return np.abs(got - ref).max() / np.abs(ref).max()


def check_fields_on_derivative_bases(tol=TOL_FIELD):
    """A field on ChebyshevT.derivative_basis(k), k = 0..6, set from random coefficients and read in grid space."""
    d3, coords, dist, xb, zb = _domain()
    stretch = 0.5
    worst = 0.0
    for k in range(7):
        rng = np.random.default_rng(40 + k)
        c = _random_coeffs(rng)
        f = dist.Field(name='f', bases=(xb, zb.derivative_basis(k)))
        f['c'] = c
        f.change_scales(1)
        got = np.asarray(f['g'])
        Bz = backward_ref(NZ, NZ, k, 0, stretch)
        ref = _fourier_backward(NX, 0) @ c @ Bz.T
        scale = (np.abs(_fourier_backward(NX, 0)).max(axis=0) @ np.abs(c) @ np.abs(Bz).max(axis=0))
        err = np.abs(got - ref).max() / scale
        assert err <= tol, (k, err)
        worst = max(worst, float(err))
    return worst


def check_fused_derivative_expressions(tol=TOL_FIELD):
    """lap(lap(b)) (fourth z-derivative and mixed x / z derivatives) in grid space, and b * dz(dz(dz(dz(b)))) in coefficient
    space (grid product on the 3/2 grids, projected back), evaluated by the product from random coefficients."""
    d3, coords, dist, xb, zb = _domain()
    stretch = 0.5
    rng = np.random.default_rng(77)
    c = _random_coeffs(rng)
    b = dist.Field(name='b', bases=(xb, zb))
    b['c'] = c
    dz = lambda A: d3.Differentiate(A, coords['z'])
    worst = 0.0
    # lap(lap(b)) = b_xxxx + 2 b_xxzz + b_zzzz, exact on the scale-1 grid
    f = d3.lap(d3.lap(b)).evaluate()
    f.change_scales(1)
    got = np.asarray(f['g'])
    terms = [(4, 0, 1.0), (2, 2, 2.0), (0, 4, 1.0)]
    ref = sum(w * _fourier_backward(NX, qx) @ c @ backward_ref(NZ, NZ, 0, qz, stretch).T for qx, qz, w in terms)
    err = _rel(got, ref)
    assert err <= tol, ("lap(lap(b))", err)
    worst = max(worst, err)
    # b * dz^4 b: the grid product on the dealiased grids, projected on the result's basis
    f = (b * dz(dz(dz(dz(b))))).evaluate()
    alpha = int(round(f.bases[1].a + 0.5))
    Ngx, Ngz = xb.grid_size(3/2), zb.grid_size(3/2)
    Bx = _fourier_backward(Ngx, 0)
    g0 = Bx @ c @ backward_ref(Ngz, NZ, 0, 0, stretch).T
    g4 = Bx @ c @ backward_ref(Ngz, NZ, 0, 4, stretch).T
    ref = _fourier_forward(Ngx) @ (g0 * g4) @ forward_matrix(Ngz, NZ, alpha).T
    got = np.asarray(f['c'])
    err = _rel(got, ref)
    assert err <= tol, ("b*dz^4(b)", err)
    worst = max(worst, err)
    return worst
