"""Device transform plans behind the reference's transform-plugin contract.

Reference contract (core/transforms.py:27-75, basis.py:416-428, 924-936): a plan is built as
`cls(grid_size, coeff_size)` (Fourier) or `cls(grid_size, coeff_size, a, b, a0, b0)` (Jacobi) and exposes
`forward(gdata, cdata, axis)` / `backward(cdata, gdata, axis)` on N-D C-contiguous arrays.  Here the arrays are
torch CUDA tensors (float64, or complex128 for ComplexFourier) and the work is one CUDA kernel launch
(csrc/fft.cu) per call; results are written into the output tensor, which must not alias the input.
"""
import ctypes as C
import functools
import os
import numpy as np
from . import jacobi
from .lib import get_lib, FftPlan, DedalusB200Error
from .fftplan import HostPlan
from .basis import RealFourier, ComplexFourier, Jacobi

_transform_registry = {}


def register_transform(basis_cls, name):
    def wrapper(cls):
        _transform_registry.setdefault(basis_cls, {})[name] = cls
        return cls
    return wrapper


def _torch():
    import torch
    return torch


def _stream():
    from .lib import current_stream
    return current_stream()


def _dptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _split(shape, axis):
    outer = int(np.prod(shape[:axis], dtype=np.int64))
    inner = int(np.prod(shape[axis + 1:], dtype=np.int64))
    return outer, inner


class DevicePlan:
    """FFT tables uploaded once; struct kept alive with its tensors."""
    _cache = {}

    def __new__(cls, n, kind, device):
        key = (n, kind, str(device))
        if key not in cls._cache:
            self = object.__new__(cls)
            torch = _torch()
            hp = HostPlan(n, kind)
            self.hp = hp
            self.tensors = [torch.from_numpy(np.ascontiguousarray(x)).to(device) for x in (hp.tw, hp.twr, hp.twq, hp.perm, hp.iperm, hp.twn)]
            s = FftPlan()
            s.n, s.nc, s.half, s.nrad = hp.n, hp.nc, hp.half, len(hp.radices)
            for i, r in enumerate(hp.radices):
                s.rad[i] = r
            s.tw, s.twr, s.twq, s.perm, s.iperm, s.twn = [t.data_ptr() for t in self.tensors]
            self.struct = s
            cls._cache[key] = self
        return cls._cache[key]

    def ref(self):
        return C.byref(self.struct)


def _check(x, name):
    from .lib import device_tensor_ok
    if not device_tensor_ok(x) or not x.is_contiguous():
        raise ValueError(f"{name} must be a contiguous CUDA tensor.")


@register_transform(RealFourier, 'b200')
class RealFourierTransform:
    """cos/-sin real Fourier transform (reference FFTWRealFFT, transforms.py:537-565)."""

    def __init__(self, grid_size, coeff_size, kscale=1.0):
        self.N, self.M = int(grid_size), int(coeff_size)
        self.kscale = kscale

    def forward(self, gdata, cdata, axis):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        if gdata.shape[axis] != self.N or cdata.shape[axis] != self.M:
            raise ValueError("Array shapes do not match the transform plan.")
        plan = DevicePlan(self.N, 'real', gdata.device)
        outer, inner = _split(gdata.shape, axis)
        get_lib().call("db_rfft_forward", plan.ref(), _dptr(gdata), _dptr(cdata), outer, self.M, inner, _stream())

    def backward(self, cdata, gdata, axis, deriv=0):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        if gdata.shape[axis] != self.N or cdata.shape[axis] != self.M:
            raise ValueError("Array shapes do not match the transform plan.")
        plan = DevicePlan(self.N, 'real', gdata.device)
        outer, inner = _split(gdata.shape, axis)
        get_lib().call("db_rfft_backward", plan.ref(), _dptr(cdata), _dptr(gdata), outer, self.M, inner, int(deriv), float(self.kscale), _stream())

    # ---- blocked row addressing: the transform writes / reads the per-peer blocks of an all-to-all buffer directly
    #      (include/dedalus_b200.h db_rfft_*_blocked); pointers are raw device addresses, block = (rows per peer, stride)
    def blocked_supported(self, inner):
        """Mirror of the coverage test in csrc/rfft_regs.cu db_rfft_regs_try."""
        return (self.N in (24, 48, 96, 192, 384, 768) and self.M % 2 == 0 and self.M >= 2 and 3 * self.M <= 2 * self.N
                and inner >= 16 and inner % 16 == 0 and os.environ.get("DB_FFT_REGS", "1") != "0"
                and os.environ.get("DB_BLOCKED_TRANSPOSE", "1") != "0")

    def backward_blocked(self, c_ptr, g_ptr, outer, inner, device, deriv=0, in_block=(0, 0), out_block=(0, 0)):
        plan = DevicePlan(self.N, 'real', device)
        ok = get_lib().call_optional("db_rfft_backward_blocked", plan.ref(), C.c_void_p(c_ptr), C.c_void_p(g_ptr), outer, self.M, inner,
                                     int(deriv), float(self.kscale), int(in_block[0]), int(in_block[1]), int(out_block[0]), int(out_block[1]), _stream())
        if not ok:
            raise RuntimeError("blocked real-Fourier transform not covered (blocked_supported() out of sync with the kernels)")

    # ---- peer variants: output block b goes to out_ptrs[b] (another GPU's receive buffer), see db_rfft_*_peer
    def backward_peer(self, c_ptr, origin_ptr, outer, inner, device, out_rpb, out_ptrs, deriv=0, in_block=(0, 0)):
        plan = DevicePlan(self.N, 'real', device)
        arr = (C.c_void_p * len(out_ptrs))(*[C.c_void_p(int(p)) for p in out_ptrs])
        ok = get_lib().call_optional("db_rfft_backward_peer", plan.ref(), C.c_void_p(c_ptr), C.c_void_p(origin_ptr), outer, self.M, inner,
                                     int(deriv), float(self.kscale), int(in_block[0]), int(in_block[1]), int(out_rpb), len(out_ptrs), arr, _stream())
        if not ok:
            raise RuntimeError("peer real-Fourier transform not covered (blocked_supported() out of sync with the kernels)")

    def forward_peer(self, g_ptr, origin_ptr, outer, inner, device, out_rpb, out_ptrs, in_block=(0, 0)):
        plan = DevicePlan(self.N, 'real', device)
        arr = (C.c_void_p * len(out_ptrs))(*[C.c_void_p(int(p)) for p in out_ptrs])
        ok = get_lib().call_optional("db_rfft_forward_peer", plan.ref(), C.c_void_p(g_ptr), C.c_void_p(origin_ptr), outer, self.M, inner,
                                     int(in_block[0]), int(in_block[1]), int(out_rpb), len(out_ptrs), arr, _stream())
        if not ok:
            raise RuntimeError("peer real-Fourier transform not covered (blocked_supported() out of sync with the kernels)")

    def forward_blocked(self, g_ptr, c_ptr, outer, inner, device, in_block=(0, 0), out_block=(0, 0)):
        plan = DevicePlan(self.N, 'real', device)
        ok = get_lib().call_optional("db_rfft_forward_blocked", plan.ref(), C.c_void_p(g_ptr), C.c_void_p(c_ptr), outer, self.M, inner,
                                     int(in_block[0]), int(in_block[1]), int(out_block[0]), int(out_block[1]), _stream())
        if not ok:
            raise RuntimeError("blocked real-Fourier transform not covered (blocked_supported() out of sync with the kernels)")


@register_transform(ComplexFourier, 'b200')
class ComplexFourierTransform:
    """Complex Fourier transform (reference FFTWComplexFFT, transforms.py:302-330)."""

    def __init__(self, grid_size, coeff_size, kscale=1.0):
        self.N, self.M = int(grid_size), int(coeff_size)
        self.kscale = kscale

    def forward(self, gdata, cdata, axis):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        plan = DevicePlan(self.N, 'complex', gdata.device)
        outer, inner = _split(gdata.shape, axis)
        get_lib().call("db_cfft_forward", plan.ref(), _dptr(gdata), _dptr(cdata), outer, self.M, inner, _stream())

    def backward(self, cdata, gdata, axis, deriv=0):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        plan = DevicePlan(self.N, 'complex', gdata.device)
        outer, inner = _split(gdata.shape, axis)
        get_lib().call("db_cfft_backward", plan.ref(), _dptr(cdata), _dptr(gdata), outer, self.M, inner, int(deriv), float(self.kscale), _stream())


_FUSED_SCAN = os.environ.get("DB_CHEB_FUSED_SCAN", "0") == "1"


def banded_upper_diags(mat, M, ndiag):
    """Diagonals 0..ndiag-1 of a sparse upper-triangular matrix, rows < M, as (ndiag, M) float64."""
    A = mat.tocsr()
    out = np.zeros((ndiag, M))
    nrow, ncol = A.shape
    for d in range(ndiag):
        diag = A.diagonal(d)
        L = min(len(diag), M)
        out[d, :L] = diag[:L]
    return np.ascontiguousarray(out)


@register_transform(Jacobi, 'b200_dct')
class FastChebyshevTransform:
    """Chebyshev-grid ultraspherical transform (reference FFTWFastChebyshevTransform, transforms.py:801-902).

    `backward(..., deriv=d)` additionally applies (d/dz)^d in coefficient space before the transform, i.e. it
    is the backward transform of the derivative basis (a+d, b+d) composed with DifferentiateJacobi
    (basis.py:701-718); `stretch` is the affine map factor of the problem interval."""

    def __init__(self, grid_size, coeff_size, a, b, a0, b0, stretch=1.0):
        if not (a0 == b0 == -0.5):
            raise ValueError("Fast Chebyshev transform requires a0 == b0 == -1/2.")
        self.N, self.M = int(grid_size), int(coeff_size)
        self.a, self.b, self.a0, self.b0 = a, b, a0, b0
        self.stretch = stretch
        self._dev = {}

    def _diags(self, key, device):
        k = (key, str(device))
        if k not in self._dev:
            torch = _torch()
            kind, d = key
            M, N = self.M, self.N
            if kind == 'fwd':
                K = max(M, N)
                Cm = jacobi.conversion_matrix(K, self.a0, self.b0, self.a, self.b)
                nd = int(round((self.a - self.a0) + (self.b - self.b0))) + 1
                arr = banded_upper_diags(Cm, M, nd)
            elif kind == 'solve':
                Cm = jacobi.conversion_matrix(M, self.a0, self.b0, self.a + d, self.b + d)
                nd = int(round((self.a + d - self.a0) + (self.b + d - self.b0))) + 1
                arr = banded_upper_diags(Cm, M, nd)
                arr[0] = 1.0 / arr[0]            # kernel contract: row 0 of the solve matrix holds 1/diagonal
                if nd == 3 and np.abs(arr[1]).max() <= 1e-14 * np.abs(arr).max() and M % 2 == 0:     # odd diagonal = rounding noise
                    # parity-structured conversion: store diagonals 0 and 2 only (stride 2) -> warp-scan kernel
                    self._dev[(('solve2', d), str(device))] = (torch.from_numpy(np.ascontiguousarray(arr[[0, 2]])).to(device), 2)
            else:  # 'pre': derivative chain (a,b) -> (a+d,b+d)
                P = None
                for j in range(d):
                    Dj = jacobi.differentiation_matrix(M, self.a + j, self.b + j) / self.stretch
                    P = Dj if P is None else Dj @ P
                arr = banded_upper_diags(P, M, d + 1)
            self._dev[k] = (torch.from_numpy(arr).to(device), arr.shape[0])
        return self._dev[k]

    def forward(self, gdata, cdata, axis):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        if gdata.shape[axis] != self.N or cdata.shape[axis] != self.M:
            raise ValueError("Array shapes do not match the transform plan.")
        if gdata.is_complex():   # complex data = interleaved real lines (reference fftw_wrappers.pyx:244-246)
            gdata, cdata = _torch().view_as_real(gdata), _torch().view_as_real(cdata)
        plan = DevicePlan(self.N, 'real', gdata.device)
        outer, inner = _split(gdata.shape, axis)
        if (self.a, self.b) != (self.a0, self.b0):
            dg, nd = self._diags(('fwd', 0), gdata.device)
        else:
            dg, nd = None, 0
        get_lib().call("db_cheb_forward", plan.ref(), _dptr(gdata), _dptr(cdata), outer, self.M, inner, _dptr(dg), nd, _stream())

    def backward(self, cdata, gdata, axis, deriv=0):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        if gdata.shape[axis] != self.N or cdata.shape[axis] != self.M:
            raise ValueError("Array shapes do not match the transform plan.")
        if gdata.is_complex():
            gdata, cdata = _torch().view_as_real(gdata), _torch().view_as_real(cdata)
        plan = DevicePlan(self.N, 'real', gdata.device)
        outer, inner = _split(gdata.shape, axis)
        pre, npre = (self._diags(('pre', deriv), gdata.device) if deriv > 0 else (None, 0))
        if (self.a + deriv, self.b + deriv) != (self.a0, self.b0):
            sol, nsol = self._diags(('solve', deriv), gdata.device)
        else:
            sol, nsol = None, 0
        if inner == 1 and (npre or nsol) and self.M <= self.N:
            # contiguous lines: run the serial banded recurrence in its own one-thread-per-line kernel, then the
            # plain transform (keeps the recurrence off the FFT kernel's critical path)
            compact = self._dev.get((('solve2', deriv), str(gdata.device))) if (nsol and npre <= 3) else None
            if _FUSED_SCAN and compact is not None and cdata.data_ptr() % 16 == 0 and gdata.data_ptr() % 16 == 0:
                # derivative + back-conversion + transform in one kernel (the scan runs on the lines staged in shared
                # memory).  Opt-in (DB_CHEB_FUSED_SCAN=1): measured at 256^3 it is not faster than the separate scan
                # kernel -- 16 lines per CTA leave most warps idle during the scan (z backward 3.11 vs 2.98 ms per step)
                if get_lib().call_optional("db_cheb_backward_scan", plan.ref(), _dptr(cdata), _dptr(gdata), outer, self.M,
                                           _dptr(pre), npre, _dptr(compact[0]), _stream()):
                    return
            tmp = self._scratch(cdata)
            if compact is not None and cdata.data_ptr() % 16 == 0:
                get_lib().call("db_band_lines", _dptr(cdata), _dptr(tmp), outer, self.M, _dptr(pre), npre, _dptr(compact[0]), 2, 2, _stream())
            else:
                get_lib().call("db_band_lines", _dptr(cdata), _dptr(tmp), outer, self.M, _dptr(pre), npre, _dptr(sol), nsol, 1, _stream())
            get_lib().call("db_cheb_backward", plan.ref(), _dptr(tmp), _dptr(gdata), outer, self.M, inner, None, 0, None, 0, _stream())
        else:
            get_lib().call("db_cheb_backward", plan.ref(), _dptr(cdata), _dptr(gdata), outer, self.M, inner,
                           _dptr(pre), npre, _dptr(sol), nsol, _stream())

    def _scratch(self, like):
        key = (tuple(like.shape), str(like.device))
        t = self._dev.get(('scratch',) + key)
        if t is None:
            t = _torch().empty_like(like)
            self._dev[('scratch',) + key] = t
        return t


@register_transform(Jacobi, 'b200_matrix')
class JacobiMatrixTransform:
    """Dense Jacobi transform on its own Gauss grid (reference JacobiMMT, transforms.py:114-158), fp64 GEMM kernel."""

    def __init__(self, grid_size, coeff_size, a, b, a0, b0, stretch=1.0):
        self.N, self.M = int(grid_size), int(coeff_size)
        self.a, self.b, self.a0, self.b0 = a, b, a0, b0
        N, M = self.N, self.M
        grid, weights = jacobi.gauss_grid(N, a0, b0)
        base = jacobi.polynomials(max(M, N), a0, b0, grid) * weights
        base[N:, :] = 0
        base = base[:M, :]          # DEALIAS_BEFORE_CONVERTING = True (reference dedalus.cfg:54)
        if (a, b) != (a0, b0):
            fwd = jacobi.conversion_matrix(base.shape[0], a0, b0, a, b) @ base
        else:
            fwd = base
        self.forward_matrix = np.ascontiguousarray(fwd[:M])
        poly = jacobi.polynomials(M, a, b, grid)
        poly[N:, :] = 0
        self.backward_matrix = np.ascontiguousarray(poly.T)
        self.stretch = stretch
        self._grid = grid
        self._dev = {}

    def _derivative_backward(self, d):
        """Grid values of the d-th derivative from (a, b) coefficients: the backward matrix of the basis (a + d, b + d) times the
        differentiation matrices in between (reference DifferentiateJacobi, core/basis.py:701-718, followed by the transform)."""
        a, b = self.a, self.b
        chain = np.eye(self.M)
        for i in range(d):
            chain = (jacobi.differentiation_matrix(self.M, a + i, b + i) / self.stretch) @ chain
        poly = jacobi.polynomials(self.M, a + d, b + d, self._grid)
        poly[self.N:, :] = 0
        return np.ascontiguousarray(poly.T @ chain)

    def _mat(self, which, device):
        k = (which, str(device))
        if k not in self._dev:
            if which == 'f':
                m = self.forward_matrix
            elif which == 'b':
                m = self.backward_matrix
            else:
                m = self._derivative_backward(which)
            self._dev[k] = _torch().from_numpy(m).to(device)
        return self._dev[k]

    def forward(self, gdata, cdata, axis):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        outer, inner = _split(gdata.shape, axis)
        get_lib().call("db_mmt_apply", _dptr(self._mat('f', gdata.device)), self.M, self.N, _dptr(gdata), _dptr(cdata), outer, inner, _stream())

    def backward(self, cdata, gdata, axis, deriv=0):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        outer, inner = _split(gdata.shape, axis)
        mat = self._mat(int(deriv) if deriv else 'b', gdata.device)        # derivatives fold into the matrix
        get_lib().call("db_mmt_apply", _dptr(mat), self.N, self.M, _dptr(cdata), _dptr(gdata), outer, inner, _stream())


class SWSHColatitudeTransform:
    """Spin-weighted spherical harmonic colatitude transform (reference SWSHColatitudeTransform, core/transforms.py:1251-1340).

    Same constructor contract as the reference plugin -- `cls(Ntheta, Lmax, m_maps, s)` with `m_maps` the tuple of
    (m, mg_slice, mc_slice, ell_slice) produced by SphereBasis.m_maps (core/basis.py:2940-2970; rows of 8 integers
    (m, mg0, mg1, mc0, mc1, ell_start, ell_stop or -1, ell_step) are accepted as well) -- and the same
    `forward(gdata, cdata, axis)` / `backward(cdata, gdata, axis)` on arrays whose axis - 1 carries the azimuthal
    coefficients and whose `axis` carries colatitude / degree.  The harmonics are built on the host from the unit-normalised
    Jacobi polynomials (dedalus_b200/jacobi.py):  Y_{l,m,s}(z) = (-1)^max(m,-s) sqrt((1-z)^a (1+z)^b) p_k^(a,b)(z), a = |m+s|,
    b = |m-s|, k = l - max(|m|,|s|) (reference libraries/dedalus_sphere/sphere.py:43-64), on the Ntheta Gauss-Legendre nodes;
    all per-m matrices live in one device buffer and one kernel launch (db_ragged_matvec) serves every local m."""

    def __init__(self, Ntheta, Lmax, m_maps, s):
        self.Ntheta, self.Lmax, self.s = int(Ntheta), int(Lmax), int(s)
        rows = []
        for e in m_maps:
            if len(e) == 4:
                m, mg, mc, ell = e
                rows.append((int(m), int(mg.start), int(mg.stop), int(mc.start), int(mc.stop), int(ell.start),
                             -1 if ell.stop is None else int(ell.stop), -1 if ell.step == -1 else 1))
            else:
                rows.append(tuple(int(v) for v in e))
        self.m_maps = rows
        self._dev = {}

    @staticmethod
    @functools.lru_cache(maxsize=None)
    def quadrature(Ntheta):
        """Gauss-Legendre nodes and weights in long double: scipy's float64 nodes refined by Newton steps on P_Ntheta.  At
        degree ~250 a node rounded to float64 moves the harmonics by ~1e-12, which the forward-backward round trip
        accumulates to ~1e-10; the reference builds its colatitude quadrature in long double for the same reason.
        Cached per Ntheta (matrices() asks for it once per m); callers must not modify the arrays."""
        from scipy.special import roots_jacobi
        z = roots_jacobi(Ntheta, 0.0, 0.0)[0].astype(jacobi.LD)

        def legendre(z):
            p0, p1 = np.ones_like(z), z.copy()
            for n in range(1, Ntheta):
                p0, p1 = p1, ((2 * n + 1) * z * p1 - n * p0) / (n + 1)
            return p1, Ntheta * (z * p1 - p0) / (z * z - 1)        # P_N, P_N'

        for _ in range(2):
            p, dp = legendre(z)
            z = z - p / dp
        _, dp = legendre(z)
        return z, 2 / ((1 - z * z) * dp * dp)

    def matrices(self, m):
        """(forward (Lmax+1-|m|, Ntheta), backward (Ntheta, Lmax+1-|m|)), zero rows for l < |s| and l >= Ntheta."""
        Nt, Lmax, s = self.Ntheta, self.Lmax, self.s
        z, w = self.quadrature(Nt)
        n = Lmax + 1 - max(abs(m), abs(s))
        a, b = abs(m + s), abs(m - s)
        F = np.zeros((Lmax + 1 - abs(m), Nt)); B = np.zeros((Nt, Lmax + 1 - abs(m)))
        if n > 0:
            Y = jacobi.polynomials(n, a, b, z, half_log_weight=True) * ((-1.0) ** max(m, -s))
            Lmin = max(abs(m), abs(s))
            F[Lmin - abs(m):, :] = Y * w[None, :]
            B[:, Lmin - abs(m):] = Y.T
        F[max(Nt - abs(m), 0):, :] = 0
        B[:, max(Nt - abs(m), 0):] = 0
        return F, B

    def _program(self, device, nell):
        """Device buffers: concatenated matrices + the two entry tables (forward / backward)."""
        key = (str(device), nell)
        if key in self._dev:
            return self._dev[key]
        from .lib import RaggedEntry
        torch = _torch()
        mats, off = [], 0
        fwd = (RaggedEntry * len(self.m_maps))(); bwd = (RaggedEntry * len(self.m_maps))()
        cache = {}
        maxf = maxb = 1
        for q, (m, mg0, mg1, mc0, mc1, e0, e1, estep) in enumerate(self.m_maps):
            nm = mg1 - mg0
            ells = np.arange(nell)[slice(e0, None if e1 < 0 else e1, estep)]
            if abs(m) > self.Lmax:
                # nothing to do forward; zeros written backward (they feed the inverse azimuthal transform)
                f, b = fwd[q], bwd[q]
                f.nrow = 0; f.ncol = 0; f.nm = nm; f.zero = 0
                b.mat_off = 0; b.nrow = self.Ntheta; b.ncol = 0; b.in_i0 = mc0; b.in_row0 = 0; b.in_step = 1
                b.out_i0 = mg0; b.out_row0 = 0; b.out_step = 1; b.nm = nm; b.zero = 1
                maxb = max(maxb, self.Ntheta)
                continue
            if m not in cache:
                F, B = self.matrices(m)
                cache[m] = (off, off + F.size)
                mats += [F.ravel(), B.ravel()]
                off += F.size + B.size
            nl = self.Lmax + 1 - abs(m)
            if len(ells) != nl:
                raise ValueError("m_maps degree slice does not have Lmax + 1 - |m| entries")
            f, b = fwd[q], bwd[q]
            f.mat_off = cache[m][0]; f.nrow = nl; f.ncol = self.Ntheta
            f.in_i0 = mg0; f.in_row0 = 0; f.in_step = 1
            f.out_i0 = mc0; f.out_row0 = int(ells[0]); f.out_step = int(estep); f.nm = nm; f.zero = 0
            b.mat_off = cache[m][1]; b.nrow = self.Ntheta; b.ncol = nl
            b.in_i0 = mc0; b.in_row0 = int(ells[0]); b.in_step = int(estep)
            b.out_i0 = mg0; b.out_row0 = 0; b.out_step = 1; b.nm = nm; b.zero = 0
            maxf = max(maxf, nl); maxb = max(maxb, self.Ntheta)
        mats_t = torch.from_numpy(np.concatenate(mats) if mats else np.zeros(1)).to(device)
        tab = lambda arr: torch.from_numpy(np.frombuffer(bytes(arr), dtype=np.uint8).copy()).to(device)
        prog = dict(mats=mats_t, fwd=tab(fwd), bwd=tab(bwd), n=len(self.m_maps), maxf=maxf, maxb=maxb)
        self._dev[key] = prog
        return prog

    def matrix_bytes(self):
        """Bytes of the per-m matrices one application streams (one direction): sum over m of Ntheta * (Lmax + 1 - m) * 8."""
        return 8 * sum(self.Ntheta * (self.Lmax + 1 - abs(r[0])) for r in self.m_maps if abs(r[0]) <= self.Lmax)

    @staticmethod
    def _reduced(t, axis):
        """(N0, N1, N2, N3) view with N1 = axis - 1, N2 = axis (reference reduced_view_4, tools/array.py)."""
        shp = t.shape
        n0 = int(np.prod(shp[:axis - 1], dtype=np.int64)); n3 = int(np.prod(shp[axis + 1:], dtype=np.int64))
        return n0, int(shp[axis - 1]), int(shp[axis]), n3

    def forward(self, gdata, cdata, axis):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        n0, n1g, n2g, n3 = self._reduced(gdata, axis)
        _, n1c, n2c, _ = self._reduced(cdata, axis)
        if n2g != self.Ntheta:
            raise ValueError("Array shapes do not match the transform plan.")
        p = self._program(gdata.device, n2c)
        get_lib().call("db_ragged_matvec", _dptr(p['mats']), _dptr(p['fwd']), p['n'], p['maxf'], _dptr(gdata), _dptr(cdata),
                       n0, n1g, n2g, n1c, n2c, n3, _stream())

    def backward(self, cdata, gdata, axis):
        _check(gdata, "gdata"); _check(cdata, "cdata")
        n0, n1g, n2g, n3 = self._reduced(gdata, axis)
        _, n1c, n2c, _ = self._reduced(cdata, axis)
        if n2g != self.Ntheta:
            raise ValueError("Array shapes do not match the transform plan.")
        p = self._program(gdata.device, n2c)
        get_lib().call("db_ragged_matvec", _dptr(p['mats']), _dptr(p['bwd']), p['n'], p['maxb'], _dptr(cdata), _dptr(gdata),
                       n0, n1c, n2c, n1g, n2g, n3, _stream())


def transform_plan(basis, scale):
    """Plan for one basis at one scale (reference basis.transform_plan, basis.py:506-509, 915-922)."""
    N = basis.grid_size(scale)
    if isinstance(basis, RealFourier):
        return RealFourierTransform(N, basis.size, kscale=1.0 / basis.COV.stretch)
    if isinstance(basis, ComplexFourier):
        return ComplexFourierTransform(N, basis.size, kscale=1.0 / basis.COV.stretch)
    if isinstance(basis, Jacobi):
        if basis.a0 == basis.b0 == -0.5:
            return FastChebyshevTransform(N, basis.size, basis.a, basis.b, basis.a0, basis.b0, stretch=basis.COV.stretch)
        return JacobiMatrixTransform(N, basis.size, basis.a, basis.b, basis.a0, basis.b0, stretch=basis.COV.stretch)
    raise NotImplementedError(f"No transform for basis {basis}")


_plan_cache = {}


def cached_plan(basis, scale):
    key = (basis, scale)
    if key not in _plan_cache:
        _plan_cache[key] = transform_plan(basis, scale)
    return _plan_cache[key]


def transform_field(field, layout):
    """Move a Field between full coefficient ('c') and full grid ('g') layouts on the device.

    Single-GPU chain: axes last -> first towards grid space (reference Distributor._build_layouts,
    distributor.py:131-175, with an empty mesh); the multi-GPU chain with its transpose hop is handled by
    dedalus_b200/transposes.py."""
    torch = _torch()
    from .sphere import sphere_basis_of, transform_sphere_field
    if sphere_basis_of(field) is not None:
        return transform_sphere_field(field, layout)
    from .shell import shell_basis_of, transform_shell_field
    if shell_basis_of(field) is not None:
        return transform_shell_field(field, layout)
    from .shell import ShellRadialBasis, transform_radial_field
    if any(isinstance(b, ShellRadialBasis) for b in field.bases):
        return transform_radial_field(field, layout)
    if field.dist.size > 1:
        from .transposes import transform_field_distributed
        return transform_field_distributed(field, layout)
    data = field.device_data()
    nt = len(field.tensorsig)
    dim = field.dist.dim
    scales = field.scales
    if layout == 'g':
        cur = data
        for ax in range(dim - 1, -1, -1):
            b = field.bases[ax]
            if b is None:
                continue
            plan = cached_plan(b, scales[ax])
            shp = list(cur.shape); shp[nt + ax] = plan.N
            out = torch.empty(shp, dtype=cur.dtype, device=cur.device)
            plan.backward(cur.contiguous(), out, nt + ax)
            cur = out
        field.set_device_data(cur, 'g')
    else:
        cur = data
        for ax in range(dim):
            b = field.bases[ax]
            if b is None:
                continue
            plan = cached_plan(b, scales[ax])
            shp = list(cur.shape); shp[nt + ax] = plan.M
            out = torch.empty(shp, dtype=cur.dtype, device=cur.device)
            plan.forward(cur.contiguous(), out, nt + ax)
            cur = out
        field.set_device_data(cur, 'c')
