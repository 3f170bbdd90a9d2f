// Batched 1-D spectral transforms along one axis of an N-D array (T1, T2, T3).
//
// One CTA owns a tile of T adjacent lines of the (outer, n, inner) view, stages it in shared memory as
// complex[nc][T+1], runs an in-place mixed-radix FFT (DIF forward: natural in -> digit-reversed out;
// DIT backward: digit-reversed in -> natural out, so no separate permutation pass is ever made: the
// reference's pack / scale / truncate / zero-pad steps read or write through the permutation), and fuses the
// Dedalus conventions into the load and store stages:
//   * RealFourier  : cos/-sin interleaving, 1/N and 2/N scaling, Nyquist drop, dealias pad / truncate,
//                    optional coefficient-space derivative (i k)^m on the backward load
//   * Chebyshev    : DCT-II / DCT-III through the same half-length complex FFT (even/odd reordering +
//                    quarter-wave twiddle), Jacobi normalisation, odd-mode sign flip, truncation,
//                    banded ultraspherical conversion apply (forward) / apply + back-substitution (backward)
//   * ComplexFourier: [0..K,(Nyq),-K..-1] ordering, 1/N scaling
// HBM traffic is exactly one read of the input and one write of the output; loads / stores are coalesced
// along the contiguous direction of the view (across lines when inner > 1, along the line when inner == 1).
#include "db_common.cuh"
#include <cstdlib>

enum { K_RFWD = 0, K_RBWD = 1, K_CFWD = 2, K_CBWD = 3, K_CHFWD = 4, K_CHBWD = 5 };
#define FFT_THREADS 256

struct FftArgs {
    db_fft_plan plan;
    const double* in;
    double* out;
    int64_t outer, inner;
    int32_t n_coeff;
    int32_t T, TP, lgT;
    int32_t deriv;
    double kscale;
    const double* diags_a; int32_t nd_a;    // forward: conversion apply ; backward: pre-apply
    const double* diags_b; int32_t nd_b;    // backward: upper solve
    int32_t cof_off;                        // offset (doubles) of the coefficient staging area in smem
    int64_t tiles_per_outer;
};

__device__ __forceinline__ double2 cmul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ double2 cmulc(double2 a, double2 b) { return make_double2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); }   // a * conj(b)
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ double2 cconj(double2 a) { return make_double2(a.x, -a.y); }
__device__ __forceinline__ double2 ldtw(const double* tw, int j) { return reinterpret_cast<const double2*>(tw)[j]; }

// small DFTs; INV selects exp(+i...) kernels
template <bool INV> __device__ __forceinline__ void dft2(double2* v)
{
    double2 a = v[0], b = v[1];
    v[0] = cadd(a, b); v[1] = csub(a, b);
}
template <bool INV> __device__ __forceinline__ void dft4(double2* v)
{
    double2 a = cadd(v[0], v[2]), b = csub(v[0], v[2]), c = cadd(v[1], v[3]), d = csub(v[1], v[3]);
    // forward: -i*d ; inverse: +i*d
    double2 jd = INV ? make_double2(-d.y, d.x) : make_double2(d.y, -d.x);
    v[0] = cadd(a, c); v[2] = csub(a, c);
    v[1] = cadd(b, jd); v[3] = csub(b, jd);
}
template <bool INV> __device__ __forceinline__ void dft3(double2* v)
{
    const double s = 0.86602540378443864676372317075294;   // sin(pi/3)
    double2 t1 = cadd(v[1], v[2]);
    double2 t2 = make_double2(v[0].x - 0.5 * t1.x, v[0].y - 0.5 * t1.y);
    double2 d = csub(v[1], v[2]);
    // forward: -i*s*d ; inverse: +i*s*d
    double2 t3 = INV ? make_double2(-s * d.y, s * d.x) : make_double2(s * d.y, -s * d.x);
    v[0] = cadd(v[0], t1);
    v[1] = cadd(t2, t3);
    v[2] = csub(t2, t3);
}
// generic odd radix through the twiddle table: w_r^j = tw[(nc/r) * j]
template <bool INV, int R> __device__ __forceinline__ void dftr(double2* v, const double* tw, int nc)
{
    double2 y[R];
    const int step = nc / R;
#pragma unroll
    for (int qp = 0; qp < R; ++qp) {
        double2 acc = v[0];
#pragma unroll
        for (int q = 1; q < R; ++q) {
            double2 w = ldtw(tw, step * ((q * qp) % R));
            acc = cadd(acc, INV ? cmulc(v[q], w) : cmul(v[q], w));
        }
        y[qp] = acc;
    }
#pragma unroll
    for (int q = 0; q < R; ++q) v[q] = y[q];
}

// one radix-R pass over the whole tile; R is a template parameter so the butterfly lives in registers
template <bool INV, int R>
__device__ __forceinline__ void fft_pass_r(double2* buf, int nc, int TP, int lgT, int L, const double* tw)
{
    // all T = 2^lgT columns of the tile are processed (unused columns of a partial tile hold garbage that is never
    // stored), so the column index is a mask and the butterfly index a shift; the division by m uses a 24-bit
    // reciprocal (exact for bf * m < 2^24, i.e. any nc that fits shared memory)
    const int m = L / R;
    const int nbf = nc / R;
    const int tstep = nc / L;
    const unsigned inv_m = (unsigned)(((1u << 24) + m - 1) / m);
    const int Tmask = (1 << lgT) - 1;
    for (int w = threadIdx.x; w < (nbf << lgT); w += blockDim.x) {
        const int t = w & Tmask;
        const int bf = w >> lgT;
        const int b = (int)(((unsigned long long)bf * inv_m) >> 24), k = bf - b * m;
        double2 v[R];
        const int i0 = b * L + k;
#pragma unroll
        for (int q = 0; q < R; ++q) v[q] = buf[(i0 + q * m) * TP + t];
        const int tk = tstep * k;          // tk * q < nc for all q < R: no modulo needed
        if (INV) {   // DIT: twiddle first (conjugate), then butterfly
#pragma unroll
            for (int q = 1; q < R; ++q) v[q] = cmulc(v[q], ldtw(tw, tk * q));
        }
        if (R == 4) dft4<INV>(v);
        else if (R == 2) dft2<INV>(v);
        else if (R == 3) dft3<INV>(v);
        else dftr<INV, R>(v, tw, nc);
        if (!INV) {  // DIF: butterfly first, then twiddle
#pragma unroll
            for (int q = 1; q < R; ++q) v[q] = cmul(v[q], ldtw(tw, tk * q));
        }
#pragma unroll
        for (int q = 0; q < R; ++q) buf[(i0 + q * m) * TP + t] = v[q];
    }
}

// rare large odd radices (7, 11, 13): runtime-radix fallback with the butterfly in local memory
template <bool INV>
__device__ __noinline__ void fft_pass_generic(double2* buf, int nc, int TP, int Tc, int r, int L, const double* tw)
{
    const int m = L / r;
    const int nbf = nc / r;
    const int tstep = nc / L;
    const int step = nc / r;
    for (int w = threadIdx.x; w < nbf * Tc; w += blockDim.x) {
        const int t = w % Tc;
        const int bf = w / Tc;
        const int b = bf / m, k = bf - b * m;
        double2 v[16], y[16];
        const int i0 = b * L + k;
        for (int q = 0; q < r; ++q) {
            v[q] = buf[(i0 + q * m) * TP + t];
            if (INV && q > 0) v[q] = cmulc(v[q], ldtw(tw, tstep * k * q));
        }
        for (int qp = 0; qp < r; ++qp) {
            double2 acc = v[0];
            for (int q = 1; q < r; ++q) {
                double2 ww = ldtw(tw, step * ((q * qp) % r));
                acc = cadd(acc, INV ? cmulc(v[q], ww) : cmul(v[q], ww));
            }
            y[qp] = acc;
        }
        for (int q = 0; q < r; ++q) {
            double2 o = y[q];
            if (!INV && q > 0) o = cmul(o, ldtw(tw, tstep * k * q));
            buf[(i0 + q * m) * TP + t] = o;
        }
    }
}

template <bool INV>
__device__ void fft_pass(double2* buf, int nc, int TP, int lgT, int r, int L, const double* tw)
{
    switch (r) {
        case 4: fft_pass_r<INV, 4>(buf, nc, TP, lgT, L, tw); break;
        case 2: fft_pass_r<INV, 2>(buf, nc, TP, lgT, L, tw); break;
        case 3: fft_pass_r<INV, 3>(buf, nc, TP, lgT, L, tw); break;
        case 5: fft_pass_r<INV, 5>(buf, nc, TP, lgT, L, tw); break;
        default: fft_pass_generic<INV>(buf, nc, TP, 1 << lgT, r, L, tw); break;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Compile-time specialised passes for the benchmark line lengths (tile width 16): every index, stride and twiddle
// step is a constant, the per-thread butterfly loop is fully unrolled and the division bf / m is by a constant.
// ---------------------------------------------------------------------------------------------------------
template <bool INV, int NC, int L, int R>
__device__ __forceinline__ void fft_pass_static(double2* buf, const double* __restrict__ tw)
{
    constexpr int m = L / R, nbf = NC / R, tstep = NC / L, TP = 17;
    constexpr int ITER = (nbf * 16 + FFT_THREADS - 1) / FFT_THREADS;
    const int t = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
    for (int it = 0; it < ITER; ++it) {
        const int bf = ty + 16 * it;
        if ((nbf % 16 != 0) && bf >= nbf) break;
        const int b = bf / m, k = bf - b * m;
        double2* base = buf + (b * L + k) * TP + t;
        double2 v[R];
#pragma unroll
        for (int q = 0; q < R; ++q) v[q] = base[q * m * TP];
        const int tk = tstep * k;
        if (INV) {
#pragma unroll
            for (int q = 1; q < R; ++q) v[q] = cmulc(v[q], ldtw(tw, tk * q));
        }
        if (R == 4) dft4<INV>(v);
        else if (R == 2) dft2<INV>(v);
        else if (R == 3) dft3<INV>(v);
        else dftr<INV, R>(v, tw, NC);
        if (!INV) {
#pragma unroll
            for (int q = 1; q < R; ++q) v[q] = cmul(v[q], ldtw(tw, tk * q));
        }
#pragma unroll
        for (int q = 0; q < R; ++q) base[q * m * TP] = v[q];
    }
}

template <int NC, int L, int R, int... REST>
__device__ __forceinline__ void static_dif(double2* buf, const double* tw)
{
    fft_pass_static<false, NC, L, R>(buf, tw);
    __syncthreads();
    if constexpr (sizeof...(REST) > 0) static_dif<NC, L / R, REST...>(buf, tw);
}
template <int NC, int L, int R, int... REST>
__device__ __forceinline__ void static_dit(double2* buf, const double* tw)
{
    if constexpr (sizeof...(REST) > 0) static_dit<NC, L / R, REST...>(buf, tw);
    fft_pass_static<true, NC, L, R>(buf, tw);
    __syncthreads();
}

// returns true if a specialised path handled the transform (radix lists must match dedalus_b200/fftplan.py factorize)
template <bool INV>
__device__ __forceinline__ bool fft_static_dispatch(double2* buf, const db_fft_plan& p, int T)
{
    if (T != 16) return false;
    const double* tw = p.tw;
    switch (p.nc) {
        case 192: if (INV) static_dit<192, 192, 4, 4, 4, 3>(buf, tw); else static_dif<192, 192, 4, 4, 4, 3>(buf, tw); return true;
        case 384: if (INV) static_dit<384, 384, 4, 4, 4, 2, 3>(buf, tw); else static_dif<384, 384, 4, 4, 4, 2, 3>(buf, tw); return true;
        case 96:  if (INV) static_dit<96, 96, 4, 4, 2, 3>(buf, tw); else static_dif<96, 96, 4, 4, 2, 3>(buf, tw); return true;
        case 48:  if (INV) static_dit<48, 48, 4, 4, 3>(buf, tw); else static_dif<48, 48, 4, 4, 3>(buf, tw); return true;
        default: return false;
    }
}

__device__ void fft_dif(double2* buf, const db_fft_plan& p, int TP, int lgT)
{
    if (fft_static_dispatch<false>(buf, p, 1 << lgT)) return;
    int L = p.nc;
    for (int s = 0; s < p.nrad; ++s) {
        fft_pass<false>(buf, p.nc, TP, lgT, p.rad[s], L, p.tw);
        L /= p.rad[s];
        __syncthreads();
    }
}
__device__ void fft_dit(double2* buf, const db_fft_plan& p, int TP, int lgT)
{
    if (fft_static_dispatch<true>(buf, p, 1 << lgT)) return;
    int Ls[16];
    int L = p.nc;
    for (int s = 0; s < p.nrad; ++s) { Ls[s] = L; L /= p.rad[s]; }
    for (int s = p.nrad - 1; s >= 0; --s) {
        fft_pass<true>(buf, p.nc, TP, lgT, p.rad[s], Ls[s], p.tw);
        __syncthreads();
    }
}

// element (j, t) of the tile in global memory: lines are adjacent along `inner` (strided mode) or whole
// contiguous lines (inner == 1)
struct TileGeom {
    int64_t base;     // offset of (line 0 of tile, element 0)
    int64_t estride;  // stride between consecutive elements of a line
    int64_t lstride;  // stride between consecutive lines of the tile
    int Tc;           // lines in this tile
};

__device__ __forceinline__ TileGeom tile_geom(const FftArgs& a, int len, int cplx)
{
    // strided axis: grid = (tiles per outer slab, outer) so no division is needed; contiguous axis: grid.x = tile
    TileGeom g;
    if (a.inner == 1) {
        const int64_t l0 = ((int64_t)blockIdx.y * gridDim.x + blockIdx.x) * a.T;
        const int64_t rem = a.outer - l0;
        g.Tc = rem < a.T ? (int)rem : a.T;
        g.base = l0 * len * cplx;
        g.estride = cplx;
        g.lstride = (int64_t)len * cplx;
    } else {
        const int64_t o = blockIdx.y;
        const int64_t i0 = (int64_t)blockIdx.x * a.T;
        const int64_t rem = a.inner - i0;
        g.Tc = rem < a.T ? (int)rem : a.T;
        g.base = (o * len * a.inner + i0) * cplx;
        g.estride = a.inner * cplx;
        g.lstride = cplx;
    }
    return g;
}

// Visit every element (j, t) of the tile with the global-memory-contiguous index fastest across lanes and
// only additions in the inner loop: f(j, t, global offset).
template <class F>
__device__ __forceinline__ void tile_iter(int len, const TileGeom& g, bool contiguous, int lgT, F f)
{
    if (contiguous) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
        for (int t = warp; t < g.Tc; t += nw) {
            const int64_t off = g.base + t * g.lstride;
            for (int j = lane; j < len; j += 32) f(j, t, off + j * g.estride);
        }
    } else {
        const int t = threadIdx.x & ((1 << lgT) - 1);
        if (t < g.Tc) {
            const int js = blockDim.x >> lgT;
            int j = threadIdx.x >> lgT;
            int64_t off = g.base + t * g.lstride + j * g.estride;
            const int64_t step = js * g.estride;
            for (; j < len; j += js, off += step) f(j, t, off);
        }
    }
}

__device__ __forceinline__ double2 rot_i_pow(double2 z, int ph)
{
    // z * i^ph
    return (ph == 0) ? z : (ph == 1) ? make_double2(-z.y, z.x) : (ph == 2) ? make_double2(-z.x, -z.y) : make_double2(z.y, -z.x);
}

// DIRECT: real-Fourier kernels on a strided axis read / write the coefficient rows straight from / to global memory
// (each row segment is already a coalesced run across the tile's lines), skipping the shared-memory staging area:
// one fewer shared round trip and barrier, and 40% less shared memory per CTA (-> 3-4 CTAs per SM)
template <int KIND, bool DIRECT>
__global__ void __launch_bounds__(FFT_THREADS, DIRECT ? 3 : 2) k_fft(FftArgs a)
{
    DB_SMEM(double, smem);
    double2* buf = reinterpret_cast<double2*>(smem);
    double* cof = smem + a.cof_off;
    const db_fft_plan& p = a.plan;
    const int n = p.n, nc = p.nc, M = a.n_coeff, TP = a.TP, lgT = a.lgT, T = a.T;
    const bool contiguous = (a.inner == 1);
    const bool is_fwd = (KIND == K_RFWD || KIND == K_CFWD || KIND == K_CHFWD);
    const bool is_cplx = (KIND == K_CFWD || KIND == K_CBWD);
    const int cplx = is_cplx ? 2 : 1;
    const TileGeom gi = tile_geom(a, is_fwd ? n : M, cplx);
    const TileGeom go = tile_geom(a, is_fwd ? M : n, cplx);
    if (gi.Tc <= 0) return;                       // padding block of a 2-D grid over contiguous lines
    const int Tmask = T - 1;
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const double* __restrict__ gin = a.in;
    double* __restrict__ gout = a.out;

    if (is_fwd) {
        // ---------------- load grid data straight into the complex work buffer ----------------
        if (KIND == K_CFWD) {
            tile_iter(n, gi, contiguous, lgT, [&](int j, int t, int64_t off) {
                buf[j * TP + t] = make_double2(gin[off], gin[off + 1]);
            });
        } else {
            double* rb = smem;   // real view: element pp of line t at ((pp>>1)*TP + t)*2 + (pp&1) (half) or (pp*TP+t)*2 (full)
            const int half = p.half;
            tile_iter(n, gi, contiguous, lgT, [&](int j, int t, int64_t off) {
                const double v = gin[off];
                int pp = j;
                if (KIND == K_CHFWD) pp = (j & 1) ? (n - 1 - (j >> 1)) : (j >> 1);
                if (half) rb[(((pp >> 1) * TP + t) << 1) + (pp & 1)] = v;
                else { rb[(pp * TP + t) << 1] = v; rb[((pp * TP + t) << 1) + 1] = 0.0; }
            });
        }
        __syncthreads();
        fft_dif(buf, p, TP, lgT);
        // ---------------- post-processing into the coefficient staging area ----------------
        if (KIND == K_CFWD) {
            const int KM = (M - 1) / 2;
            int Kmax = (n - 1) / 2; if (KM < Kmax) Kmax = KM;
            const double sc = 1.0 / n;
            for (int w = tid; w < (M << lgT); w += nthreads) {
                const int t = w & Tmask, c = w >> lgT;
                const int k = (c + KM) % M - KM;
                double2 z = make_double2(0.0, 0.0);
                if (k <= Kmax && -k <= Kmax) {
                    const int kk = (k < 0) ? k + n : k;
                    z = buf[p.iperm[kk] * TP + t];
                    z.x *= sc; z.y *= sc;
                }
                cof[(c * TP + t) * 2] = z.x; cof[(c * TP + t) * 2 + 1] = z.y;
            }
        } else if (p.half) {
            // pairs (k, nc-k): X_k = E + w^k O, X_{nc-k} = conj(E - w^k O)
            const int npair = nc / 2 + 1;
            int Kmax, Kin = 0;
            double s0 = 0.0, s1 = 0.0;
            if (KIND == K_RFWD) {
                Kmax = (n - 1) / 2; { int KM = (M - 1) / 2; if (KM < Kmax) Kmax = KM; }
                // coefficient slots beyond the pairs' reach (M > n + 2) are zero
                for (int w = tid + ((2 * (nc + 1)) << lgT); w < (M << lgT); w += nthreads) {
                    if (DIRECT) { if ((w & Tmask) < go.Tc) gout[go.base + (int64_t)(w >> lgT) * go.estride + (w & Tmask) * go.lstride] = 0.0; }
                    else cof[(w >> lgT) * TP + (w & Tmask)] = 0.0;
                }
            } else {
                Kmax = 0;
                Kin = (M < n) ? M : n;
                s0 = 0.5 / n * 1.7724538509055160272981674833411;      // sqrt(pi)/(2N)
                s1 = 1.0 / n * 1.2533141373155002512078826424055;      // sqrt(pi/2)/N
                for (int w = tid + (Kin << lgT); w < (M << lgT); w += nthreads) cof[(w >> lgT) * TP + (w & Tmask)] = 0.0;
            }
            const double rsc = 2.0 / n;
            for (int w = tid; w < (npair << lgT); w += nthreads) {
                const int t = w & Tmask, ka = w >> lgT, kb = nc - ka;
                const double2 za = buf[p.iperm[ka] * TP + t];
                const double2 zb = buf[p.iperm[(kb == nc) ? 0 : kb] * TP + t];
                const double2 E = make_double2(0.5 * (za.x + zb.x), 0.5 * (za.y - zb.y));
                const double2 D = make_double2(za.x - zb.x, za.y + zb.y);          // za - conj(zb)
                const double2 O = make_double2(0.5 * D.y, -0.5 * D.x);             // -i/2 * D
                const double2 W = cmul(ldtw(p.twr, ka), O);
                const double2 Xa = cadd(E, W);
                const double2 Xb = make_double2(E.x - W.x, -(E.y - W.y));
                if (KIND == K_RFWD) {
                    // coefficient pair (2k, 2k+1) = (2/N) (Re, Im) X_k ; k = 0: (Re X_0 / N, 0); k > Kmax: 0
                    if (2 * ka < M) {
                        const bool ok = ka <= Kmax;
                        const double vr = ok ? Xa.x * ((ka == 0) ? 0.5 * rsc : rsc) : 0.0;
                        const double vi = (ok && ka > 0) ? Xa.y * rsc : 0.0;
                        if (DIRECT) {
                            if (t < go.Tc) {
                                const int64_t o = go.base + (int64_t)(2 * ka) * go.estride + t * go.lstride;
                                gout[o] = vr;
                                if (2 * ka + 1 < M) gout[o + go.estride] = vi;
                            }
                        } else {
                            cof[(2 * ka) * TP + t] = vr;
                            if (2 * ka + 1 < M) cof[(2 * ka + 1) * TP + t] = vi;
                        }
                    }
                    if (kb != ka && 2 * kb < M) {
                        const bool ok = kb <= Kmax;
                        const double vr = ok ? Xb.x * rsc : 0.0, vi = ok ? Xb.y * rsc : 0.0;
                        if (DIRECT) {
                            if (t < go.Tc) {
                                const int64_t o = go.base + (int64_t)(2 * kb) * go.estride + t * go.lstride;
                                gout[o] = vr;
                                if (2 * kb + 1 < M) gout[o + go.estride] = vi;
                            }
                        } else {
                            cof[(2 * kb) * TP + t] = vr;
                            if (2 * kb + 1 < M) cof[(2 * kb + 1) * TP + t] = vi;
                        }
                    }
                } else {
                    // C_k = 2 Re(q^k X_k) (k <= nc), C_{n-k} = -2 Im(q^k X_k) (0 < k < nc); scaled, odd modes negated
                    const double2 Wa = cmul(ldtw(p.twq, ka), Xa);
                    if (ka < Kin) { double v = 2.0 * Wa.x * ((ka == 0) ? s0 : s1); cof[ka * TP + t] = (ka & 1) ? -v : v; }
                    const int ka2 = n - ka;
                    if (ka >= 1 && ka < nc && ka2 < Kin) { double v = -2.0 * Wa.y * s1; cof[ka2 * TP + t] = (ka2 & 1) ? -v : v; }
                    if (kb != ka) {
                        const double2 Wb = cmul(ldtw(p.twq, kb), Xb);
                        if (kb < Kin) { double v = 2.0 * Wb.x * s1; cof[kb * TP + t] = (kb & 1) ? -v : v; }
                        const int kb2 = n - kb;
                        if (kb < nc && kb2 < Kin) { double v = -2.0 * Wb.y * s1; cof[kb2 * TP + t] = (kb2 & 1) ? -v : v; }
                    }
                }
            }
        } else if (KIND == K_RFWD) {
            int Kmax = (n - 1) / 2; { int KM = (M - 1) / 2; if (KM < Kmax) Kmax = KM; }
            const int nk = (M + 1) / 2;
            for (int w = tid; w < (nk << lgT); w += nthreads) {
                const int t = w & Tmask, k = w >> lgT;
                double re = 0.0, im = 0.0;
                if (k <= Kmax) {
                    const double2 X = buf[p.iperm[k] * TP + t];
                    const double sc = (k == 0) ? 1.0 / n : 2.0 / n;
                    re = X.x * sc; im = (k == 0) ? 0.0 : X.y * sc;
                }
                cof[(2 * k) * TP + t] = re;
                if (2 * k + 1 < M) cof[(2 * k + 1) * TP + t] = im;
            }
        } else {  // K_CHFWD, odd n: full complex FFT of the reordered real data
            const int Kin = (M < n) ? M : n;
            const double s0 = 0.5 / n * 1.7724538509055160272981674833411;
            const double s1 = 1.0 / n * 1.2533141373155002512078826424055;
            for (int w = tid; w < (Kin << lgT); w += nthreads) {
                const int t = w & Tmask, k = w >> lgT;
                const double2 W = cmul(ldtw(p.twq, k), buf[p.iperm[k] * TP + t]);
                const double v = 2.0 * W.x * ((k == 0) ? s0 : s1);
                cof[k * TP + t] = (k & 1) ? -v : v;
            }
            for (int w = tid + (Kin << lgT); w < (M << lgT); w += nthreads) cof[(w >> lgT) * TP + (w & Tmask)] = 0.0;
        }
        if (KIND == K_RFWD && DIRECT) return;          // coefficients already written from the pair loop
        __syncthreads();
        // ---------------- store (with the banded conversion fused for Chebyshev) ----------------
        if (KIND == K_CFWD) {
            tile_iter(M, go, contiguous, lgT, [&](int c, int t, int64_t off) {
                gout[off] = cof[(c * TP + t) * 2]; gout[off + 1] = cof[(c * TP + t) * 2 + 1];
            });
        } else if (KIND == K_CHFWD && a.nd_a > 0) {
            // banded conversion fused into the store; its diagonals are staged in the (now free) work buffer
            const int Kin = (M < n) ? M : n;
            const int nd = a.nd_a;
            double* dg = smem;
            for (int e = tid; e < nd * M; e += nthreads) dg[e] = a.diags_a[e];
            __syncthreads();
            tile_iter(M, go, contiguous, lgT, [&](int i, int t, int64_t off) {
                double acc = 0.0;
                if (i < Kin) {
                    for (int d = 0; d < nd && i + d < Kin; ++d)
                        acc = fma(dg[d * M + i], cof[(i + d) * TP + t], acc);
                }
                gout[off] = acc;
            });
        } else {
            tile_iter(M, go, contiguous, lgT, [&](int c, int t, int64_t off) { gout[off] = cof[c * TP + t]; });
        }
    } else {
        // ================= backward: stage coefficients =================
        if (KIND == K_CBWD) {
            tile_iter(M, gi, contiguous, lgT, [&](int c, int t, int64_t off) {
                cof[(c * TP + t) * 2] = gin[off]; cof[(c * TP + t) * 2 + 1] = gin[off + 1];
            });
            __syncthreads();
        } else if (!(KIND == K_RBWD && DIRECT)) {
            tile_iter(M, gi, contiguous, lgT, [&](int c, int t, int64_t off) { cof[c * TP + t] = gin[off]; });
            __syncthreads();
        }
        if (KIND == K_CHBWD) {
            int Kmax = n - 1; if (M - 1 < Kmax) Kmax = M - 1;
            // banded work on the staged coefficients: pre-apply, then truncate (parallel, cof -> tmp), back-substitution
            // (one thread per line, solved values kept in a register window; tmp -> cof).  Without banded work the
            // modes above Kmax are dropped when the spectrum is built.
            double* tmp = smem;                           // the complex work buffer is still unused here
            if (a.nd_a > 0 || a.nd_b > 0) {
                // the derivative reads all M coefficients; the transform of the derivative basis then drops the modes
                // above Kmax (M > n), as DifferentiateJacobi followed by the backward transform does
                for (int w = tid; w < (M << lgT); w += nthreads) {
                    const int t = w & Tmask, i = w >> lgT;
                    double acc;
                    if (i > Kmax) {
                        acc = 0.0;
                    } else if (a.nd_a > 0) {
                        acc = 0.0;
                        for (int d = 0; d < a.nd_a && i + d < M; ++d)
                            acc = fma(a.diags_a[(int64_t)d * M + i], cof[(i + d) * TP + t], acc);
                    } else {
                        acc = cof[i * TP + t];
                    }
                    tmp[i * TP + t] = acc;
                }
                __syncthreads();
                if (a.nd_b > 0) {
                    if (tid < T) {
                        const int t = tid;
                        double win[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};       // x_{i+1} .. x_{i+7}
                        const int nd = a.nd_b < 8 ? a.nd_b : 8;
                        for (int i = M - 1; i >= 0; --i) {
                            double acc = tmp[i * TP + t];
#pragma unroll
                            for (int d = 1; d < 8; ++d)
                                if (d < nd) acc = fma(-a.diags_b[(int64_t)d * M + i], win[d - 1], acc);
                            // wider bands (alpha + deriv >= 4): x_{i+8} .. are already stored in cof
                            for (int d = 8; d < a.nd_b && i + d < M; ++d)
                                acc = fma(-a.diags_b[(int64_t)d * M + i], cof[(i + d) * TP + t], acc);
                            const double xi = acc * a.diags_b[i];                  // row 0 = reciprocal diagonal
#pragma unroll
                            for (int d = 6; d > 0; --d) win[d] = win[d - 1];
                            win[0] = xi;
                            cof[i * TP + t] = xi;
                        }
                    }
                } else {
                    for (int w = tid; w < (M << lgT); w += nthreads) {
                        const int t = w & Tmask, i = w >> lgT;
                        cof[i * TP + t] = tmp[i * TP + t];
                    }
                }
                __syncthreads();
            }
        }
        // ================= build the (digit-reversed) spectrum for the DIT passes =================
        if (KIND == K_CBWD) {
            const int KM = (M - 1) / 2;
            int Kmax = (n - 1) / 2; if (KM < Kmax) Kmax = KM;
            for (int w = tid; w < (nc << lgT); w += nthreads) {
                const int t = w & Tmask, pos = w >> lgT;
                int k = p.perm[pos];
                if (k > n / 2) k -= n;                       // signed wavenumber
                double2 z = make_double2(0.0, 0.0);
                if (k <= Kmax && -k <= Kmax) {
                    const int c = (k >= 0) ? k : M + k;
                    z = make_double2(cof[(c * TP + t) * 2], cof[(c * TP + t) * 2 + 1]);
                    if (a.deriv > 0) {
                        double f = 1.0;
                        for (int d = 0; d < a.deriv; ++d) f *= a.kscale * k;
                        z = rot_i_pow(z, a.deriv & 3);
                        z.x *= f; z.y *= f;
                    }
                }
                buf[pos * TP + t] = z;
            }
        } else {
            // half-spectrum value X_k (k = 0..nc) as a function of the staged real coefficients
            int Kmax;
            if (KIND == K_RBWD) { Kmax = (n - 1) / 2; int KM = (M - 1) / 2; if (KM < Kmax) Kmax = KM; }
            else { Kmax = n - 1; if (M - 1 < Kmax) Kmax = M - 1; }
            const double c0 = 0.56418958354775628694807945156077;     // 1/sqrt(pi)
            const double c1 = 0.39894228040143267793994605993438;     // 1/sqrt(2 pi)
            const int deriv = a.deriv, dph = a.deriv & 3;
            const double kscale = a.kscale;
            auto chat = [&](int k, int t) -> double {              // scaled, sign-flipped Chebyshev coefficient
                if (k > Kmax || k >= n) return 0.0;
                const double v = cof[k * TP + t] * ((k == 0) ? c0 : c1);
                return (k & 1) ? -v : v;
            };
            auto getX = [&](int k, int t) -> double2 {
                if (KIND == K_RBWD) {
                    if (k > Kmax) return make_double2(0.0, 0.0);
                    double2 z;
                    if (DIRECT) {
                        if (t >= gi.Tc) return make_double2(0.0, 0.0);
                        const int64_t o = gi.base + (int64_t)(2 * k) * gi.estride + t * gi.lstride;
                        if (k == 0) return make_double2((deriv > 0) ? 0.0 : gin[o], 0.0);
                        z = make_double2(0.5 * gin[o], 0.5 * gin[o + gi.estride]);
                    } else {
                        if (k == 0) return make_double2((deriv > 0) ? 0.0 : cof[t], 0.0);
                        z = make_double2(0.5 * cof[(2 * k) * TP + t], 0.5 * cof[(2 * k + 1) * TP + t]);
                    }
                    if (deriv > 0) {
                        double f = 1.0;
                        for (int d = 0; d < deriv; ++d) f *= kscale * k;
                        z = rot_i_pow(z, dph);
                        z.x *= f; z.y *= f;
                    }
                    return z;
                } else {
                    if (k == 0) return make_double2(chat(0, t), 0.0);
                    const double2 w = cconj(ldtw(p.twq, k));                  // exp(+i pi k / 2n)
                    return cmul(w, make_double2(chat(k, t), -chat(n - k, t))); // H_k = q^-k (c_k - i c_{n-k})
                }
            };
            if (p.half) {
                // pairs (k, nc-k): Z_k = E + iO, Z_{nc-k} = conj(E - iO), E = X_k + conj X_{nc-k}, O = (X_k - conj X_{nc-k}) w^{-k}
                const int npair = nc / 2 + 1;
                for (int w = tid; w < (npair << lgT); w += nthreads) {
                    const int t = w & Tmask, ka = w >> lgT, kb = nc - ka;
                    const double2 xa = getX(ka, t);
                    const double2 xb = getX(kb, t);
                    const double2 E = make_double2(xa.x + xb.x, xa.y - xb.y);
                    const double2 D = make_double2(xa.x - xb.x, xa.y + xb.y);
                    const double2 O = cmulc(D, ldtw(p.twr, ka));
                    buf[p.iperm[ka] * TP + t] = make_double2(E.x - O.y, E.y + O.x);
                    if (kb != ka && kb < nc) buf[p.iperm[kb] * TP + t] = make_double2(E.x + O.y, -(E.y - O.x));
                }
            } else {
                for (int w = tid; w < (nc << lgT); w += nthreads) {
                    const int t = w & Tmask, pos = w >> lgT;
                    const int k = p.perm[pos];
                    double2 z;
                    if (KIND == K_RBWD) {
                        // hermitian extension: Z_k = X_k (k <= n/2), Z_k = conj X_{n-k} otherwise; X holds c_k/2
                        if (2 * k <= n) z = getX(k, t);
                        else z = cconj(getX(n - k, t));
                    } else {
                        // G_k = c'_k exp(i pi k / 2n), c'_0 = c_0, c'_k = 2 c_k ; output = Re IDFT(G)
                        const double ck = chat(k, t) * ((k == 0) ? 1.0 : 2.0);
                        const double2 ww = cconj(ldtw(p.twq, k));
                        z = make_double2(ww.x * ck, ww.y * ck);
                    }
                    buf[pos * TP + t] = z;
                }
            }
        }
        __syncthreads();
        fft_dit(buf, p, TP, lgT);
        // ================= store grid data =================
        if (KIND == K_CBWD) {
            tile_iter(n, go, contiguous, lgT, [&](int j, int t, int64_t off) {
                const double2 z = buf[j * TP + t];
                gout[off] = z.x; gout[off + 1] = z.y;
            });
        } else {
            const double* rb = smem;
            const int half = p.half;
            tile_iter(n, go, contiguous, lgT, [&](int j, int t, int64_t off) {
                int pp = j;
                if (KIND == K_CHBWD) pp = (j & 1) ? (n - 1 - (j >> 1)) : (j >> 1);
                gout[off] = half ? rb[(((pp >> 1) * TP + t) << 1) + (pp & 1)] : rb[(pp * TP + t) << 1];
            });
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
int db_rfft_regs_try(bool fwd, const db_fft_plan* plan, const double* in, double* out, int64_t outer, int32_t n_coeff,
                     int64_t inner, int32_t deriv, double kscale, void* stream,
                     int32_t in_rpb, int64_t in_blk_stride, int32_t out_rpb, int64_t out_blk_stride,
                     int32_t out_peers, double* const* out_blk_ptr);       // rfft_regs.cu
int db_cheb_regs_try(bool fwd, const db_fft_plan* plan, const double* in, double* out, int64_t lines, int32_t n_coeff,
                     const double* diags, int32_t nd, const double* pre, int32_t npre, const double* sol2, void* stream);

template <int KIND>
static int launch_fft(const db_fft_plan* plan, const double* in, double* out, int64_t outer, int32_t n_coeff, int64_t inner,
                      int32_t deriv, double kscale, const double* da, int32_t nda, const double* db_, int32_t ndb,
                      void* stream, const char* name)
{
    if (outer <= 0 || inner <= 0) return 0;
    if (plan->n <= 0 || plan->nc <= 0 || n_coeff <= 0) { db_set_error("%s: bad sizes", name); return 1; }
    if (KIND == K_RFWD || KIND == K_RBWD) {
        // dealiased sizes on a strided axis: register-resident two-stage kernels (rfft_regs.cu)
        const int rc = db_rfft_regs_try(KIND == K_RFWD, plan, in, out, outer, n_coeff, inner, deriv, kscale, stream, 0, 0, 0, 0, 0, nullptr);
        if (rc >= 0) return rc;
    }
    if ((KIND == K_CHFWD || (KIND == K_CHBWD && nda == 0 && ndb == 0)) && inner == 1) {
        const int rc = db_cheb_regs_try(KIND == K_CHFWD, plan, in, out, outer, n_coeff, KIND == K_CHFWD ? da : nullptr, KIND == K_CHFWD ? nda : 0,
                                        nullptr, 0, nullptr, stream);
        if (rc >= 0) return rc;
    }
    FftArgs a;
    a.plan = *plan; a.in = in; a.out = out; a.outer = outer; a.inner = inner; a.n_coeff = n_coeff;
    a.deriv = deriv; a.kscale = kscale; a.diags_a = da; a.nd_a = nda; a.diags_b = db_; a.nd_b = ndb;
    const bool is_cplx = (KIND == K_CFWD || KIND == K_CBWD);
    const bool direct = (KIND == K_RFWD || KIND == K_RBWD) && inner > 1 && plan->half;
    // choose the tile width: up to 16 lines, shrunk until the CTA fits ~110 KB (2 CTAs / SM) or, failing that,
    // the 227 KB per-CTA limit
    int T = 16;
    { const char* e = getenv("DB_FFT_T"); if (e) { int v = atoi(e); if (v == 1 || v == 2 || v == 4 || v == 8 || v == 16 || v == 32) T = v; } }
    const int64_t lines_dir = (inner == 1) ? outer : inner;
    // work-buffer rows (doubles per column): the complex FFT buffer, which the Chebyshev backward kernel also uses
    // as scratch for n_coeff staged coefficients
    size_t buf_rows = (size_t)2 * plan->nc;
    if (KIND == K_CHBWD && (size_t)n_coeff > buf_rows) buf_rows = (size_t)n_coeff;
    if (KIND == K_CHFWD && nda > 0 && (size_t)nda * n_coeff > buf_rows * 2) buf_rows = ((size_t)nda * n_coeff + 1) / 2;   // >= nd*M doubles even at T = 1
    auto smem_bytes = [&](int t) -> size_t {
        return (buf_rows * (t + 1) + (direct ? 0 : (size_t)(is_cplx ? 2 : 1) * n_coeff * (t + 1))) * sizeof(double);
    };
    while (T > 1 && smem_bytes(T) > (size_t)110 * 1024) T /= 2;
    while (T > 1 && T / 2 >= lines_dir) T /= 2;    // do not waste lanes on tiny problems
    size_t bytes = smem_bytes(T);
    if (bytes > (size_t)DB_MAX_SMEM) { db_set_error("%s: transform length %d too large for shared memory", name, plan->n); return 1; }
    a.T = T; a.TP = T + 1;
    a.lgT = 0; while ((1 << a.lgT) < T) ++a.lgT;
    a.cof_off = (int32_t)(buf_rows * a.TP);
    dim3 grid;
    if (inner == 1) {
        a.tiles_per_outer = 0;
        const int64_t tiles = (outer + T - 1) / T;
        const int64_t gx = tiles < 32768 ? tiles : 32768;
        const int64_t gy = (tiles + gx - 1) / gx;
        if (gy > 65535) { db_set_error("%s: too many tiles", name); return 1; }
        grid = dim3((unsigned)gx, (unsigned)gy);
    } else {
        a.tiles_per_outer = (inner + T - 1) / T;
        if (outer > 65535 || a.tiles_per_outer > 2147483647LL) { db_set_error("%s: outer extent %lld too large for a strided transform", name, (long long)outer); return 1; }
        grid = dim3((unsigned)a.tiles_per_outer, (unsigned)outer);
    }
#ifndef DB_EMU
    static bool attr_set[6][2] = {{false, false}, {false, false}, {false, false}, {false, false}, {false, false}, {false, false}};
    if (!attr_set[KIND][direct ? 1 : 0]) {
        if (direct) cudaFuncSetAttribute(k_fft<KIND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DB_MAX_SMEM);
        else cudaFuncSetAttribute(k_fft<KIND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DB_MAX_SMEM);
        attr_set[KIND][direct ? 1 : 0] = true;
    }
#endif
    if (direct) DB_LAUNCH((k_fft<KIND, true>), grid, dim3(FFT_THREADS), bytes, stream, a);
    else DB_LAUNCH((k_fft<KIND, false>), grid, dim3(FFT_THREADS), bytes, stream, a);
    return db_check_launch(name);
}

extern "C" int db_rfft_forward(const db_fft_plan* plan, const double* g, double* c, int64_t outer, int32_t n_coeff, int64_t inner, void* stream)
{ return launch_fft<K_RFWD>(plan, g, c, outer, n_coeff, inner, 0, 0.0, nullptr, 0, nullptr, 0, stream, "rfft_forward"); }

extern "C" int db_rfft_backward(const db_fft_plan* plan, const double* c, double* g, int64_t outer, int32_t n_coeff, int64_t inner,
                                int32_t deriv, double kscale, void* stream)
{ return launch_fft<K_RBWD>(plan, c, g, outer, n_coeff, inner, deriv, kscale, nullptr, 0, nullptr, 0, stream, "rfft_backward"); }

// Blocked variants (X1): see include/dedalus_b200.h.  Only the register-resident kernels implement them; 2 = not covered.
extern "C" int db_rfft_forward_blocked(const db_fft_plan* plan, const double* g, double* c, int64_t outer, int32_t n_coeff, int64_t inner,
                                       int32_t in_rpb, int64_t in_blk_stride, int32_t out_rpb, int64_t out_blk_stride, void* stream)
{
    if (outer <= 0 || inner <= 0) return 0;
    const int rc = db_rfft_regs_try(true, plan, g, c, outer, n_coeff, inner, 0, 0.0, stream, in_rpb, in_blk_stride, out_rpb, out_blk_stride, 0, nullptr);
    return rc < 0 ? 2 : rc;
}

extern "C" int db_rfft_backward_blocked(const db_fft_plan* plan, const double* c, double* g, int64_t outer, int32_t n_coeff, int64_t inner,
                                        int32_t deriv, double kscale,
                                        int32_t in_rpb, int64_t in_blk_stride, int32_t out_rpb, int64_t out_blk_stride, void* stream)
{
    if (outer <= 0 || inner <= 0) return 0;
    const int rc = db_rfft_regs_try(false, plan, c, g, outer, n_coeff, inner, deriv, kscale, stream, in_rpb, in_blk_stride, out_rpb, out_blk_stride, 0, nullptr);
    return rc < 0 ? 2 : rc;
}

// Peer variants (X1 as the transform's own stores): output block b goes to out_blocks[b] (a peer GPU's receive buffer mapped
// into this process) instead of out + b * blk_stride.  `local_out` is only the 16-byte-aligned origin of the column offsets.
extern "C" int db_rfft_forward_peer(const db_fft_plan* plan, const double* g, double* local_out, int64_t outer, int32_t n_coeff, int64_t inner,
                                    int32_t in_rpb, int64_t in_blk_stride, int32_t out_rpb, int32_t n_peers, double* const* out_blocks, void* stream)
{
    if (outer <= 0 || inner <= 0) return 0;
    const int rc = db_rfft_regs_try(true, plan, g, local_out, outer, n_coeff, inner, 0, 0.0, stream, in_rpb, in_blk_stride, out_rpb, 0, n_peers, out_blocks);
    return rc < 0 ? 2 : rc;
}

extern "C" int db_rfft_backward_peer(const db_fft_plan* plan, const double* c, double* local_out, int64_t outer, int32_t n_coeff, int64_t inner,
                                     int32_t deriv, double kscale, int32_t in_rpb, int64_t in_blk_stride, int32_t out_rpb,
                                     int32_t n_peers, double* const* out_blocks, void* stream)
{
    if (outer <= 0 || inner <= 0) return 0;
    const int rc = db_rfft_regs_try(false, plan, c, local_out, outer, n_coeff, inner, deriv, kscale, stream, in_rpb, in_blk_stride, out_rpb, 0, n_peers, out_blocks);
    return rc < 0 ? 2 : rc;
}

extern "C" int db_cfft_forward(const db_fft_plan* plan, const double* g, double* c, int64_t outer, int32_t n_coeff, int64_t inner, void* stream)
{ return launch_fft<K_CFWD>(plan, g, c, outer, n_coeff, inner, 0, 0.0, nullptr, 0, nullptr, 0, stream, "cfft_forward"); }

extern "C" int db_cfft_backward(const db_fft_plan* plan, const double* c, double* g, int64_t outer, int32_t n_coeff, int64_t inner,
                                int32_t deriv, double kscale, void* stream)
{ return launch_fft<K_CBWD>(plan, c, g, outer, n_coeff, inner, deriv, kscale, nullptr, 0, nullptr, 0, stream, "cfft_backward"); }

extern "C" int db_cheb_forward(const db_fft_plan* plan, const double* g, double* c, int64_t outer, int32_t n_coeff, int64_t inner,
                               const double* conv_diags, int32_t conv_ndiag, void* stream)
{ return launch_fft<K_CHFWD>(plan, g, c, outer, n_coeff, inner, 0, 0.0, conv_diags, conv_ndiag, nullptr, 0, stream, "cheb_forward"); }

extern "C" int db_cheb_backward_scan(const db_fft_plan* plan, const double* c, double* g, int64_t lines, int32_t n_coeff,
                                     const double* pre_diags, int32_t pre_ndiag, const double* solve2_diags, void* stream)
{
    if (lines <= 0) return 0;
    const int rc = db_cheb_regs_try(false, plan, c, g, lines, n_coeff, nullptr, 0, pre_diags, pre_ndiag, solve2_diags, stream);
    return rc < 0 ? 2 : rc;            // 2: this size / alignment is not covered (no error recorded): use db_band_lines + db_cheb_backward
}

extern "C" int db_cheb_backward(const db_fft_plan* plan, const double* c, double* g, int64_t outer, int32_t n_coeff, int64_t inner,
                                const double* pre_diags, int32_t pre_ndiag, const double* solve_diags, int32_t solve_ndiag, void* stream)
{ return launch_fft<K_CHBWD>(plan, c, g, outer, n_coeff, inner, 0, 0.0, pre_diags, pre_ndiag, solve_diags, solve_ndiag, stream, "cheb_backward"); }


// ---------------------------------------------------------------------------------------------------------
// banded apply + upper back-substitution along contiguous lines: one warp per 32 lines
// ---------------------------------------------------------------------------------------------------------
#define BL_LINES 32
#define BL_THREADS 256
__global__ void __launch_bounds__(BL_THREADS)
k_band_lines(const double* __restrict__ in, double* __restrict__ out, int64_t lines, int n,
             const double* __restrict__ pre, int npre, const double* __restrict__ sol, int nsol)
{
    // 32 lines per CTA staged as sm[j][line] (conflict-free for both phases).  The banded pre-apply is evaluated
    // while loading (each output element reads its npre neighbours straight from global memory: fully parallel,
    // overlapping reads hit L1); the back-substitution diagonals are staged in shared memory so that the serial
    // recurrence of warp 0 (one line per lane, solved values in a register window) never waits on global memory.
    DB_SMEM(double, sm);                       // [n][BL_LINES + 1] then [nsol][n]
    const int P = BL_LINES + 1;
    double* sols = sm + (size_t)n * P;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = BL_THREADS / 32;
    const int64_t l0 = (int64_t)blockIdx.x * BL_LINES;
    const int nl = (lines - l0 < BL_LINES) ? (int)(lines - l0) : BL_LINES;
    for (int e = threadIdx.x; e < nsol * n; e += BL_THREADS) sols[e] = sol[e];
    for (int l = warp; l < nl; l += nw) {
        const double* __restrict__ src = in + (l0 + l) * n;
        if (npre > 0) {
            for (int j = lane; j < n; j += 32) {
                double acc = 0.0;
                for (int d = 0; d < npre && j + d < n; ++d) acc = fma(pre[(int64_t)d * n + j], src[j + d], acc);
                sm[j * P + l] = acc;
            }
        } else {
#pragma unroll 8
            for (int j = lane; j < n; j += 32) sm[j * P + l] = src[j];
        }
    }
    __syncthreads();
    if (nsol > 0 && warp == 0 && lane < nl) {
        double win[7] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        const int nd = nsol < 8 ? nsol : 8;
        for (int i = n - 1; i >= 0; --i) {
            double acc = sm[i * P + lane];
#pragma unroll
            for (int d = 1; d < 8; ++d)
                if (d < nd) acc = fma(-sols[d * n + i], win[d - 1], acc);
            for (int d = 8; d < nsol && i + d < n; ++d)          // wider bands: x_{i+8} .. are already stored in sm
                acc = fma(-sols[d * n + i], sm[(i + d) * P + lane], acc);
            const double xi = acc * sols[i];
#pragma unroll
            for (int d = 6; d > 0; --d) win[d] = win[d - 1];
            win[0] = xi;
            sm[i * P + lane] = xi;
        }
    }
    __syncthreads();
    for (int l = warp; l < nl; l += nw) {
        double* __restrict__ dst = out + (l0 + l) * n;
#pragma unroll 8
        for (int j = lane; j < n; j += 32) dst[j] = sm[j * P + l];
    }
}

// Parity-structured conversions (ultraspherical: only even diagonals) with one off-diagonal: the back-substitution
// x_i = r_i (t_i - u_i x_{i+2}) is two interleaved first-order linear recurrences, i.e. a suffix scan over the affine
// maps x -> A_i x + B_i.  One warp per line, lane l of round q owns the element pair (2m, 2m+1), m = 32 q + l, the
// scan runs on shuffles: no shared memory, no block barrier, every global access a coalesced 16-byte load / store.
__device__ __forceinline__ double shfl_down_d(double v, int off) { return __shfl_down_sync(0xffffffffu, v, off); }
__device__ __forceinline__ double shfl_idx_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

__global__ void __launch_bounds__(BL_THREADS)
k_band_scan2(const double* __restrict__ in, double* __restrict__ out, int64_t lines, int n,
             const double* __restrict__ pre, int npre, const double* __restrict__ sol)
{
    const int lane = threadIdx.x & 31;
    const int64_t line = (int64_t)blockIdx.x * (BL_THREADS / 32) + (threadIdx.x >> 5);
    if (line >= lines) return;
    const double* __restrict__ src = in + line * n;
    double* __restrict__ dst = out + line * n;
    const int rounds = (n + 63) / 64;
    double carry0 = 0.0, carry1 = 0.0;                      // x_{i+2} entering the round from above (even / odd chain)
    for (int q = rounds - 1; q >= 0; --q) {
        const int i0 = 2 * (32 * q + lane);
        // c_{i0 .. i0+3}: own pair + the next lane's pair (the last lane reads it from memory)
        double c0 = 0.0, c1 = 0.0;
        if (i0 + 1 < n) { const double2 v = *reinterpret_cast<const double2*>(src + i0); c0 = v.x; c1 = v.y; }
        else if (i0 < n) c0 = src[i0];
        double c2 = shfl_down_d(c0, 1), c3 = shfl_down_d(c1, 1);
        if (lane == 31) { c2 = (i0 + 2 < n) ? src[i0 + 2] : 0.0; c3 = (i0 + 3 < n) ? src[i0 + 3] : 0.0; }
        double t0 = c0, t1 = c1;
        if (npre > 0) {
            t0 = 0.0; t1 = 0.0;
            if (i0 < n) {
                t0 = pre[i0] * c0;
                if (npre > 1) t0 = fma(pre[n + i0], c1, t0);
                if (npre > 2) t0 = fma(pre[2 * n + i0], c2, t0);
            }
            if (i0 + 1 < n) {
                t1 = pre[i0 + 1] * c1;
                if (npre > 1) t1 = fma(pre[n + i0 + 1], c2, t1);
                if (npre > 2) t1 = fma(pre[2 * n + i0 + 1], c3, t1);
            }
        }
        // affine maps x_i = A x_{i+2} + B
        double A0 = 0.0, B0 = 0.0, A1 = 0.0, B1 = 0.0;
        if (i0 < n) { const double r = sol[i0]; B0 = r * t0; A0 = (i0 + 2 < n) ? -r * sol[n + i0] : 0.0; }
        if (i0 + 1 < n) { const double r = sol[i0 + 1]; B1 = r * t1; A1 = (i0 + 3 < n) ? -r * sol[n + i0 + 1] : 0.0; }
        // inclusive suffix scan over lanes: compose with the maps of higher lanes
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const double a0 = shfl_down_d(A0, off), b0 = shfl_down_d(B0, off);
            const double a1 = shfl_down_d(A1, off), b1 = shfl_down_d(B1, off);
            if (lane + off < 32) { B0 = fma(A0, b0, B0); A0 *= a0; B1 = fma(A1, b1, B1); A1 *= a1; }
        }
        const double x0 = fma(A0, carry0, B0), x1 = fma(A1, carry1, B1);
        if (i0 + 1 < n) *reinterpret_cast<double2*>(dst + i0) = make_double2(x0, x1);
        else if (i0 < n) dst[i0] = x0;
        carry0 = shfl_idx_d(x0, 0); carry1 = shfl_idx_d(x1, 0);
    }
}

extern "C" int db_band_lines(const double* in, double* out, int64_t lines, int32_t n,
                             const double* pre_diags, int32_t pre_ndiag, const double* solve_diags, int32_t solve_ndiag,
                             int32_t solve_stride, void* stream)
{
    if (lines <= 0 || n <= 0) return 0;
    if (solve_ndiag > 0 && solve_stride == 2) {
        // compact even-diagonal storage: only the two-diagonal (first-order) case has a kernel
        if (solve_ndiag != 2 || pre_ndiag > 3 || (n & 1) || ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15)) {
            db_set_error("band_lines: stride-2 solve needs 2 stored diagonals, <= 3 pre-apply diagonals, even n, 16-byte aligned lines");
            return 1;
        }
        const int64_t blocks = (lines + BL_THREADS / 32 - 1) / (BL_THREADS / 32);
        DB_LAUNCH(k_band_scan2, dim3((unsigned)blocks), dim3(BL_THREADS), 0, stream, in, out, lines, n, pre_diags, pre_ndiag, solve_diags);
        return db_check_launch("band_lines(scan)");
    }
    if (solve_ndiag > 0 && solve_stride != 1) { db_set_error("band_lines: unsupported diagonal stride %d", solve_stride); return 1; }
    size_t smem = ((size_t)n * (BL_LINES + 1) + (size_t)(solve_ndiag > 0 ? solve_ndiag : 0) * n) * sizeof(double);
    if (smem > (size_t)DB_MAX_SMEM) { db_set_error("band_lines: line length %d too large", n); return 1; }
    int64_t blocks = (lines + BL_LINES - 1) / BL_LINES;
#ifndef DB_EMU
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(k_band_lines, cudaFuncAttributeMaxDynamicSharedMemorySize, DB_MAX_SMEM); attr = true; }
#endif
    DB_LAUNCH(k_band_lines, dim3((unsigned)blocks), dim3(BL_THREADS), smem, stream, in, out, lines, n, pre_diags, pre_ndiag, solve_diags, solve_ndiag);
    return db_check_launch("band_lines");
}
