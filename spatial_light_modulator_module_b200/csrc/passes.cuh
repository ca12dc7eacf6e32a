// The pass kernels of the hologram loops (sm_100a).
//
// A 2-D transform is a row pass and a column pass.  Because the in-CTA line FFT returns every
// point to the thread that loaded it (fft_tile.cuh), two transforms that meet at a pointwise
// step are fused into ONE pass over HBM:
//
//   SLM-plane pass  (rows)    : finish ifft2  ->  phase-only projection (GS) / tangent-gradient
//                               update of x (GD)  ->  start fft2
//   Fourier-plane pass (cols) : finish fft2   ->  amplitude replacement + error sums (GS) /
//                               mask*F*(I-T) + error sum (GD)  ->  start ifft2
//
// so one GS iteration (algorithms.py:30-38) reads and writes the field twice instead of four
// times, and one GD iteration (algorithms.py:84-92) adds a read-only column pass for the global
// max that line 86 needs before the gradient can be formed.
#pragma once
#include "engine_types.h"
#include "fft_tile.cuh"
#include "tma.cuh"

namespace slm {

// ---- pointwise pieces ---------------------------------------------------------------------------
// exp(1j*angle(z)) as written at algorithms.py:30,33: z/|z|, with angle(+0)=0 -> 1, angle(-0)=pi -> -1
template <typename R> SLM_DEV cpx<R> unit_phasor(cpx<R> z) {
    const R m2 = cnorm2(z);
    if (m2 == (R)0) return mk<R>(copysign((R)1, z.x), (R)0);
    return cscale(z, rsqrt_fast(m2));
}
// unit_phasor of N register values.  Exact zeros are rare (symmetric targets at the first iterations), so the
// per-element special case -- a predicate, two selects and a constant move each, kept in bit masks by the
// compiler: a fifth of the GS row kernel's instructions -- is taken out of the common path: one min over the
// squared moduli decides between a plain z * rsqrt(|z|^2) loop and the careful one.
template <int N, typename R> SLM_DEV void unit_phasors(cpx<R>* v) {
    R m2[N];
    R mn;
#pragma unroll
    for (int r = 0; r < N; ++r) { m2[r] = cnorm2(v[r]); mn = r ? fmin(mn, m2[r]) : m2[r]; }
    if (mn > (R)0) {
#pragma unroll
        for (int r = 0; r < N; ++r) v[r] = cscale(v[r], rsqrt_fast(m2[r]));
    } else {
#pragma unroll
        for (int r = 0; r < N; ++r) v[r] = unit_phasor(v[r]);
    }
}

// dEdX_complex (algorithms.py:179-185) == (g - xh <xh, g>) / |x| with xh = x/|x|; returns the
// updated x (algorithms.py:91).
template <typename R> SLM_DEV cpx<R> tangent_step(cpx<R> x, cpx<R> g, R lr) {
    const R inv = rsqrt_fast(cnorm2(x));
    const cpx<R> xh = cscale(x, inv);
    const cpx<R> pr = pk_mul(xh, g);
    const R dot = pr.x + pr.y;
    const R step = -(lr * inv);
    const cpx<R> tang = pk_fma(mk<R>(-dot, -dot), xh, g);          // g - xh <xh, g>
    return pk_fma(mk<R>(step, step), tang, x);                     // x - lr * tang / |x|
}

// The Fourier-plane step of one point, shared by the kernels that iterate (row_fourier_kernel writes out its GD step).
// m2 = |C|^2 (GS) / |F|^2 (GD).
// GS error sums (algorithms.py:36-38), taken against the scale s0 of the previous iteration: u = s0 |C|^2, d = u - T;
// max |C|^2, sum d^2, sum d u, sum u^2.  The exact scale s = norm/max is folded in when the plane closes (gs_error).
// t may be a grey level (an integer): it is converted to R where d is formed.
template <typename R, typename T> SLM_DEV void gs_sums(R m2, T t, R s0r, R& mx, R& sa, R& sb, R& sc) {
    const R u = s0r * m2, d = u - (R)t;
    mx = fmax(mx, m2); sa += d * d; sb += d * u; sc += u * u;
}
// D = |amp| * exp(1j*angle(C)), algorithms.py:33
template <typename R> SLM_DEV void replace_amplitude(cpx<R>& v, R m2, R amp) {
    if (m2 == (R)0) v = mk<R>(copysign(amp, v.x), (R)0);
    else v = cscale(v, amp * rsqrt_fast(m2));
}
// GD output = |F|^2 * norm / max, algorithms.py:85-86.  fp32: gdk = (R)(norm / max), formed once per plane.
template <typename R> SLM_DEV R gd_output(R m2, R gdk, double norm, double imax) {
    if (sizeof(R) == 8) return (R)(((double)m2 * norm) / imax);
    return m2 * gdk;
}
// mask * med_output * (output - T), algorithms.py:88, and its error sum sum (output - T)^2, :92
template <typename R> SLM_DEV cpx<R> gd_point(cpx<R> v, R output, R t, R mask, R& sa) {
    const R d = output - t;
    sa += d * d;
    return cscale(cscale(v, mask), d);
}

// ---- deterministic reductions ---------------------------------------------------------------------
// FIELDS selects which members of Partial a kernel actually uses (bit 0 mx, 1 a, 2 b, 3 c) so the
// shuffle trees only move those.
enum { F_MX = 1, F_A = 2, F_B = 4, F_C = 8, F_ALL = 15 };
template <int FIELDS> SLM_DEV Partial combine(Partial p, Partial q) {
    if (FIELDS & F_MX) p.mx = fmax(p.mx, q.mx);
    if (FIELDS & F_A) p.a += q.a;
    if (FIELDS & F_B) p.b += q.b;
    if (FIELDS & F_C) p.c += q.c;
    return p;
}
template <int FIELDS> SLM_DEV Partial warp_reduce(Partial p) {
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        Partial q = p;
        if (FIELDS & F_MX) q.mx = shfl_xor(p.mx, m);
        if (FIELDS & F_A) q.a = shfl_xor(p.a, m);
        if (FIELDS & F_B) q.b = shfl_xor(p.b, m);
        if (FIELDS & F_C) q.c = shfl_xor(p.c, m);
        p = combine<FIELDS>(p, q);
    }
    return p;
}
// Result valid in thread 0.  NT = threads per CTA (multiple of 32).  OWNER: calls with different values use separate
// `red` arrays.  The weighted-GS kernels pass 1, so that they share no array with the other kernels: an array that one
// kernel alone uses is allocated with it, one that several use is a module variable, and that alone changed the
// registers the GS column kernel got.
template <int NT, int FIELDS, int OWNER = 0> SLM_DEV Partial block_reduce(Partial p, int t) {
    static_assert(NT % 32 == 0 && NT <= 1024, "CTA size");
    SLM_STATIC_SMEM Partial red[32];
    p = warp_reduce<FIELDS>(p);
    if (t % 32 == 0) red[t / 32] = p;
    sync_cta();
    if (t < 32) {
        Partial q; q.mx = 0; q.a = 0; q.b = 0; q.c = 0;
        if (t < NT / 32) q = red[t];
        p = warp_reduce<FIELDS>(q);
    }
    return p;
}
SLM_DEV Partial ld_partial(const Partial* p) {
    Partial q; q.mx = ld_cg(&p->mx); q.a = ld_cg(&p->a); q.b = ld_cg(&p->b); q.c = ld_cg(&p->c); return q;
}
// Split form used by the loop's column pass: thread 0 publishes right after the block reduce (the
// atomic's round trip overlaps the inverse transform) and warp 0 alone looks at the ticket afterwards.
SLM_DEV unsigned publish_partial(Partial mine, Partial* plane_partials, int tile, int tiles, unsigned* counter) {
    plane_partials[tile] = mine;
    fence_device();
    return atomic_inc_wrap(counter, (unsigned)tiles - 1);                        // wraps to 0: reusable
}
// warp 0, all 32 lanes: `ticket` is valid in lane 0.  True (with the plane total in every lane) for the last tile.
template <int FIELDS> SLM_DEV bool collect_if_last(unsigned ticket, int t, const Partial* plane_partials, int tiles, Partial& total) {
    ticket = shfl_idx(ticket, 0);
    if (ticket != (unsigned)tiles - 1) return false;
    fence_device();
    Partial q; q.mx = 0; q.a = 0; q.b = 0; q.c = 0;
    for (int i = t; i < tiles; i += 32) q = combine<FIELDS>(q, ld_partial(plane_partials + i));
    total = warp_reduce<FIELDS>(q);
    return true;
}
// warp 0 of a plane's last tile, after collect_if_last: the plane total of one more per-tile sum, in every lane
SLM_DEV double collect_sum(int t, const double* plane_partials, int tiles) {
    double q = 0;
    for (int i = t; i < tiles; i += 32) q += ld_cg(plane_partials + i);
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) q += shfl_xor(q, m);
    return q;
}

// ---- closing a plane's Fourier-plane pass ---------------------------------------------------------------
// The Partial fields the tiles reduce for a closing of kind KIND (PlaneClose)
SLM_HOSTDEV constexpr int close_fields(int kind) { return kind == CLOSE_GS ? F_ALL : (kind == CLOSE_GD ? F_A : F_MX); }
// GS error of an iteration from sums taken against the scale s0 of the previous one (a = sum d^2, b = sum d u,
// c = sum u^2 with u = s0 I, d = u - T): with the exact scale s, sum((s I - T)^2) / HW (algorithms.py:38,162)
SLM_DEV double gs_error(double a, double b, double c, double s, double s0, double hw) {
    const double dl = (s0 != 0.0) ? s / s0 - 1.0 : 0.0;
    return (a + 2.0 * dl * b + dl * dl * c) / hw;
}
// One thread closes plane `st` from the total of its tiles' sums: max and scale, and for an iteration the error, its
// entry in the plane's error curve `err_row`, the iteration count and the loop condition.  s0 / norm: the plane's
// scale and norm as read by the tiles, which computed in R.
template <typename R, int KIND>
SLM_DEV void close_plane(PlaneStats* st, const Partial& tot, double s0, double norm, double hw, double* err_row, double tolerance) {
    double err = 0;
    if constexpr (KIND == CLOSE_GD) {
        err = tot.a / hw;                                        // algorithms.py:92
    } else {
        const double s = norm / tot.mx;                          // algorithms.py:37
        if constexpr (KIND == CLOSE_GS) err = gs_error(tot.a, tot.b, tot.c, s, (double)(R)s0, hw);
        st->imax = tot.mx; st->scale = s;
    }
    if constexpr (KIND != CLOSE_MAX) {
        const int k = st->iters;
        err_row[k] = err;
        st->err = err; st->iters = k + 1;
        st->done = !(err > tolerance);                           // loop condition, algorithms.py:29,83
    }
}

// ---- geometry --------------------------------------------------------------------------------------
constexpr int floor_pow2(int v) { int p = 1; while (2 * p <= v) p *= 2; return p; }
constexpr int whole_warp_columns(int tc, int m) { while ((tc * m) % 32 != 0) tc *= 2; return tc; }
template <typename R, int L> struct RowGeom {
    using P = FftPlan<L>;
    static constexpr int M = P::M;
    static constexpr int NR = floor_pow2(256 / M);           // rows per CTA (power of two)
    static constexpr int THREADS = NR * M;
    static constexpr size_t SMEM = (size_t)NR * P::NP * sizeof(cpx<R>);
#ifndef SLM_ROW_THREADS_PER_SM
#define SLM_ROW_THREADS_PER_SM 768
#endif
    // fp32 register budget: 3 x 256 threads (<= 80 registers) for 16 points per thread, 512 threads
    // (<= 128 registers) for the 32-point long lines
    static constexpr int BUDGET = P::E == 32 ? 512 : SLM_ROW_THREADS_PER_SM;
    static constexpr int MIN_CTAS = sizeof(R) == 4 ? (BUDGET / THREADS > 0 ? BUDGET / THREADS : 1) : 1;
    // the multi-plane row pass holds the field sum S[E] beside the plane being transformed: 512 threads (<= 128
    // registers) in fp32
    static constexpr int MP_MIN_CTAS = sizeof(R) == 4 ? (512 / THREADS > 0 ? 512 / THREADS : 1) : 1;
    // rows are transformed independently: the threads of LPG rows (whole warps) share a named barrier
    static constexpr int LPG = M % 32 == 0 ? 1 : (M % 16 == 0 ? 2 : (M % 8 == 0 ? 4 : 8));
    static constexpr int GROUPS = NR / LPG;
    static constexpr int GROUP_THREADS = (NR % LPG == 0 && GROUPS > 1 && GROUPS <= 15) ? LPG * M : 0;   // 0: CTA barrier
    using Sync = GroupSync<GROUP_THREADS>;
};
template <typename R, int L> struct ColGeom {
    using P = ColPlan<L>;
    static constexpr int M = P::M;
#ifndef SLM_TCMAX_F32
#define SLM_TCMAX_F32 8
#endif
#ifndef SLM_TCMAX_F64
#define SLM_TCMAX_F64 4
#endif
    static constexpr int TMAX = sizeof(R) == 4 ? 512 : 256;
    static constexpr int TCMAX = sizeof(R) == 4 ? SLM_TCMAX_F32 : SLM_TCMAX_F64;
    static constexpr int TCRAW = (TMAX / M) < TCMAX ? (TMAX / M) : TCMAX;
    static constexpr int TC0 = TCRAW >= 8 ? 8 : TCRAW >= 4 ? 4 : TCRAW >= 2 ? 2 : 1;
    // columns per CTA: doubled until the CTA is whole warps (M = 144 or 240 points in fp64: 2 columns)
    static constexpr int TC = whole_warp_columns(TC0, M);
    static constexpr int THREADS = TC * M;
    static constexpr size_t SMEM = (size_t)TC * P::NP * sizeof(cpx<R>);
    static_assert(THREADS % 32 == 0, "column CTA must be whole warps");
};

// ---- SLM-plane pass ------------------------------------------------------------------------------
// FINAL = 1 is the pass after the loop: it emits the hologram (angle) instead of starting the next
// forward transform; a separate instantiation keeps the atan2 code out of the loop kernel.
template <typename R, int W, int ALG, int FINAL>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((RowGeom<R, W>::THREADS), (RowGeom<R, W>::MIN_CTAS)) row_pass_kernel(RowArgs a) {
    using G = RowGeom<R, W>;
    using P = FftPlan<W>;
    constexpr int E = P::E, M = P::M;
    SLM_DYN_SMEM(raw);
    const int t = threadIdx.x, rr = t / M, j = t % M;
    const long long grow = (long long)blockIdx.x * G::NR + rr;
    const int b = (int)(grow / a.H), y = (int)(grow % a.H);
    griddep_launch();                                 // the next pass may begin its prologue while this one drains
    griddep_wait();                                   // ... and this one starts only when its predecessor's data is complete
    const PlaneStats* st = a.stats + b;
    const int done = ld_cg(&st->done);
    if (!FINAL && done) return;                       // uniform: a CTA never straddles planes
    cpx<R>* line = reinterpret_cast<cpx<R>*>(raw) + (size_t)rr * P::NP;
    const typename G::Sync sync{1 + rr / G::LPG};
    const cpx<R>* tw = static_cast<const cpx<R>*>(a.tw);
    const size_t base = ((size_t)b * a.H + y) * W + j;
    const size_t ibase = (size_t)y * W + j;
    const R* inc = static_cast<const R*>(a.inc);
    cpx<R> v[E];

    if (ALG == ALG_GS) {
        if (a.source == ROW_FROM_Y) {
            const cpx<R>* Y = static_cast<const cpx<R>*>(a.Y) + base;
#pragma unroll
            for (int r = 0; r < E; ++r) v[r] = ld_plane(Y + r * M);
            line_fft<R, W, +1, 1>(v, line, j, tw, sync);           // A = ifft2(D) up to a positive scale
            if (!FINAL) unit_phasors<E>(v);
        } else if (a.source == ROW_FROM_A32) {
            // first phasor in complex64, as the reference computes it (algorithms.py:27,30; SURVEY A.1)
            const cpx<float>* A = static_cast<const cpx<float>*>(a.A32) + base;
#pragma unroll
            for (int r = 0; r < E; ++r) {
                cpx<float> z = ld_plane(A + r * M);
                if (!FINAL) z = unit_phasor(z);
                v[r].x = (R)z.x; v[r].y = (R)z.y;
            }
        } else {
            const cpx<R>* F = static_cast<const cpx<R>*>(a.field) + base;
#pragma unroll
            for (int r = 0; r < E; ++r) {
                v[r] = ld_plane(F + r * M);
                if (a.source == ROW_FROM_A && !FINAL) v[r] = unit_phasor(v[r]);
            }
        }
        if (FINAL) {                                   // hologram = angle(A), algorithms.py:48
            double* h = a.hologram + base;
#pragma unroll
            for (int r = 0; r < E; ++r) h[r * M] = atan2((double)v[r].y, (double)v[r].x);
            return;
        }
        if (inc && a.source != ROW_FROM_FIELD) {
#pragma unroll
            for (int r = 0; r < E; ++r) v[r] = cscale(v[r], ld_ro(inc + ibase + r * M));
        }
    } else {
        cpx<R>* xp = static_cast<cpx<R>*>(a.x) + base;
        cpx<R> xx[E];
#pragma unroll
        for (int r = 0; r < E; ++r) xx[r] = ld_plane(xp + r * M);
        if (a.source == ROW_FROM_Y) {
            const cpx<R>* Y = static_cast<const cpx<R>*>(a.Y) + base;
#pragma unroll
            for (int r = 0; r < E; ++r) v[r] = ld_plane(Y + r * M);
            line_fft<R, W, +1, 1>(v, line, j, tw, sync);
            // the update of the iteration whose Fourier-plane pass produced Y: lr of THAT iteration
            const R lr = (R)ld_ro(a.lr + (ld_cg(&st->iters) - 1));
            const R nrm = (R)a.inv_hw;
#pragma unroll
            for (int r = 0; r < E; ++r) {
                R gs = nrm;                                     // dEdF = ifft2(...) * inc_amp, algorithms.py:87-89
                if (inc) gs *= ld_ro(inc + ibase + r * M);
                xx[r] = tangent_step(xx[r], cscale(v[r], gs), lr);   // algorithms.py:90-91
                st_plane(xp + r * M, xx[r]);
            }
        }
        if (FINAL) {                                   // hologram = angle(input), algorithms.py:111
            double* h = a.hologram + base;
#pragma unroll
            for (int r = 0; r < E; ++r) h[r * M] = atan2((double)xx[r].y, (double)xx[r].x);
            return;
        }
#pragma unroll
        for (int r = 0; r < E; ++r) {                            // input / abs(input) * inc_amp, algorithms.py:84
            R inv = rsqrt_fast(cnorm2(xx[r]));
            if (inc) inv *= ld_ro(inc + ibase + r * M);
            v[r] = cscale(xx[r], inv);
        }
    }
    line_fft<R, W, -1, 1>(v, line, j, tw, sync);
    cpx<R>* X = static_cast<cpx<R>*>(a.X) + base;
#pragma unroll
    for (int r = 0; r < E; ++r) st_plane(X + r * M, v[r]);
}

// ---- multi-plane SLM-plane pass ------------------------------------------------------------------
// Multi-plane GS (Haist et al., Opt. Commun. 140, 299 (1997)): K target planes at defocus L_k = exp(i alpha_k rho^2)
// share one hologram.  Their Fourier-plane steps are K planes of GS's column pass; this pass joins them.  A CTA takes
// NR rows of hologram g and, plane by plane (b = g K + k), finishes the inverse transform, takes off the defocus and
// adds the field into S[E]:  S = sum_k ifft2(D_k) conj(L_k).  Then B = inc exp(i angle(S)), and per plane the rows of
// B L_k are forward-transformed into X.  FINAL = 1 writes angle(S) to the hologram instead.
// Other sources: ROW_FROM_A32 / ROW_FROM_A sum the setup's A_k (already transformed) the same way; ROW_FROM_FIELD
// takes B of iteration 0 from `field` (one plane per hologram).
// K = 1 with alpha = 0 is GS's arithmetic: S starts from the first term (not 0 + term), a plane without defocus is not
// multiplied, and the phasor and `inc` are applied as row_pass_kernel applies them.
// Loop condition: each plane's column pass closes with its own `done`; a hologram iterates while any of its planes
// has not converged.  All flags set: return; otherwise every CTA of the hologram clears them (all CTAs decide alike,
// in any order: a flag that was clear stays clear), so the planes keep iterating together and their curves stay
// equal in length.
//
// ALG = ALG_MPGD is multi-plane GD: the planes' Fourier-plane steps are K planes of GD's column pass, and the pass
// takes the gradient of the mean of their errors.  From Y: S = sum_k ifft2(G_k) conj(L_k) as above, then x is loaded
// (into the registers the plane's transform has freed) and takes row_pass_kernel<ALG_GD>'s step with dEdF = S inc /
// (K H W) (ra.inv_hw = 1 / (K H W)) and lr[iters - 1]; ROW_FROM_FIELD takes x as given (iteration 0).  Then B =
// x rsqrt(|x|^2) inc, forward-transformed per plane as above; FINAL = 1 writes angle(x) instead.  The FINAL pass does
// not test the flags: it applies the update of the last iteration that ran, once, as row_pass_kernel<ALG_GD> does.
// K = 1 with alpha = 0 is row_pass_kernel<ALG_GD>'s arithmetic; the engine runs that case with row_pass_kernel itself
// (slm_gd_multiplane_run).
template <typename R, int W, int ALG, int FINAL>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((RowGeom<R, W>::THREADS), (RowGeom<R, W>::MP_MIN_CTAS)) row_multiplane_kernel(RowArgs a) {
    using G = RowGeom<R, W>;
    using P = FftPlan<W>;
    constexpr int E = P::E, M = P::M;
    SLM_DYN_SMEM(raw);
    const int t = threadIdx.x, rr = t / M, j = t % M;
    const long long grow = (long long)blockIdx.x * G::NR + rr;
    const int g = (int)(grow / a.H), y = (int)(grow % a.H);
    const int K = a.planes;
    griddep_launch();
    griddep_wait();
    if (!FINAL) {
        // (the PlaneStats of the context, handed over as const for the single-plane passes)
        PlaneStats* st = const_cast<PlaneStats*>(a.stats) + (size_t)g * K;
        bool all = true;
        for (int k = 0; k < K; ++k) all = all && ld_cg(&st[k].done) != 0;
        if (all) return;                              // uniform: a CTA never straddles holograms
        if (t == 0)
            for (int k = 0; k < K; ++k) st[k].done = 0;
    }
    cpx<R>* line = reinterpret_cast<cpx<R>*>(raw) + (size_t)rr * P::NP;
    const typename G::Sync sync{1 + rr / G::LPG};
    const cpx<R>* tw = static_cast<const cpx<R>*>(a.tw);
    const cpx<R>* ly = static_cast<const cpx<R>*>(a.lens_y);
    const cpx<R>* lx = static_cast<const cpx<R>*>(a.lens_x) + j;
    const size_t plane = (size_t)a.H * W, pix = (size_t)y * W + j;
    const size_t gbase = (size_t)g * plane + pix;                   // one plane per hologram (field, hologram)
    const size_t kbase = (size_t)g * K * plane + pix;               // plane 0 of the hologram's K planes
    const R* inc = static_cast<const R*>(a.inc);
    cpx<R> s[E], v[E];

    if constexpr (ALG == ALG_MPGD) {
        cpx<R>* xp = static_cast<cpx<R>*>(a.x) + gbase;
        if (a.source == ROW_FROM_Y) {
            for (int k = 0; k < K; ++k) {
                const cpx<R>* Y = static_cast<const cpx<R>*>(a.Y) + kbase + (size_t)k * plane;
#pragma unroll
                for (int r = 0; r < E; ++r) v[r] = ld_plane(Y + r * M);
                line_fft<R, W, +1, 1>(v, line, j, tw, sync);
                if (a.lens_mask & (1 << k)) {
                    const cpx<R> cy = ld_const(ly + (size_t)k * a.H + y);
#pragma unroll
                    for (int r = 0; r < E; ++r) v[r] = cmul(v[r], cconj(cmul(cy, ld_const(lx + (size_t)k * W + r * M))));
                }
#pragma unroll
                for (int r = 0; r < E; ++r) s[r] = k ? cadd(s[r], v[r]) : v[r];
            }
            // the update of the iteration whose Fourier-plane passes produced Y: lr of THAT iteration (the K planes of
            // a hologram count alike)
            const R lr = (R)ld_ro(a.lr + (ld_cg(&a.stats[(size_t)g * K].iters) - 1));
            const R nrm = (R)a.inv_hw;
#pragma unroll
            for (int r = 0; r < E; ++r) v[r] = ld_plane(xp + r * M);
#pragma unroll
            for (int r = 0; r < E; ++r) {
                R gs = nrm;
                if (inc) gs *= ld_ro(inc + pix + r * M);
                v[r] = tangent_step(v[r], cscale(s[r], gs), lr);
                st_plane(xp + r * M, v[r]);
            }
        } else {
#pragma unroll
            for (int r = 0; r < E; ++r) v[r] = ld_plane(xp + r * M);
        }
        if (FINAL) {                                   // hologram = angle(x)
            double* h = a.hologram + gbase;
#pragma unroll
            for (int r = 0; r < E; ++r) h[r * M] = atan2((double)v[r].y, (double)v[r].x);
            return;
        }
#pragma unroll
        for (int r = 0; r < E; ++r) {                  // B = x / |x| inc
            R inv = rsqrt_fast(cnorm2(v[r]));
            if (inc) inv *= ld_ro(inc + pix + r * M);
            s[r] = cscale(v[r], inv);
        }
    } else if (a.source == ROW_FROM_FIELD) {
        const cpx<R>* F = static_cast<const cpx<R>*>(a.field) + gbase;
#pragma unroll
        for (int r = 0; r < E; ++r) s[r] = ld_plane(F + r * M);
    } else if (a.source == ROW_FROM_A32 && K == 1 && !(a.lens_mask & 1)) {
        // GS's first phasor, in complex64 (row_pass_kernel)
        const cpx<float>* A = static_cast<const cpx<float>*>(a.A32) + kbase;
#pragma unroll
        for (int r = 0; r < E; ++r) {
            cpx<float> z = ld_plane(A + r * M);
            if (!FINAL) z = unit_phasor(z);
            s[r].x = (R)z.x; s[r].y = (R)z.y;
        }
    } else {
        for (int k = 0; k < K; ++k) {
            const size_t off = kbase + (size_t)k * plane;
            if (a.source == ROW_FROM_Y) {
                const cpx<R>* Y = static_cast<const cpx<R>*>(a.Y) + off;
#pragma unroll
                for (int r = 0; r < E; ++r) v[r] = ld_plane(Y + r * M);
                line_fft<R, W, +1, 1>(v, line, j, tw, sync);       // A_k = ifft2(D_k) up to a positive scale
            } else if (a.source == ROW_FROM_A32) {
                const cpx<float>* A = static_cast<const cpx<float>*>(a.A32) + off;
#pragma unroll
                for (int r = 0; r < E; ++r) { const cpx<float> z = ld_plane(A + r * M); v[r].x = (R)z.x; v[r].y = (R)z.y; }
            } else {
                const cpx<R>* A = static_cast<const cpx<R>*>(a.field) + off;
#pragma unroll
                for (int r = 0; r < E; ++r) v[r] = ld_plane(A + r * M);
            }
            if (a.lens_mask & (1 << k)) {
                const cpx<R> cy = ld_const(ly + (size_t)k * a.H + y);
#pragma unroll
                for (int r = 0; r < E; ++r) v[r] = cmul(v[r], cconj(cmul(cy, ld_const(lx + (size_t)k * W + r * M))));
            }
#pragma unroll
            for (int r = 0; r < E; ++r) s[r] = k ? cadd(s[r], v[r]) : v[r];
        }
        if (!FINAL) {
            if (a.source == ROW_FROM_Y) unit_phasors<E>(s);
            else {
#pragma unroll
                for (int r = 0; r < E; ++r) s[r] = unit_phasor(s[r]);
            }
        }
    }
    if (FINAL) {                                       // hologram = angle(S) (GD has returned above)
        double* h = a.hologram + gbase;
#pragma unroll
        for (int r = 0; r < E; ++r) h[r * M] = atan2((double)s[r].y, (double)s[r].x);
        return;
    }
    if (ALG == ALG_MP && inc && a.source != ROW_FROM_FIELD) {
#pragma unroll
        for (int r = 0; r < E; ++r) s[r] = cscale(s[r], ld_ro(inc + pix + r * M));
    }
    for (int k = 0; k < K; ++k) {                      // X_k = rows of fft2(B L_k)
#pragma unroll
        for (int r = 0; r < E; ++r) v[r] = s[r];
        if (a.lens_mask & (1 << k)) {
            const cpx<R> cy = ld_const(ly + (size_t)k * a.H + y);
#pragma unroll
            for (int r = 0; r < E; ++r) v[r] = cmul(v[r], cmul(cy, ld_const(lx + (size_t)k * W + r * M)));
        }
        line_fft<R, W, -1, 1>(v, line, j, tw, sync);
        cpx<R>* X = static_cast<cpx<R>*>(a.X) + kbase + (size_t)k * plane;
#pragma unroll
        for (int r = 0; r < E; ++r) st_plane(X + r * M, v[r]);
    }
}

// ---- Fourier-plane pass ---------------------------------------------------------------------------
// One column tile of the loop's Fourier-plane step.  v = the tile's points (thread (j,c) holds rows
// j + r*M of column c); lut_s = the 256-entry amplitude (GS) / weight (GD) table in shared memory.
// Ordering is chosen so no warp waits on a dependent global access: the grey levels are requested
// before the forward transform and only looked up (in shared memory) after it; the tile's partial
// sums are published before the inverse transform, whose work covers the atomic's round trip.
//
// ALG_GSW is GS with per-pixel weights w on the amplitude (weighted GS, Di Leonardo, Ianni & Ruocco, Opt. Express 15,
// 1913 (2007)): on the signal set {T > 0} where |C|^2 > 0, w_k = clamp(w_{k-1} amp / sqrt(sigma |C|^2), 1/c, c) with
// sigma = S_T / P_{k-1} (P: the signal set's sum of |C|^2 of the previous pass -- of this one at iteration 0, from the
// pre-pass), and D = (amp w) C/|C|.  Scale, error and loop condition are GS's.  amp * w is formed first, so with c = 1
// (w == 1.0 exactly) the arithmetic is GS's, bit for bit.
template <typename R, int H, int ALG>
SLM_DEV void col_pass_tile(const ColArgs& a, int b, int tile, int tiles, cpx<R>* v, cpx<R>* line, const R* lut_s,
                           int t, int c, int j) {
    using G = ColGeom<R, H>;
    using P = ColPlan<H>;
    constexpr int E = P::E, M = P::M, TC = G::TC;
    constexpr bool GSW = ALG == ALG_GSW;
    PlaneStats* st = a.stats + b;
    const size_t W = a.W;
    const size_t off = (size_t)b * H * W + (size_t)j * W + tile * TC + c;
    const cpx<R>* tw = static_cast<const cpx<R>*>(a.tw);
    const double s0 = ld_cg(&st->scale), imax = ld_cg(&st->imax), norm = ld_ro(a.norm + b);
    int grey[E];
    R tv[E], aux[E];
    if (a.T8) {
        const uint8_t* T = a.T8 + off;
#pragma unroll
        for (int r = 0; r < E; ++r) grey[r] = ld_ro(T + (size_t)r * M * W);
    } else {
        const R* T = static_cast<const R*>(a.Treal) + off;
        const R* Q = static_cast<const R*>(a.plane2) + off;
#pragma unroll
        for (int r = 0; r < E; ++r) { tv[r] = ld_ro(T + (size_t)r * M * W); aux[r] = ld_ro(Q + (size_t)r * M * W); }
    }
    if (!a.skip_forward) line_fft<R, H, -1, TC, CtaSync, false, column_points(H)>(v, line, j, tw);   // C = fft2(B)  /  med_output
    if (a.T8) {
#pragma unroll
        for (int r = 0; r < E; ++r) { tv[r] = (R)grey[r]; aux[r] = lut_s[grey[r]]; }
    }

    // per-thread sums in R (E terms), widened to double before they meet other threads
    R mx = 0, sa = 0, sb = 0, sc = 0;
    R sp = 0;                                                   // GSW: P, the signal set's sum of |C|^2
    const R s0r = (R)s0;                                        // GS: scale of the previous iteration
    const R gdk = sizeof(R) == 8 ? (R)0 : (R)(norm / imax);    // GD fp32: output = |F|^2 * (norm/max)
    const R sig = GSW ? (R)(ld_ro(a.target_sum + b) / ld_cg(a.signal_sum + b)) : (R)0;   // sigma_k = S_T / P_{k-1}
    const R wlo = GSW ? (R)(1.0 / a.weight_limit) : (R)0, whi = GSW ? (R)a.weight_limit : (R)0;
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const R m2 = cnorm2(v[r]);
        if (ALG == ALG_GS || GSW) {
            gs_sums(m2, tv[r], s0r, mx, sa, sb, sc);
            R amp = aux[r];
            if (GSW) {
                // the weights are read here, after the forward transform, not before it like the target: held through
                // the transform they would not fit in registers at the long lines
                R* const wp = static_cast<R*>(a.weights) + off + (size_t)r * M * W;
                R w = ld_cg(wp);
                if (tv[r] > (R)0) {
                    sp += m2;
                    if (m2 > (R)0) w = fmin(fmax(w * aux[r] * rsqrt_fast(sig * m2), wlo), whi);
                }
                st_cg(wp, w);
                amp = aux[r] * w;
            }
            replace_amplitude(v[r], m2, amp);
        } else {
            v[r] = gd_point(v[r], gd_output(m2, gdk, norm, imax), tv[r], aux[r], sa);
        }
    }
    constexpr int KIND = ALG == ALG_GD ? CLOSE_GD : CLOSE_GS, FIELDS = close_fields(KIND);
    Partial p; p.mx = (double)mx; p.a = (double)sa; p.b = (double)sb; p.c = (double)sc;
    p = block_reduce<G::THREADS, FIELDS, GSW ? 1 : 0>(p, t);
    double* sig_partials = GSW ? a.signal_partial + (size_t)b * tiles : nullptr;
    if (GSW) {
        Partial q; q.mx = 0; q.a = 0; q.b = (double)sp; q.c = 0;
        q = block_reduce<G::THREADS, F_B, 1>(q, t);           // (F_B: shared memory of its own, apart from the reduce above)
        if (t == 0) sig_partials[tile] = q.b;                   // published by the fence in publish_partial
    }
    Partial* plane_partials = a.partial + (size_t)b * tiles;
    unsigned ticket = 0;
    if (t == 0) ticket = publish_partial(p, plane_partials, tile, tiles, a.counter + b);

    line_fft<R, H, +1, TC, CtaSync, false, column_points(H)>(v, line, j, tw);
    cpx<R>* Y = static_cast<cpx<R>*>(a.Y) + off;
#pragma unroll
    for (int r = 0; r < E; ++r) st_plane(Y + (size_t)r * M * W, v[r]);

    if (t >= 32) return;
    Partial tot;
    if (!collect_if_last<FIELDS>(ticket, t, plane_partials, tiles, tot)) return;
    if (GSW) {
        const double psum = collect_sum(t, sig_partials, tiles);
        if (t == 0) a.signal_sum[b] = psum;
    }
    if (t == 0) close_plane<R, KIND>(st, tot, s0, norm, (double)H * (double)W, a.err_curve + (size_t)b * a.max_loops, a.tolerance);
}

// One column tile of a plain transform: complex out, max-only, or normalised intensity out.
template <typename R, int H>
SLM_DEV void col_plain_tile(const PlainColArgs& a, int b, int tile, int tiles, cpx<R>* v, cpx<R>* line, int t, int c, int j) {
    using G = ColGeom<R, H>;
    using P = ColPlan<H>;
    constexpr int E = P::E, M = P::M, TC = G::TC;
    PlaneStats* st = a.stats ? a.stats + b : nullptr;
    const size_t W = a.W;
    const size_t off = (size_t)b * H * W + (size_t)j * W + tile * TC + c;
    const cpx<R>* tw = static_cast<const cpx<R>*>(a.tw);
    if (!a.skip_fft) {
        if (a.inverse) line_fft<R, H, +1, TC, CtaSync, false, column_points(H)>(v, line, j, tw);
        else line_fft<R, H, -1, TC, CtaSync, false, column_points(H)>(v, line, j, tw);
    }

    if (a.output == OUT_COMPLEX) {
        cpx<R>* out = static_cast<cpx<R>*>(a.out) + off;
        const R s = (R)a.scale;
#pragma unroll
        for (int r = 0; r < E; ++r) st_plane(out + (size_t)r * M * W, cscale(v[r], s));
    } else if (a.output == OUT_STATS) {
        if (a.keep) {                                               // the transformed field goes back (in place)
            cpx<R>* out = static_cast<cpx<R>*>(a.out) + off;
#pragma unroll
            for (int r = 0; r < E; ++r) st_plane(out + (size_t)r * M * W, v[r]);
        }
        Partial p; p.mx = 0; p.a = 0; p.b = 0; p.c = 0;
        R mx = 0;
#pragma unroll
        for (int r = 0; r < E; ++r) mx = fmax(mx, cnorm2(v[r]));
        p.mx = (double)mx;
        constexpr int FIELDS = close_fields(CLOSE_MAX);
        p = block_reduce<G::THREADS, FIELDS>(p, t);
        if (t >= 32) return;
        Partial* plane_partials = a.partial + (size_t)b * tiles;
        unsigned ticket = 0;
        if (t == 0) ticket = publish_partial(p, plane_partials, tile, tiles, a.counter + b);
        Partial tot;
        if (!collect_if_last<FIELDS>(ticket, t, plane_partials, tiles, tot)) return;
        if (t == 0) close_plane<R, CLOSE_MAX>(st, tot, 0.0, ld_ro(a.norm + b), 0.0, nullptr, 0.0);
    } else {
        double* out = static_cast<double*>(a.out) + off;
        const double imax = ld_cg(&st->imax), scale = ld_cg(&st->scale), norm = ld_ro(a.norm + b);
#pragma unroll
        for (int r = 0; r < E; ++r) {
            const double m2 = (double)cnorm2(v[r]);
            double I;
            if (a.output == OUT_INTENSITY_GS) I = m2 * scale;
            else if (a.output == OUT_INTENSITY_GD) I = (m2 * norm) / imax;
            else I = (m2 / imax) * norm;
            out[(size_t)r * M * W] = I;
        }
    }
}

// One CTA per column tile: points straight from global memory (64-byte row segments), CTA-wide barriers.
// Used where the warp-specialised kernel (col_groups.cuh) does not apply: intensity outputs, the
// complex64 setup inside an fp64 context, line lengths whose tile rows are not 32 or 64 bytes.
template <typename R, int H, class Skip, class Body>
SLM_DEV void col_tiles(const void* in, int W, unsigned char* raw, Skip skip, Body body) {
    using G = ColGeom<R, H>;
    using P = ColPlan<H>;
    constexpr int E = P::E, M = P::M, TC = G::TC;
    const int tiles = W / TC;
    const int t = threadIdx.x, c = t % TC, j = t / TC;
    cpx<R> v[E];
    const int b = blockIdx.x / tiles, tile = blockIdx.x % tiles;
    if (skip(b)) return;
    const cpx<R>* X = static_cast<const cpx<R>*>(in) + (size_t)b * H * W + (size_t)j * W + tile * TC + c;
#pragma unroll
    for (int r = 0; r < E; ++r) v[r] = ld_plane(X + (size_t)r * M * W);
    body(b, tile, tiles, v, reinterpret_cast<cpx<R>*>(raw) + c, t, c, j);
}

template <typename R, int H, int ALG>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((ColGeom<R, H>::THREADS), 1) col_pass_kernel(ColArgs a) {
    SLM_DYN_SMEM(raw);
    SLM_STATIC_SMEM R lut_s[256];
    if (a.T8) {                                                 // visible after the first barrier of the transform
        const R* lut = static_cast<const R*>(a.lut);
        for (int i = threadIdx.x; i < 256; i += ColGeom<R, H>::THREADS) lut_s[i] = ld_ro(lut + i);
    }
    if (a.skip_forward) sync_cta();                             // no forward transform whose barriers would publish the table
    col_tiles<R, H>(a.X, a.W, raw,
        [&](int b) { return ld_cg(&a.stats[b].done) != 0; },
        [&](int b, int tile, int tiles, cpx<R>* v, cpx<R>* line, int t, int c, int j) {
            col_pass_tile<R, H, ALG>(a, b, tile, tiles, v, line, lut_s, t, c, j);
        });
}

// Weighted GS, iteration 0: the forward transform's max |C|^2 -> stats (as col_plain_tile's OUT_STATS takes it, so the
// scale is GS's) and the signal set's sum P_0 of |C|^2 -> signal_sum, for sigma_0 = S_T / P_0 of the first ALG_GSW pass.
template <typename R, int H>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((ColGeom<R, H>::THREADS), 1) col_gsw_stats_kernel(ColArgs a) {
    SLM_DYN_SMEM(raw);
    col_tiles<R, H>(a.X, a.W, raw,
        [&](int b) { return ld_cg(&a.stats[b].done) != 0; },
        [&](int b, int tile, int tiles, cpx<R>* v, cpx<R>* line, int t, int c, int j) {
            using G = ColGeom<R, H>;
            using P = ColPlan<H>;
            constexpr int E = P::E, M = P::M, TC = G::TC;
            const size_t W = a.W;
            const size_t off = (size_t)b * H * W + (size_t)j * W + tile * TC + c;
            bool sig[E];                                                // the point lies in the signal set {T > 0}
            if (a.T8) {
#pragma unroll
                for (int r = 0; r < E; ++r) sig[r] = ld_ro(a.T8 + off + (size_t)r * M * W) != 0;
            } else {
                const R* T = static_cast<const R*>(a.Treal) + off;
#pragma unroll
                for (int r = 0; r < E; ++r) sig[r] = ld_ro(T + (size_t)r * M * W) > (R)0;
            }
            line_fft<R, H, -1, TC, CtaSync, false, column_points(H)>(v, line, j, static_cast<const cpx<R>*>(a.tw));
            R mx = 0, sp = 0;
#pragma unroll
            for (int r = 0; r < E; ++r) {
                const R m2 = cnorm2(v[r]);
                mx = fmax(mx, m2);
                if (sig[r]) sp += m2;
            }
            constexpr int FIELDS = close_fields(CLOSE_MAX);
            Partial p; p.mx = (double)mx; p.a = 0; p.b = 0; p.c = 0;
            p = block_reduce<G::THREADS, FIELDS, 1>(p, t);
            Partial q; q.mx = 0; q.a = 0; q.b = (double)sp; q.c = 0;
            q = block_reduce<G::THREADS, F_B, 1>(q, t);
            if (t >= 32) return;
            Partial* plane_partials = a.partial + (size_t)b * tiles;
            double* sig_partials = a.signal_partial + (size_t)b * tiles;
            unsigned ticket = 0;
            if (t == 0) {
                sig_partials[tile] = q.b;
                ticket = publish_partial(p, plane_partials, tile, tiles, a.counter + b);
            }
            Partial tot;
            if (!collect_if_last<FIELDS>(ticket, t, plane_partials, tiles, tot)) return;
            const double psum = collect_sum(t, sig_partials, tiles);
            if (t == 0) {
                close_plane<R, CLOSE_MAX>(a.stats + b, tot, 0.0, ld_ro(a.norm + b), 0.0, nullptr, 0.0);
                a.signal_sum[b] = psum;
            }
        });
}

// Element n of local line `row` in the slab-exchange layout of block width wb (rows = lines per rank):
// block n / wb holds [rows][wb], i.e. what one peer sends or receives in the all-to-all (slab.cuh).
SLM_DEV size_t line_offset(int wb, int rows, int W, long long row, int n) {
    if (wb == 0) return (size_t)row * W + n;
    return (size_t)(n / wb) * ((size_t)rows * wb) + (size_t)row * wb + (n % wb);
}

// The same for the E points j + r*M (r < E) one thread of the slab path's Fourier-plane kernel holds, without a
// division per point: a block is a whole power-of-two number q of M-element runs (the host checks this:
// slm_rows_fourier_pass), so point r lies in block r / q at run r % q; 32-bit element offsets (one slab has
// fewer than 2^32 elements).  With the general div / mod form inlined at each of its ~100 uses the 16384-point
// kernel was 9000 instructions and its warps waited for instruction fetches (ncu: no_instruction 38 %);
// 3.8 -> 3.1 ms per pass, 136 -> 145 iterations/s on one GPU (same box, two runs each).
struct LineLayout { int lq, qmask; unsigned block_stride, base; };
template <int M> SLM_DEV LineLayout line_layout(int wb, int rows, int W, long long row, int j) {
    LineLayout L; L.lq = 31; L.qmask = -1; L.block_stride = 0;
    L.base = (unsigned)(row * W + j);                               // wb == 0: plain [row][W]  (planes of < 2^32 elements)
    if (wb != 0) {
        const int q = wb / M;
        int lq = 0;
        while ((1 << lq) < q) ++lq;
        L.lq = lq; L.qmask = q - 1; L.block_stride = (unsigned)rows * (unsigned)wb; L.base = (unsigned)(row * wb + j);
    }
    return L;
}
template <int M> SLM_DEV unsigned line_off(const LineLayout& L, int r) {
    return (unsigned)(r >> L.lq) * L.block_stride + L.base + (unsigned)(r & L.qmask) * M;
}
// f(r, offset of point r) for r < E with the block size q = 2^LQ a compile-time number, so that a thread's points are
// (a few block bases) + immediates -- like the plain layout's.  With the run-time form above the 32 offsets of a thread
// were formed once, kept from its loads to its stores and spilled (16384-point lines: 128 registers, one 512-thread CTA
// per SM and a small L1 beside 135 KB of shared memory -- every spill an exposed round trip to L2).
template <int E, int M, int LQ, class F> SLM_DEV void each_point_lq(const LineLayout& L, F f) {
#pragma unroll
    for (int r = 0; r < E; ++r) f(r, (unsigned)(r >> LQ) * L.block_stride + L.base + (unsigned)((r & ((1 << LQ) - 1)) * M));
}
template <int E, int M, class F> SLM_DEV void each_point(const LineLayout& L, F f) {
    constexpr int LE = E >= 32 ? 5 : (E >= 16 ? 4 : 3);               // log2(E): one block holds the whole line (and the plain layout)
    switch (L.lq) {
        case 0: each_point_lq<E, M, 0>(L, f); break;
        case 1: each_point_lq<E, M, 1>(L, f); break;
        case 2: each_point_lq<E, M, 2>(L, f); break;
        case 3: each_point_lq<E, M, (3 < LE ? 3 : LE)>(L, f); break;
        case 4: each_point_lq<E, M, (4 < LE ? 4 : LE)>(L, f); break;
        default: each_point_lq<E, M, LE>(L, f); break;
    }
}

// ---- plain row transform (setup, preview, slm_fft2) --------------------------------------------------
template <typename R, int W>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((RowGeom<R, W>::THREADS), 1) row_plain_kernel(PlainRowArgs a) {
    using G = RowGeom<R, W>;
    using P = FftPlan<W>;
    constexpr int E = P::E, M = P::M;
    SLM_DYN_SMEM(raw);
    const int t = threadIdx.x, rr = t / M, j = t % M;
    const long long grow = (long long)blockIdx.x * G::NR + rr;
    cpx<R>* line = reinterpret_cast<cpx<R>*>(raw) + (size_t)rr * P::NP;
    const typename G::Sync sync{1 + rr / G::LPG};
    const cpx<R>* tw = static_cast<const cpx<R>*>(a.tw);
    const long long total_rows = (long long)a.B * a.H;
    cpx<R> v[E];
    if (a.input == IN_COMPLEX) {
        const cpx<R>* in = static_cast<const cpx<R>*>(a.in);
#pragma unroll
        for (int r = 0; r < E; ++r) v[r] = ld_plane(in + line_offset(a.block_in, (int)total_rows, W, grow, j + r * M));
    } else if (a.input == IN_LUT_U8) {
        const R* lut = static_cast<const R*>(a.lut);
#pragma unroll
        for (int r = 0; r < E; ++r) { v[r].x = ld_ro(lut + ld_ro(a.T8 + line_offset(a.block_in, (int)total_rows, W, grow, j + r * M))); v[r].y = 0; }
    } else if (a.input == IN_REAL) {
        const R* in = static_cast<const R*>(a.in);
#pragma unroll
        for (int r = 0; r < E; ++r) { v[r].x = ld_ro(in + line_offset(a.block_in, (int)total_rows, W, grow, j + r * M)); v[r].y = 0; }
    } else {
        const double* in = static_cast<const double*>(a.in);
#pragma unroll
        for (int r = 0; r < E; ++r) { const double h = ld_ro(in + line_offset(a.block_in, (int)total_rows, W, grow, j + r * M)); v[r].x = (R)cos(h); v[r].y = (R)sin(h); }
    }
    if (a.inverse) line_fft<R, W, +1, 1>(v, line, j, tw, sync);
    else line_fft<R, W, -1, 1>(v, line, j, tw, sync);
    cpx<R>* out = static_cast<cpx<R>*>(a.out);
#pragma unroll
    for (int r = 0; r < E; ++r) st_plane(out + line_offset(a.block_out, (int)total_rows, W, grow, j + r * M), v[r]);
}

// ---- GS Fourier-plane step on the rows of a transposed slab (slab-decomposed transform) ------------------
// Same arithmetic as col_pass_tile<GS>; a line here is one COLUMN of the global plane, held by this rank
// after the all-to-all.  Per-line partial sums go to `partial`; the ranks' totals are combined by the
// caller (NCCL all-reduce), which also closes the iteration (scale, error).
template <typename R, int W, int MODE>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((RowGeom<R, W>::THREADS), (RowGeom<R, W>::MIN_CTAS)) row_fourier_kernel(RowFourierArgs a) {
    using G = RowGeom<R, W>;
    using P = FftPlan<W>;
    constexpr int E = P::E, M = P::M;
    constexpr bool HAS_T = MODE != RF_GD_MAX;                 // needs the target's grey levels and a table
    SLM_DYN_SMEM(raw);
    const int t = threadIdx.x, rr = t / M, j = t % M;
    const long long row = (long long)blockIdx.x * G::NR + rr;
    cpx<R>* line = reinterpret_cast<cpx<R>*>(raw) + (size_t)rr * P::NP;
    const typename G::Sync sync{1 + rr / G::LPG};
    const cpx<R>* tw = static_cast<const cpx<R>*>(a.tw);
    const cpx<R>* in = static_cast<const cpx<R>*>(a.in);
    const R* lut = static_cast<const R*>(a.lut);
    const LineLayout lay = line_layout<M>(a.block_w, a.rows, W, row, j);
    // the table in shared memory, the loop's scalars in registers: asked for here, needed after the first transform
    // (one CTA per SM and nothing to hide a global load behind)
    SLM_STATIC_SMEM R lut_s[256];
    if (HAS_T) for (int i = t; i < 256; i += G::THREADS) lut_s[i] = ld_ro(lut + i);
    const R s0r = MODE == RF_GS ? (R)ld_cg(&a.stats->scale) : (R)0;
    const double gd_scale = MODE == RF_GD_POST ? ld_cg(&a.stats->scale) : 0.0, gd_max = MODE == RF_GD_POST ? ld_cg(&a.stats->imax) : 0.0;
    sync_cta();
    cpx<R> v[E];
    unsigned grey4[(E + 3) / 4];                              // the points' grey levels, four to a register (they wait through a transform)
#pragma unroll
    for (int r = 0; r < (E + 3) / 4; ++r) grey4[r] = 0u;
    each_point<E, M>(lay, [&](int r, unsigned off) {
        v[r] = ld_plane(in + off);
        if (HAS_T) grey4[r / 4] |= (unsigned)ld_ro(a.T8 + off) << (8 * (r % 4));
    });
    if (MODE != RF_GD_POST) line_fft<R, W, -1, 1>(v, line, j, tw, sync);      // second half of C = fft2(B) / of med_output
    R mx = 0, sa = 0, sb = 0, sc = 0;
    if (MODE != RF_GD_MAX && a.intensity) each_point<E, M>(lay, [&](int r, unsigned off) { a.intensity[off] = (double)cnorm2(v[r]); });
    const R gdk = (R)gd_scale;                                // GD fp32: output = |F|^2 * (norm / max), like the column kernels
#pragma unroll
    for (int r = 0; r < E; ++r) {
        const R m2 = cnorm2(v[r]);
        const int grey = (int)((grey4[r / 4] >> (8 * (r % 4))) & 0xffu);
        if (MODE == RF_GS) {
            const R amp = lut_s[grey];
            gs_sums(m2, grey, s0r, mx, sa, sb, sc);
            replace_amplitude(v[r], m2, amp);
        } else if (MODE == RF_GD_MAX) {
            mx = fmax(mx, m2);                                                 // amax(output_unnormed), algorithms.py:86
        } else {
            // gd_output / gd_point written out: the table is read after the error sum here; a call reads it first, and that
            // changes the compiled fp64 kernels
            R I;                                                               // output, algorithms.py:86
            if (sizeof(R) == 8) I = (R)(((double)m2 * a.norm) / gd_max);
            else I = m2 * gdk;
            const R d = I - (R)grey;
            sa += d * d;                                                       // algorithms.py:92
            v[r] = cscale(cscale(v[r], lut_s[grey]), d);                       // mask * med_output * (output - T), :88
        }
    }
    if (MODE != RF_GD_MAX) line_fft<R, W, +1, 1>(v, line, j, tw, sync);       // first half of A = ifft2(D) / of dEdF
    cpx<R>* out = static_cast<cpx<R>*>(a.out);
    each_point<E, M>(lay, [&](int r, unsigned off) { st_plane(out + off, v[r]); });

    // per-line reduction over its M threads
    Partial p; p.mx = (double)mx; p.a = (double)sa; p.b = (double)sb; p.c = (double)sc;
    Partial q; q.mx = 0; q.a = 0; q.b = 0; q.c = 0;
    if (M >= 32) {                                            // a line is whole warps
        SLM_STATIC_SMEM Partial red[32];
        p = warp_reduce<F_ALL>(p);
        if (t % 32 == 0) red[t / 32] = p;
        sync_cta();
        if (j == 0)
            for (int w = 0; w < M / 32; ++w) q = combine<F_ALL>(q, red[rr * (M / 32) + w]);
    } else {                                                  // several short lines share a warp
        SLM_STATIC_SMEM Partial pt[M >= 32 ? 1 : G::THREADS];
        pt[M >= 32 ? 0 : t] = p;
        sync_cta();
        if (j == 0)
            for (int i = 0; i < M; ++i) q = combine<F_ALL>(q, pt[M >= 32 ? 0 : t + i]);
    }
    if (j == 0) {
        double* dst = a.partial + 4 * row;
        dst[0] = q.mx; dst[1] = q.a; dst[2] = q.b; dst[3] = q.c;
    }
}

// ---- plain column transform kernel -------------------------------------------------------------------
template <typename R, int H>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((ColGeom<R, H>::THREADS), 1) col_plain_kernel(PlainColArgs a) {
    SLM_DYN_SMEM(raw);
    col_tiles<R, H>(a.in, a.W, raw,
        [&](int b) { return a.output == OUT_STATS && ld_cg(&a.stats[b].done) != 0; },   // in-loop use (GD): finished planes rest
        [&](int b, int tile, int tiles, cpx<R>* v, cpx<R>* line, int t, int c, int j) {
            col_plain_tile<R, H>(a, b, tile, tiles, v, line, t, c, j);
        });
}

}  // namespace slm
