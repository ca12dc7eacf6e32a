// In-CTA line FFTs for the hologram passes (sm_100a).
//
// A "line" is one row or one column of an H x W plane.  Each thread owns E points of a line
// in registers; a line of N = E * m * E points is transformed by
//   stage 1 : radix-E butterflies on register data            -> shared memory
//   middle  : one radix-m stage, shared -> registers -> shared (m in {1,2,3,4,8,16}), or for any other
//             5-smooth m one such stage per radix of m (radices 2..16, 3, 5: mid_stages)
//   last    : radix-E butterflies, shared -> registers
// (Stockham autosort, so results come out in natural order and thread j again owns the
// points j + r*N/E, r = 0..E-1: exactly the mapping stage 1 consumes.  A fused
// inverse-FFT -> pointwise -> forward-FFT chain therefore never leaves registers between the
// two transforms, and global loads/stores are always unit-stride across threads.)
//
// Arithmetic: a complex number is one 64-bit register pair.  In fp32 every complex add, real
// scaling and complex multiply is issued as Blackwell's packed FADD2 / FMUL2 / FFMA2
// (PTX add/mul/fma.rn.f32x2): ptxas folds the half swaps, broadcasts and per-half negations of
// the formulas below into operand modifiers, so a complex multiply is 2 instructions and a
// radix-4 butterfly 8.  All shared-memory addresses are (per-thread base) + (compile-time offset).
//
// Replaces scipy.fft.fft2/ifft2 (pocketfft/DUCC) at the reference call sites
// algorithms.py:27,31,34,84,88,155 and generate_hologram.py:25.  Convention follows scipy:
// forward unnormalised; the 1/(H*W) of the inverse is applied by the caller where it matters.
#pragma once
#include "cuda_compat.h"

namespace slm {

template <typename R> struct cpx;
template <> struct alignas(8) cpx<float> { float x, y; };
template <> struct alignas(16) cpx<double> { double x, y; };

template <typename R> struct vec2;
template <> struct vec2<float> { using type = float2; };
template <> struct vec2<double> { using type = double2; };

// Plane data is streamed (read once / written once per pass): keep it out of L1.
template <typename R> SLM_DEV cpx<R> ld_plane(const cpx<R>* p) {
    typename vec2<R>::type v = ld_cg(reinterpret_cast<const typename vec2<R>::type*>(p));
    cpx<R> r; r.x = v.x; r.y = v.y; return r;
}
template <typename R> SLM_DEV void st_plane(cpx<R>* p, cpx<R> v) {
    typename vec2<R>::type t; t.x = v.x; t.y = v.y;
    st_cg(reinterpret_cast<typename vec2<R>::type*>(p), t);
}
template <typename R> SLM_DEV cpx<R> ld_const(const cpx<R>* p) {
    typename vec2<R>::type v = ld_ro(reinterpret_cast<const typename vec2<R>::type*>(p));
    cpx<R> r; r.x = v.x; r.y = v.y; return r;
}

// ---- packed pair arithmetic: (x, y) lanes ---------------------------------------------------
template <typename R> SLM_DEV cpx<R> mk(R x, R y) { cpx<R> r; r.x = x; r.y = y; return r; }
template <typename R> SLM_DEV cpx<R> pk_add(cpx<R> a, cpx<R> b) { return mk<R>(a.x + b.x, a.y + b.y); }
template <typename R> SLM_DEV cpx<R> pk_mul(cpx<R> a, cpx<R> b) { return mk<R>(a.x * b.x, a.y * b.y); }
template <typename R> SLM_DEV cpx<R> pk_fma(cpx<R> a, cpx<R> b, cpx<R> c) { return mk<R>(a.x * b.x + c.x, a.y * b.y + c.y); }
#if defined(__CUDA_ARCH__) && !defined(SLM_EMULATE)
SLM_DEV unsigned long long pk_bits(cpx<float> a) {
    unsigned long long r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a.x), "f"(a.y)); return r;
}
SLM_DEV cpx<float> pk_val(unsigned long long v) {
    cpx<float> r; asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v)); return r;
}
SLM_DEV cpx<float> pk_add(cpx<float> a, cpx<float> b) {
    unsigned long long r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk_bits(a)), "l"(pk_bits(b))); return pk_val(r);
}
SLM_DEV cpx<float> pk_mul(cpx<float> a, cpx<float> b) {
    unsigned long long r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(pk_bits(a)), "l"(pk_bits(b))); return pk_val(r);
}
SLM_DEV cpx<float> pk_fma(cpx<float> a, cpx<float> b, cpx<float> c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(pk_bits(a)), "l"(pk_bits(b)), "l"(pk_bits(c)));
    return pk_val(r);
}
#endif

// Hide a value's provenance from the optimiser (keeps per-thread constants from being expanded into tables of
// loop-invariant products that then live in local memory).
#if defined(__CUDA_ARCH__) && !defined(SLM_EMULATE)
SLM_DEV void opaque(cpx<float>& a) { asm volatile("" : "+f"(a.x), "+f"(a.y)); }
SLM_DEV void opaque(cpx<double>& a) { asm volatile("" : "+d"(a.x), "+d"(a.y)); }
SLM_DEV void opaque(unsigned& a) { asm volatile("" : "+r"(a)); }
#else
template <typename R> SLM_DEV void opaque(cpx<R>&) {}
SLM_DEV void opaque(unsigned&) {}
#endif

template <typename R> SLM_DEV cpx<R> cadd(cpx<R> a, cpx<R> b) { return pk_add(a, b); }
template <typename R> SLM_DEV cpx<R> csub(cpx<R> a, cpx<R> b) { return pk_add(a, mk<R>(-b.x, -b.y)); }
// a * w = a.x*(w.x, w.y) + a.y*(-w.y, w.x)
template <typename R> SLM_DEV cpx<R> cmul(cpx<R> a, cpx<R> w) {
    const cpx<R> t = pk_mul(mk<R>(a.y, a.y), mk<R>(w.y, w.x));
    return pk_fma(mk<R>(a.x, a.x), w, mk<R>(-t.x, t.y));
}
template <typename R> SLM_DEV cpx<R> cconj(cpx<R> a) { a.y = -a.y; return a; }
template <typename R> SLM_DEV cpx<R> cscale(cpx<R> a, R s) { return pk_mul(a, mk<R>(s, s)); }
// squared modulus and its two halves
template <typename R> SLM_DEV R cnorm2(cpx<R> a) { const cpx<R> q = pk_mul(a, a); return q.x + q.y; }

// multiply by exp(DIR * i * pi/2): DIR=-1 (forward) -> -i ; DIR=+1 (inverse) -> +i
template <int DIR, typename R> SLM_DEV cpx<R> rot90(cpx<R> a) {
    return DIR < 0 ? mk<R>(a.y, -a.x) : mk<R>(-a.y, a.x);
}
// multiply by exp(DIR * 2*pi*i * P/16)
template <int DIR, int P, typename R> SLM_DEV cpx<R> mul_w16(cpx<R> a) {
    constexpr int p = ((P % 16) + 16) % 16;
    if constexpr (p == 0) return a;
    else if constexpr (p == 4) return rot90<DIR>(a);
    else if constexpr (p == 8) return mk<R>(-a.x, -a.y);
    else if constexpr (p == 12) return rot90<-DIR>(a);
    else if constexpr (p % 2 == 0) {
        // odd multiples of pi/4: (cos, sin) = (+-h, +-h):  a*(c + i s) = (c*a.x - s*a.y, s*a.x + c*a.y)
        constexpr double h = 0.70710678118654752440;
        constexpr double C = (p == 2 || p == 14) ? h : -h;
        constexpr double S0 = (p == 2 || p == 6) ? h : -h;
        constexpr double S = DIR < 0 ? -S0 : S0;
        // = h * ( sc*a.x - ss*a.y, ss*a.x + sc*a.y ) with signs sc, ss
        const cpx<R> u = (C > 0) == (S > 0) ? pk_add(a, mk<R>(-a.y, a.x)) : pk_add(a, mk<R>(a.y, -a.x));
        return pk_mul(u, mk<R>((R)C, (R)C));
    } else {
        constexpr double CS[16] = {1.0, 0.92387953251128673848, 0.70710678118654752440, 0.38268343236508977173,
                                   0.0, -0.38268343236508977173, -0.70710678118654752440, -0.92387953251128673848,
                                   -1.0, -0.92387953251128673848, -0.70710678118654752440, -0.38268343236508977173,
                                   0.0, 0.38268343236508977173, 0.70710678118654752440, 0.92387953251128673848};
        constexpr double SN[16] = {0.0, 0.38268343236508977173, 0.70710678118654752440, 0.92387953251128673848,
                                   1.0, 0.92387953251128673848, 0.70710678118654752440, 0.38268343236508977173,
                                   0.0, -0.38268343236508977173, -0.70710678118654752440, -0.92387953251128673848,
                                   -1.0, -0.92387953251128673848, -0.70710678118654752440, -0.38268343236508977173};
        return cmul(a, mk<R>((R)CS[p], (R)(DIR < 0 ? -SN[p] : SN[p])));
    }
}

// ---- small DFTs on register arrays, natural order in and out -----------------------------
template <int DIR, typename R> SLM_DEV void dft2(cpx<R>& a, cpx<R>& b) {
    cpx<R> t = csub(a, b); a = cadd(a, b); b = t;
}
template <int DIR, typename R> SLM_DEV void dft3(cpx<R>& a, cpx<R>& b, cpx<R>& c) {
    const R h = (R)0.86602540378443864676;          // sin(2*pi/3)
    const cpx<R> s = cadd(b, c), d = csub(b, c);
    const cpx<R> m = pk_fma(mk<R>((R)-0.5, (R)-0.5), s, a);
    const cpx<R> q = pk_mul(rot90<DIR>(d), mk<R>(h, h));   // DIR * i * sin(2pi/3) * (b - c)
    a = cadd(a, s);
    b = cadd(m, q);
    c = csub(m, q);
}
template <int DIR, typename R> SLM_DEV void dft4(cpx<R>& a0, cpx<R>& a1, cpx<R>& a2, cpx<R>& a3) {
    const cpx<R> t0 = cadd(a0, a2), t1 = csub(a0, a2), t2 = cadd(a1, a3), t3 = rot90<DIR>(csub(a1, a3));
    a0 = cadd(t0, t2); a1 = cadd(t1, t3); a2 = csub(t0, t2); a3 = csub(t1, t3);
}
template <int DIR, typename R> SLM_DEV void dft8(cpx<R>* v) {
    // 8 = 4 x 2 : DFT4 over n1 (stride 2), twiddle W8^(n2*k1), DFT2 over n2
    dft4<DIR>(v[0], v[2], v[4], v[6]);
    dft4<DIR>(v[1], v[3], v[5], v[7]);
    v[3] = mul_w16<DIR, 2>(v[3]);
    v[5] = rot90<DIR>(v[5]);
    v[7] = mul_w16<DIR, 6>(v[7]);
    dft2<DIR>(v[0], v[1]); dft2<DIR>(v[2], v[3]); dft2<DIR>(v[4], v[5]); dft2<DIR>(v[6], v[7]);
    // position 2*k1 + k2 holds X[k1 + 4*k2]
    cpx<R> x1 = v[2], x2 = v[4], x3 = v[6], x4 = v[1], x5 = v[3], x6 = v[5];
    v[1] = x1; v[2] = x2; v[3] = x3; v[4] = x4; v[5] = x5; v[6] = x6;
}
template <int DIR, typename R> SLM_DEV void dft16(cpx<R>* v) {
    // 16 = 4 x 4
#pragma unroll
    for (int n2 = 0; n2 < 4; ++n2) dft4<DIR>(v[n2], v[n2 + 4], v[n2 + 8], v[n2 + 12]);
    // position n2 + 4*k1 *= W16^(n2*k1)
    v[5] = mul_w16<DIR, 1>(v[5]);  v[9] = mul_w16<DIR, 2>(v[9]);   v[13] = mul_w16<DIR, 3>(v[13]);
    v[6] = mul_w16<DIR, 2>(v[6]);  v[10] = mul_w16<DIR, 4>(v[10]); v[14] = mul_w16<DIR, 6>(v[14]);
    v[7] = mul_w16<DIR, 3>(v[7]);  v[11] = mul_w16<DIR, 6>(v[11]); v[15] = mul_w16<DIR, 9>(v[15]);
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) dft4<DIR>(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);
    // position 4*k1 + k2 holds X[k1 + 4*k2] : transpose
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = a + 1; b < 4; ++b) { cpx<R> t = v[4 * a + b]; v[4 * a + b] = v[4 * b + a]; v[4 * b + a] = t; }
}
// multiply by exp(DIR * 2*pi*i * P/32)
template <int DIR, int P, typename R> SLM_DEV cpx<R> mul_w32(cpx<R> a) {
    constexpr int p = ((P % 32) + 32) % 32;
    if constexpr (p % 2 == 0) return mul_w16<DIR, p / 2>(a);
    else {
        constexpr double C32[8] = {0.98078528040323044913, 0.83146961230254523708, 0.55557023301960222474, 0.19509032201612826785,
                                   -0.19509032201612826785, -0.55557023301960222474, -0.83146961230254523708, -0.98078528040323044913};
        constexpr double S32[8] = {0.19509032201612826785, 0.55557023301960222474, 0.83146961230254523708, 0.98078528040323044913,
                                   0.98078528040323044913, 0.83146961230254523708, 0.55557023301960222474, 0.19509032201612826785};
        // odd p = 2q+1, q = 0..15: angle (2q+1)*pi/16; second half of the circle by symmetry
        constexpr int q = p / 2;
        constexpr double c = q < 8 ? C32[q] : -C32[q - 8];
        constexpr double sn = q < 8 ? S32[q] : -S32[q - 8];
        return cmul(a, mk<R>((R)c, (R)(DIR < 0 ? -sn : sn)));
    }
}
template <int DIR, int K, typename R> struct Dft32Combine {
    static SLM_DEV void run(cpx<R>* v, const cpx<R>* e, const cpx<R>* o) {
        const cpx<R> t = mul_w32<DIR, K>(o[K]);
        v[K] = cadd(e[K], t);
        v[K + 16] = csub(e[K], t);
        if constexpr (K + 1 < 16) Dft32Combine<DIR, K + 1, R>::run(v, e, o);
    }
};
template <int DIR, typename R> SLM_DEV void dft32(cpx<R>* v) {
    // 32 = 2 x 16 (decimation in time): X[k] = E[k] + W32^k O[k], X[k+16] = E[k] - W32^k O[k]
    cpx<R> e[16], o[16];
#pragma unroll
    for (int m = 0; m < 16; ++m) { e[m] = v[2 * m]; o[m] = v[2 * m + 1]; }
    dft16<DIR>(e);
    dft16<DIR>(o);
    Dft32Combine<DIR, 0, R>::run(v, e, o);
}
template <int DIR, typename R> SLM_DEV void dft5(cpx<R>* v) {
    const R c1 = (R)0.30901699437494742410, c2 = (R)-0.80901699437494742410;     // cos(2pi/5), cos(4pi/5)
    const R s1 = (R)0.95105651629515357212, s2 = (R)0.58778525229247312917;      // sin(2pi/5), sin(4pi/5)
    const cpx<R> t1 = cadd(v[1], v[4]), t2 = cadd(v[2], v[3]), t3 = csub(v[1], v[4]), t4 = csub(v[2], v[3]);
    const cpx<R> a1 = pk_fma(mk<R>(c2, c2), t2, pk_fma(mk<R>(c1, c1), t1, v[0]));
    const cpx<R> a2 = pk_fma(mk<R>(c1, c1), t2, pk_fma(mk<R>(c2, c2), t1, v[0]));
    const cpx<R> b1 = rot90<DIR>(pk_fma(mk<R>(s2, s2), t4, cscale(t3, s1)));    // DIR * i * (s1 t3 + s2 t4)
    const cpx<R> b2 = rot90<DIR>(pk_fma(mk<R>(-s1, -s1), t4, cscale(t3, s2)));  // DIR * i * (s2 t3 - s1 t4)
    v[0] = cadd(v[0], cadd(t1, t2));
    v[1] = cadd(a1, b1); v[4] = csub(a1, b1);
    v[2] = cadd(a2, b2); v[3] = csub(a2, b2);
}
template <int RAD, int DIR, typename R> SLM_DEV void dft_small(cpx<R>* v) {
    if constexpr (RAD == 2) dft2<DIR>(v[0], v[1]);
    else if constexpr (RAD == 3) dft3<DIR>(v[0], v[1], v[2]);
    else if constexpr (RAD == 5) dft5<DIR>(v);
    else if constexpr (RAD == 4) dft4<DIR>(v[0], v[1], v[2], v[3]);
    else if constexpr (RAD == 8) dft8<DIR>(v);
    else if constexpr (RAD == 16) dft16<DIR>(v);
    else if constexpr (RAD == 32) dft32<DIR>(v);
    else static_assert(RAD == 2, "unsupported radix");
}

// ---- twiddles ----------------------------------------------------------------------------
// tw[q] = exp(-2*pi*i*q/N), q in [0,N), computed in extended precision on the host.
// TW_SHARED: the table has been copied to shared memory (plain load); otherwise read-only global path.
template <int DIR, bool TW_SHARED, typename R> SLM_DEV cpx<R> tw_load(const cpx<R>* tw, int q) {
    cpx<R> w = TW_SHARED ? tw[q] : ld_const(tw + q);
    if (DIR > 0) w.y = -w.y;
    return w;
}
// w[r] = w1^r for r = 1..RAD-1 by a depth-log2 product tree (error ~ log2(RAD) ulp)
template <int RAD, typename R> SLM_DEV void twiddle_powers(cpx<R>* w, cpx<R> w1) {
    w[1] = w1;
#pragma unroll
    for (int r = 2; r < RAD; ++r) w[r] = cmul(w[r / 2], w[r - r / 2]);
}

// ---- line FFT ----------------------------------------------------------------------------
#ifndef SLM_E32_LEN
#define SLM_E32_LEN 0          // tuning builds: one more line length transformed with 32 points per thread
#endif
// The middle of a plan is a list of Stockham stages, one per radix: the power-of-two part of m as one radix (at most 16),
// then the 3s, then the 5s.  E.g. 1152 = 8 * (2*3*3) * 8, 1920 = 8 * (2*3*5) * 8, 1280 = 16 * 5 * 16.
struct MidRadices { int n; int r[8]; };
SLM_HOSTDEV constexpr MidRadices mid_radices(int m) {
    MidRadices s{0, {0, 0, 0, 0, 0, 0, 0, 0}};
    int p2 = 1;
    while (m > 0 && m % 2 == 0) { p2 *= 2; m /= 2; }
    if (p2 > 1) s.r[s.n++] = p2;
    while (m > 0 && m % 3 == 0 && s.n < 8) { s.r[s.n++] = 3; m /= 3; }
    while (m > 0 && m % 5 == 0 && s.n < 8) { s.r[s.n++] = 5; m /= 5; }
    if (m != 1 || p2 > 16) s.n = -1;               // a prime factor above 5, or a power-of-two part above 16
    return s;
}
SLM_HOSTDEV constexpr bool valid_middle(int m) { return m >= 1 && mid_radices(m).n >= 0; }
SLM_HOSTDEV constexpr int default_points(int N) {
    return (N >= 8192 || N == SLM_E32_LEN) ? 32 : (N % 256 == 0 && valid_middle(N / 256)) ? 16 : 8;
}
// Column transforms of 4096 points keep 32 points per thread: 128 threads per column let a CTA hold FOUR columns
// (32-byte row segments, whole sectors) instead of two; measured 0.48 -> 0.36 ms per Fourier-plane pass (2 x 4096^2).
// The row kernels stay at 16 (the GD row pass holds x beside the field and would spill).
#ifndef SLM_COL_E32_LEN
#define SLM_COL_E32_LEN 0      // tuning builds: one more COLUMN length with 32 points per thread
#endif
SLM_HOSTDEV constexpr int column_points(int N) { return (N == 4096 || N == SLM_COL_E32_LEN) ? 32 : default_points(N); }
template <int N, int EP = default_points(N)> struct FftPlan {
    static constexpr int E = EP;                       // points per thread
    static constexpr int M = N / E;                    // threads per line
    static constexpr int MID = N / (E * E);            // middle radix (1 = none)
    static constexpr int NP = N + N / E;               // padded line length in shared memory
    // ONE_STAGE: the middle radices with their own stage code (one butterfly set per thread, or radix 3 predicated);
    // every other middle runs as the Stockham stages of mid_radices(MID)
    static constexpr bool ONE_STAGE = MID == 1 || MID == 2 || MID == 3 || MID == 4 || MID == 8 || MID == 16;
    static_assert(E * E * MID == N, "line length must be E*E*m");
    static_assert(valid_middle(MID), "unsupported line length: the middle must be 5-smooth with a power-of-two part <= 16");
    static_assert(M % 8 == 0, "threads per line must be a multiple of 8");
    static_assert(!ONE_STAGE || MID <= E || MID == 3, "middle radix must fit the per-thread register tile");
    SLM_HOSTDEV static constexpr int pad(int i) { return i + i / E; }
};
template <int N> using ColPlan = FftPlan<N, column_points(N)>;

// Transform one line.  v[r] = x[j + r*M] on entry, X[j + r*M] on exit.  `line` points at the
// line's element 0 in shared memory; element i lives at line[pad(i) * STRIDE], pad(i) = i + i/E.
// `sync` is the barrier over the threads that share the shared-memory lines being transformed
// together (the whole CTA, or a named barrier over the warps of one line group); every thread of
// that group must call line_fft together.
//
// Address algebra (M = MID*E, so every index below splits into a per-thread base and a
// compile-time offset):
//   stage-1 store   j*E + r                    -> pad = j*(E+1) + r
//   loads           j + e*M                    -> pad = (j + j/E) + e*(M + MID)
//   middle store    (j/E + q*MID)*E*MID + j%E + r*E
//                                              -> pad = (j/E)*(E*MID+MID) + j%E + q*MID*(E*MID+MID) + r*(E+1)
// Barrier policies for line_fft.
struct CtaSync { SLM_DEV void operator()() const { sync_cta(); } };
template <int THREADS> struct GroupSync {          // THREADS == 0: whole CTA
    int id;
    SLM_DEV void operator()() const { if (THREADS == 0) sync_cta(); else if (THREADS == 32) sync_warp(); else sync_named(id, THREADS); }
};

// Middle stages S, S+1, ... of a composite plan (FftPlan::ONE_STAGE false), shared -> registers -> shared.  Stage S
// has radix RS = mid_radices(MID).r[S] and Ns = E * (earlier middle radices): butterfly b < N/RS (k = b mod Ns) reads
// points b + p*N/RS, multiplies them by tw[k*p*N/(Ns*RS)] and writes its outputs to (b/Ns)*Ns*RS + k + p*Ns.  Thread j
// takes the butterflies b = j + q*M (q < QMAX, the last ones predicated).  Ns divides M = E*MID, so k = j mod Ns for
// every q, and every offset below is a multiple of E: pad() keeps (per-thread base) + (compile-time offset).
template <typename R, int N, int E, int DIR, int STRIDE, bool TW_SHARED, int S, int NS, class Sync>
SLM_DEV void mid_stages(cpx<R>* line, int j, const cpx<R>* SLM_RESTRICT tw, Sync sync) {
    constexpr MidRadices MR = mid_radices(N / (E * E));
    constexpr int RS = MR.r[S], M = N / E, EP = E + 1;
    constexpr int NB = N / RS, QMAX = (NB + M - 1) / M;
    const int k = j % NS, o = (j / NS) * NS * RS + k;
    cpx<R>* const ldp = line + (j + j / E) * STRIDE;
    cpx<R>* const stp = line + (o + o / E) * STRIDE;
    cpx<R> w[RS];
#pragma unroll
    for (int p = 1; p < RS; ++p) w[p] = tw_load<DIR, TW_SHARED>(tw, k * p * (N / (NS * RS)));
    cpx<R> a[QMAX][RS];
#pragma unroll
    for (int q = 0; q < QMAX; ++q) {
        if (QMAX * M == NB || j + q * M < NB) {
#pragma unroll
            for (int p = 0; p < RS; ++p) a[q][p] = ldp[((q * M + p * NB) / E) * EP * STRIDE];
        }
    }
    sync();
#pragma unroll
    for (int q = 0; q < QMAX; ++q) {
        if (QMAX * M == NB || j + q * M < NB) {
#pragma unroll
            for (int p = 1; p < RS; ++p) a[q][p] = cmul(a[q][p], w[p]);
            dft_small<RS, DIR>(a[q]);
#pragma unroll
            for (int p = 0; p < RS; ++p) stp[((q * M * RS + p * NS) / E) * EP * STRIDE] = a[q][p];
        }
    }
    sync();
    if constexpr (S + 1 < MR.n) mid_stages<R, N, E, DIR, STRIDE, TW_SHARED, S + 1, NS * RS>(line, j, tw, sync);
}

template <typename R, int N, int DIR, int STRIDE, class Sync = CtaSync, bool TW_SHARED = false, int POINTS = default_points(N)>
SLM_DEV void line_fft(cpx<R>* v, cpx<R>* line, int j, const cpx<R>* SLM_RESTRICT tw, Sync sync = Sync()) {
    using P = FftPlan<N, POINTS>;
    constexpr int E = P::E, M = P::M, MID = P::MID;
    constexpr int EP = E + 1, MP = M + MID, BLK = E * MID + MID;
    cpx<R>* const st1 = line + (j * EP) * STRIDE;
    cpx<R>* const ldp = line + (j + j / E) * STRIDE;

    // stage 1 (Ns = 1): no twiddles; butterfly output r goes to position j*E + r
    dft_small<E, DIR>(v);
#pragma unroll
    for (int r = 0; r < E; ++r) st1[r * STRIDE] = v[r];
    sync();

    if constexpr (!P::ONE_STAGE) {
        mid_stages<R, N, E, DIR, STRIDE, TW_SHARED, 0, E>(line, j, tw, sync);
    } else if constexpr (MID > 1) {
        const int jh = j / E, jl = j % E;
        cpx<R>* const stm = line + (jh * BLK + jl) * STRIDE;
        cpx<R> w[MID];
        twiddle_powers<MID>(w, tw_load<DIR, TW_SHARED>(tw, jl * E));      // exp(-+2 pi i jl / (E*MID)), same for every q
        if constexpr (MID != 3) {
            constexpr int Q = E / MID;                           // butterflies per thread
#pragma unroll
            for (int e = 0; e < E; ++e) v[e] = ldp[e * MP * STRIDE];
            sync();
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                cpx<R> a[MID];
                a[0] = v[q];
#pragma unroll
                for (int r = 1; r < MID; ++r) a[r] = cmul(v[q + r * Q], w[r]);
                dft_small<MID, DIR>(a);
#pragma unroll
                for (int r = 0; r < MID; ++r) stm[(q * MID * BLK + r * EP) * STRIDE] = a[r];
            }
        } else {
            constexpr int NB = N / 3, NBP = NB + NB / E, QMAX = (NB + M - 1) / M;
            cpx<R> a[QMAX][3];
#pragma unroll
            for (int q = 0; q < QMAX; ++q) {
                if (j + q * M < NB) {
#pragma unroll
                    for (int r = 0; r < 3; ++r) a[q][r] = ldp[(q * MP + r * NBP) * STRIDE];
                }
            }
            sync();
#pragma unroll
            for (int q = 0; q < QMAX; ++q) {
                if (j + q * M < NB) {
                    a[q][1] = cmul(a[q][1], w[1]);
                    a[q][2] = cmul(a[q][2], w[2]);
                    dft3<DIR>(a[q][0], a[q][1], a[q][2]);
#pragma unroll
                    for (int r = 0; r < 3; ++r) stm[(q * MID * BLK + r * EP) * STRIDE] = a[q][r];
                }
            }
        }
        sync();
    }

    // last stage (Ns = M): twiddle W_N^(r*j), butterfly, result r is X[j + r*M]
#pragma unroll
    for (int r = 0; r < E; ++r) v[r] = ldp[r * MP * STRIDE];
    sync();                      // the tile may be overwritten by the next transform
    {
        cpx<R> w[E];
        twiddle_powers<E>(w, tw_load<DIR, TW_SHARED>(tw, j));
#pragma unroll
        for (int r = 1; r < E; ++r) v[r] = cmul(v[r], w[r]);
    }
    dft_small<E, DIR>(v);
}

}  // namespace slm
