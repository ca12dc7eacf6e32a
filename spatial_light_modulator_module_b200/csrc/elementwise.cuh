// Analytic holograms, modulo-2pi composition and the 8-bit SLM quantisers (sm_100a).
//
// These are the reference's float64 scalar expressions evaluated one pixel per thread.  Every
// operation is an explicitly rounded IEEE double operation in the reference's order (no FMA
// contraction), so results are bit-identical to numpy's.
#pragma once
#include "engine_types.h"
#include "passes.cuh"

namespace slm {

#define SLM_TWO_PI 6.283185307179586   // float(2*np.pi)

// Python / numpy `a % b` for floats with b > 0 (npy_divmod): fmod, then move into [0, b)
SLM_DEV double py_mod(double a, double b) {
    double m = fmod(a, b);
    if (m != 0.0) { if (m < 0.0) m = add_rn(m, b); }
    else m = copysign(0.0, b);
    return m;
}

// wavefront_correction.py:440-449 (deflect_2pi): const * (sin(y*u)*i + sin(x*u)*j) % 2pi
SLM_GLOBAL void deflect_kernel(double* out, int H, int W, double konst, double sy, double sx) {
    const long long n = (long long)H * W;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(p / W), j = (int)(p % W);
        const double ph = mul_rn(konst, add_rn(mul_rn(sy, (double)i), mul_rn(sx, (double)j)));
        out[p] = py_mod(ph, SLM_TWO_PI);
    }
}

// generate_hologram.py:189-203 (lens): k * (1 - sqrt(1 + r^2/f^2)) % 2pi with
// r = px*sqrt((i-h/2)^2 + (j-w/2)^2), k = 2*pi*f/lambda; `trunc` reproduces the uint8 store (:192,:202)
SLM_GLOBAL void lens_kernel(double* out, int H, int W, double px, double k, double f2, int trunc_u8) {
    const long long n = (long long)H * W;
    const double hh = (double)H / 2.0, hw = (double)W / 2.0;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(p / W), j = (int)(p % W);
        const double di = sub_rn((double)i, hh), dj = sub_rn((double)j, hw);
        const double r = mul_rn(px, sqrt_rn(add_rn(mul_rn(di, di), mul_rn(dj, dj))));
        const double q = div_rn(mul_rn(r, r), f2);
        double ph = py_mod(mul_rn(k, sub_rn(1.0, sqrt_rn(add_rn(1.0, q)))), SLM_TWO_PI);
        if (trunc_u8) ph = (double)(unsigned char)(long long)ph;
        out[p] = ph;
    }
}

// generate_hologram.py:181,186: (hologram + addend) % (2*pi).  `b` is one plane broadcast over the batch.
SLM_GLOBAL void add_mod2pi_kernel(const double* a, const double* b, double* out, long long n, long long plane) {
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x)
        out[p] = py_mod(add_rn(a[p], b[p % plane]), SLM_TWO_PI);
}

// astype(np.uint8) of a float64 on x86: convert to a wide integer, keep the low byte
SLM_DEV unsigned char wrap_u8(double v) { return (unsigned char)(long long)v; }
// PIL fromarray(float64) -> mode "F" (float32) -> convert("L"): clamp to [0,255], truncate
SLM_DEV unsigned char pil_f_to_l(double v) {
    const float f = (float)v;
    if (f <= 0.0f) return 0;
    if (f >= 255.0f) return 255;
    return (unsigned char)f;
}

enum QuantMode {
    QUANT_Q1 = 1,   // np.round(h*ct2pi/2pi).astype(uint8)            wavefront_correction.py:458-459
    QUANT_Q2 = 2,   // ((h+mask)%2pi)/2pi*ct2pi -> PIL F -> L          display_holograms.py:253-258,265
    QUANT_Q3 = 3,   // ((h[+mask])%2pi*ct2pi/2pi).astype(uint8)        move_traps.py:135-138, show_hologram.py:9-11
    QUANT_PREVIEW = 5,   // PIL fromarray(float64).convert("L")        generate_hologram_sequence.py:29
};
SLM_GLOBAL void quantize_kernel(const double* h, const double* mask, double ct2pi, int mode, unsigned char* out,
                                long long n, long long plane) {
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        double v = h[p];
        unsigned char q;
        if (mode == QUANT_Q1) {
            q = wrap_u8(rint(div_rn(mul_rn(v, ct2pi), SLM_TWO_PI)));
        } else if (mode == QUANT_Q2) {
            if (mask) v = add_rn(v, mask[p % plane]);
            q = pil_f_to_l(mul_rn(div_rn(py_mod(v, SLM_TWO_PI), SLM_TWO_PI), ct2pi));
        } else if (mode == QUANT_Q3) {
            if (mask) v = add_rn(v, mask[p % plane]);
            q = wrap_u8(div_rn(mul_rn(py_mod(v, SLM_TWO_PI), ct2pi), SLM_TWO_PI));
        } else {
            q = pil_f_to_l(v);
        }
        out[p] = q;
    }
}
// display_holograms.py:259-264: (int16(grey) + mask/2pi*ct2pi) % ct2pi -> PIL F -> L
SLM_GLOBAL void quantize_grey_kernel(const unsigned char* g, const double* mask, double ct2pi, unsigned char* out,
                                     long long n, long long plane) {
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        const double m = mul_rn(div_rn(mask[p % plane], SLM_TWO_PI), ct2pi);
        out[p] = pil_f_to_l(py_mod(add_rn((double)g[p], m), ct2pi));
    }
}

// initial guess "fourier" (algorithms.py:154-157): inc * exp(1j*angle(A)) from the setup field
template <typename R, typename RA>
SLM_GLOBAL void phasor_field_kernel(const cpx<RA>* A, const R* inc, cpx<R>* x, long long n, long long plane) {
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        cpx<RA> z = unit_phasor(A[p]);
        R s = inc ? inc[p % plane] : (R)1;
        cpx<R> o; o.x = (R)z.x * s; o.y = (R)z.y * s;
        x[p] = o;
    }
}

// initial guesses "random" / "zeros" (algorithms.py:118-124,145-151): exp(1j*2*pi*u) [/100] from the
// host-drawn MT19937 stream u.  The argument 2*pi*u is rounded to double first, as numpy does.
template <typename R>
SLM_GLOBAL void random_phasor_kernel(const double* u, cpx<R>* x, long long n, double divide_by) {
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        const double arg = mul_rn(mul_rn(2.0, 3.141592653589793), u[p]);
        double re = cos(arg), im = sin(arg);
        if (divide_by != 1.0) { re = div_rn(re, divide_by); im = div_rn(im, divide_by); }
        cpx<R> o; o.x = (R)re; o.y = (R)im;
        x[p] = o;
    }
}

// Python's random.random() stream on the device (make_initial_guess, algorithms.py:117-150): MT19937 continued
// from a 624-word state.  One CTA.  The recurrence  x[k+624] = x[k+397] ^ tw(x[k], x[k+1])  is linear over
// GF(2), so a whole block of 624 new words is written in terms of the OLD block only -- word i is the XOR of
// one old word and the tw() terms of i, i-227, i-454 (as many as exist) -- and needs ONE barrier per block
// instead of one per 227-word dependency step.  Thread t owns words 2t and 2t+1 of each block, i.e. exactly
// the pair genrand_res53 turns into a double (a>>5, b>>6), tempered in registers.
// `pos` (even) is the read position inside the incoming block; state_out = final block + final position.
constexpr int kMtThreads = 320;                      // 312 word pairs per block
SLM_DEV unsigned mt_tw(unsigned a, unsigned b) {
    const unsigned y = (a & 0x80000000u) | (b & 0x7fffffffu);
    return (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}
SLM_DEV unsigned mt_temper(unsigned y) {
    y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
    return y;
}
SLM_DEV double mt_res53(unsigned w0, unsigned w1) {
    const unsigned a = mt_temper(w0) >> 5, b = mt_temper(w1) >> 6;
    return ((double)a * 67108864.0 + (double)b) / 9007199254740992.0;
}
// word i of the next block from the old block o[0..623]
SLM_DEV unsigned mt_next_word(const unsigned* o, int i) {
    if (i < 227) return o[i + 397] ^ mt_tw(o[i], o[i + 1]);
    if (i < 454) return o[i + 170] ^ mt_tw(o[i - 227], o[i - 226]) ^ mt_tw(o[i], o[i + 1]);
    if (i < 623) return o[i - 57] ^ mt_tw(o[i - 454], o[i - 453]) ^ mt_tw(o[i - 227], o[i - 226]) ^ mt_tw(o[i], o[i + 1]);
    const unsigned n0 = o[397] ^ mt_tw(o[0], o[1]);                                       // new word 0
    const unsigned n396 = o[566] ^ mt_tw(o[169], o[170]) ^ mt_tw(o[396], o[397]);         // new word 396
    return n396 ^ mt_tw(o[623], n0);
}
SLM_GLOBAL void mt19937_uniform_kernel(const unsigned* state_in, int pos, double* u, long long n, unsigned* state_out) {
    SLM_STATIC_SMEM unsigned mt[2][624];
    const int t = threadIdx.x;
    for (int i = t; i < 624; i += kMtThreads) mt[0][i] = state_in[i];
    sync_cta();
    int cur = 0;
    long long produced = 0;                          // doubles written so far
    if (pos < 624) {                                 // what is left of the incoming block
        const long long avail = (624 - pos) / 2;
        const int take = (int)(n < avail ? n : avail);
        if (t < take) u[t] = mt_res53(mt[0][pos + 2 * t], mt[0][pos + 2 * t + 1]);
        produced = take;
        pos += 2 * take;
    }
    while (produced < n) {
        const unsigned* o = mt[cur];
        unsigned* w = mt[cur ^ 1];
        const long long want = n - produced;
        const int take = want < 312 ? (int)want : 312;
        if (t < 312) {
            const unsigned w0 = mt_next_word(o, 2 * t), w1 = mt_next_word(o, 2 * t + 1);
            w[2 * t] = w0; w[2 * t + 1] = w1;
            if (t < take) u[produced + t] = mt_res53(w0, w1);
        }
        produced += take;
        pos = 2 * take;
        cur ^= 1;
        sync_cta();                                  // the new block is complete; the old one may be overwritten next trip
    }
    for (int i = t; i < 624; i += kMtThreads) state_out[i] = mt[cur][i];
    if (t == 0) state_out[624] = (unsigned)pos;
}

// inc * exp(1j*phase): restart a GS run from a hologram (B of algorithms.py:30 with angle(A) = phase)
template <typename R>
SLM_GLOBAL void phase_phasor_kernel(const double* phase, const R* inc, cpx<R>* x, long long n, long long plane) {
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        const double h = phase[p];
        const R s = inc ? inc[p % plane] : (R)1;
        cpx<R> o; o.x = (R)cos(h) * s; o.y = (R)sin(h) * s;
        x[p] = o;
    }
}

// move_traps.update_hologram (move_traps.py:64-68): angle(ifft2(one-hot at (row, col))) in closed form,
// 2*pi*(row*i/H + col*j/W) wrapped into (-pi, pi]
SLM_GLOBAL void single_trap_kernel(double* out, int H, int W, int row, int col) {
    const long long n = (long long)H * W;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(p / W), j = (int)(p % W);
        // exact integer phase fractions: (row*i mod H)/H + (col*j mod W)/W
        const double f = (double)(((long long)row * i) % H) / (double)H + (double)(((long long)col * j) % W) / (double)W;
        double fr = f - floor(f);                       // in [0, 1)
        if (fr > 0.5) fr -= 1.0;                        // (-0.5, 0.5]
        out[p] = fr * 6.283185307179586;
    }
}

// trap frames (traps_images.py:10-16,87-91): white single pixels at (frame, y, x) on a black stack
SLM_GLOBAL void scatter_dots_kernel(unsigned char* frames, const int* fyx, int n_dots, long long plane, int W) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d < n_dots) frames[(long long)fyx[3 * d] * plane + (long long)fyx[3 * d + 1] * W + fyx[3 * d + 2]] = 255;
}

// Slab exchange layout <-> row slab (slab-decomposed 2-D transform).  With h lines per rank and P = W/h peers:
//   to_exchange : out[q][c][i] = in[i][q*h + c]     (block q is what peer q receives; each block transposed)
//   from_exchange: out[i][q*h + c] = in[q][c][i]
// 32x32 tiles through padded shared memory, coalesced on both sides.
template <typename T>
SLM_GLOBAL void transpose_blocks_kernel(const T* in, T* out, int h, int W, int from_exchange) {
    SLM_STATIC_SMEM T tile[32][33];
    const int q = blockIdx.z, tc = blockIdx.y * 32, ti = blockIdx.x * 32;    // block, first column c, first row i
    const int tx = threadIdx.x % 32, ty = threadIdx.x / 32;                   // 32 x 8 threads
    const size_t blk = (size_t)q * h * h;
    if (!from_exchange) {
#pragma unroll
        for (int k = 0; k < 32; k += 8) tile[ty + k][tx] = in[(size_t)(ti + ty + k) * W + (size_t)q * h + tc + tx];     // [i][c]
        sync_cta();
#pragma unroll
        for (int k = 0; k < 32; k += 8) out[blk + (size_t)(tc + ty + k) * h + ti + tx] = tile[tx][ty + k];              // [c][i]
    } else {
#pragma unroll
        for (int k = 0; k < 32; k += 8) tile[ty + k][tx] = in[blk + (size_t)(tc + ty + k) * h + ti + tx];               // [c][i]
        sync_cta();
#pragma unroll
        for (int k = 0; k < 32; k += 8) out[(size_t)(ti + ty + k) * W + (size_t)q * h + tc + tx] = tile[tx][ty + k];    // [i][c]
    }
}

// The same, with every block going to (or coming from the point of view of) ANOTHER device: `peers.p[q]` is the
// base of rank q's buffer, mapped into this process (peer memory over NVLink), `self` this rank.
//   push      (from_exchange = 0): peer q's receive buffer, block `self`:  p[q][self][c][i] = in[i][q*h + c]
//   push back (from_exchange = 1): peer q's row slab, my columns:           p[q][i][self*h + c] = in[q][c][i]
// The stores ARE the all-to-all: the blocks cross the links while the tiles are being transposed.
struct PeerPtrs { void* p[16]; };
template <typename T>
SLM_GLOBAL void transpose_blocks_peer_kernel(const T* in, PeerPtrs peers, int h, int W, int from_exchange, int self, int n_x) {
    SLM_STATIC_SMEM T tile[32][33];
    // Destinations vary FASTEST over the grid and start behind this rank: at any moment a rank's CTAs write to all
    // peers at once, and no two ranks begin with the same one.  (With the peer as the slowest index every rank stored
    // into rank 0 first, then into rank 1, ...: one NVLink ingress at a time carried the whole exchange -- measured
    // on 8 GPUs at 16384^2: 1.2 ms per exchange of 117 MB per rank, the time of 940 MB through ONE port.)
    const int np = gridDim.x / n_x;
    const int q = (blockIdx.x % np + self + 1) % np;
    const int tc = blockIdx.y * 32, ti = (blockIdx.x / np) * 32;
    const int tx = threadIdx.x % 32, ty = threadIdx.x / 32;
    T* out = static_cast<T*>(peers.p[q]);
    if (!from_exchange) {
#pragma unroll
        for (int k = 0; k < 32; k += 8) tile[ty + k][tx] = in[(size_t)(ti + ty + k) * W + (size_t)q * h + tc + tx];     // [i][c]
        sync_cta();
        const size_t blk = (size_t)self * h * h;
#pragma unroll
        for (int k = 0; k < 32; k += 8) out[blk + (size_t)(tc + ty + k) * h + ti + tx] = tile[tx][ty + k];              // [c][i]
    } else {
        const size_t blk = (size_t)q * h * h;
#pragma unroll
        for (int k = 0; k < 32; k += 8) tile[ty + k][tx] = in[blk + (size_t)(tc + ty + k) * h + ti + tx];               // [c][i]
        sync_cta();
#pragma unroll
        for (int k = 0; k < 32; k += 8) out[(size_t)(ti + ty + k) * W + (size_t)self * h + tc + tx] = tile[tx][ty + k];  // [i][c]
    }
}

// ---- loop state of the row-slab GS on the device (no host round trip per iteration) ---------------------------------
// partial[rows][4] (max |C|^2, sum r^2, sum r*u, sum u^2 per line) -> out[4] for this rank: ONE CTA, fixed order.
SLM_GLOBAL void rows_reduce_kernel(const double* partial, int rows, double* out, PeerPtrs peers, int n_peers, int self) {
    Partial q; q.mx = 0; q.a = 0; q.b = 0; q.c = 0;
    for (int i = threadIdx.x; i < rows; i += blockDim.x) {
        Partial r; r.mx = partial[4 * i]; r.a = partial[4 * i + 1]; r.b = partial[4 * i + 2]; r.c = partial[4 * i + 3];
        q = combine<F_ALL>(q, r);
    }
    q = block_reduce<256, F_ALL>(q, threadIdx.x);
    if (threadIdx.x == 0) {
        out[0] = q.mx; out[1] = q.a; out[2] = q.b; out[3] = q.c;
        for (int r = 0; r < n_peers; ++r) {                       // peer mode: every rank's `gathered[self]` (else the caller all-gathers)
            double* g = static_cast<double*>(peers.p[r]) + 4 * self;
            g[0] = q.mx; g[1] = q.a; g[2] = q.b; g[3] = q.c;
        }
    }
}
// gathered[world][4] -> the plane's max and sums (rank order: the same bits on every rank); closes the iteration like
// close_plane<GS>: state[0] = scale (in: the one the pass used, out: norm / max), state[1] = error, state[2] = iterations
// done (as a double), state[3] = loop-ended flag.  prepass: only the scale (exact scale of iteration 0).
// form: 0 GS iteration; 1 only the scale and the max (GS iteration 0's exact scale; the max pass of every GD iteration,
// algorithms.py:86); 2 GD iteration: error = sum (output - T)^2 / HW (algorithms.py:92), scale and max stay.  `stats`
// (nullable): the context's PlaneStats, which the GD SLM-plane pass reads (iteration count -> learning rate, loop ended).
SLM_GLOBAL void rows_close_kernel(const double* gathered, int world, double norm, double hw, int form, int as_float,
                                  double tolerance, double* state, double* err_curve, PlaneStats* stats) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double mx = 0, a = 0, b = 0, c = 0;
    for (int r = 0; r < world; ++r) {
        mx = fmax(mx, gathered[4 * r]); a += gathered[4 * r + 1]; b += gathered[4 * r + 2]; c += gathered[4 * r + 3];
    }
    if (form == 1) { state[0] = norm / mx; state[4] = mx; return; }
    double err;
    if (form == 0) {
        const double s = norm / mx;                               // algorithms.py:37
        const double s0u = as_float ? (double)(float)state[0] : state[0];      // the scale the kernel used
        const double dl = s0u != 0.0 ? s / s0u - 1.0 : 0.0;
        err = (a + 2.0 * dl * b + dl * dl * c) / hw;              // algorithms.py:38,162
        state[0] = s; state[4] = mx;
    } else {
        err = a / hw;                                             // algorithms.py:92
    }
    const int k = (int)state[2];
    err_curve[k] = err;
    state[1] = err; state[2] = (double)(k + 1);
    state[3] = !(err > tolerance) ? 1.0 : 0.0;                    // loop condition, algorithms.py:29,83
    if (stats) { stats->err = err; stats->iters = k + 1; stats->done = !(err > tolerance); }
}

// complex<R> <-> complex128 / real conversions at the boundary (numpy hands over complex128)
template <typename TS, typename TD>
SLM_GLOBAL void convert_kernel(const TS* in, TD* out, long long n) {
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (long long)gridDim.x * blockDim.x)
        out[p] = (TD)in[p];
}

}  // namespace slm
