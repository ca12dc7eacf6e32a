// Warp-per-column persistent Fourier-plane kernel (sm_100a) for fp32 columns of 1024 and 768 points
// (768 = the SLM height of the reference, constants.py:6).
//
// Why a second column kernel: the group kernel (col_groups.cuh) keeps 16 points per thread, so a column is
// shared by two warps that meet at four named barriers per transform, and one CTA of 16 compute warps
// (96 registers) is all an SM holds -- ncu shows it latency bound (issue slots ~30 % busy).  Here
//   * ONE WARP owns a column: 1024 = 32 x 32, 32 points per lane, one lane<->register transpose per
//     transform through shared memory, no barrier inside a transform (only __syncwarp); 768 = 32 lanes x 24
//     points on the SLM-plane side <-> 24 lanes x 32 points on the Fourier-plane side;
//   * the transpose is done IN PLACE in the tile buffer: the two warps of a column pair split the pair's
//     16-byte chunk of the 64B-swizzled tile image by rows (512 rows each), which makes every exchange
//     access a conflict-free 64-bit access (a single column alone only reaches half of the banks); the two
//     warps meet twice per tile (after reading the tile into registers, before writing the results back);
//   * no exchange buffer is needed, so THREE 64 KB tile buffers fit and TWO tiles are transformed
//     concurrently by two groups of eight warps, out of phase, while the third buffer is in flight
//     (TMA store of a finished tile, TMA load of the next one);
//   * a service warp sequences the tiles (descriptor + per-plane scalars in shared memory, TMA, staging of
//     the 8-bit target rows), a second one publishes the tiles' partial sums and closes a plane's iteration.
// Arithmetic, reductions and loop control are those of col_groups.cuh (same modes, same results).
#pragma once
#include "col_groups.cuh"

namespace slm {

template <typename R, int H> struct ColWarpGeom {
    static constexpr int M = 32;                                  // lanes per column
    static constexpr int RA = H / 32;                             // "side A" (tile order): lane j holds rows j + 32 p, p < RA
                                                                  // "side B" (after a forward transform): lane j < RA holds rows j + RA k, k < 32
    static constexpr int TC = 8;                                  // columns per tile (64-byte rows)
    static constexpr int GROUPS = 2, NBUF = 3;
    static constexpr int GROUP_THREADS = TC * M;                  // 256: eight warps, one per column
    static constexpr int COMPUTE = GROUPS * GROUP_THREADS;        // 512
    static constexpr int THREADS = COMPUTE + 128;                 // + service warpgroup: sequencer, 2 staging helpers, publisher
    static constexpr int COPIERS = 64;                            // two helper warps stage the 8-bit target rows
    static constexpr int ROWB = TC * (int)sizeof(cpx<R>);
    static constexpr bool OK = sizeof(R) == 4 && (H == 1024 || H == 768);
    static constexpr size_t TILE = (size_t)H * ROWB;              // 64 KB
    static constexpr size_t GREY = (size_t)H * TC;                // 8 KB
    // [tile x3][grey x3][lut][red 3 x 8][desc x3][barriers]
    static constexpr size_t OFF_GREY = NBUF * TILE;
    static constexpr size_t OFF_LUT = OFF_GREY + NBUF * GREY;
    static constexpr size_t OFF_RED = OFF_LUT + 256 * sizeof(R);
    static constexpr size_t OFF_DESC = OFF_RED + NBUF * TC * sizeof(Partial);
    static constexpr size_t OFF_ORDER = OFF_DESC + NBUF * 32;     // [NBUF] staging orders of the sequencer to its helpers
    static constexpr size_t OFF_FMX = OFF_ORDER + NBUF * 8;       // CGM_GD_FUSED: [NBUF][TC] column maxima, [NBUF] plane max
    static constexpr size_t OFF_BAR = OFF_FMX + NBUF * (TC + 2) * 4;
    static constexpr size_t SMEM = OFF_BAR + 5 * NBUF * 32;
    static_assert(!OK || SMEM <= 232448, "shared memory budget");
};

// Per-plane state of the one-pass GD forms in global memory: one 64-bit word per plane, low half = bit pattern of the
// running max |F|^2, high half = tiles that have contributed -- so that ONE load tells a waiting tile both whether its
// plane is complete and what the max is (a round trip to L2 less on its critical path).  Contributors update the max,
// fence, then the count; word [max_planes] is the passes' time-out flag.
SLM_DEV unsigned* plane_max_word(const ColArgs& a, int b) { return a.fused_max + 2 * (size_t)b; }
SLM_DEV unsigned* plane_count_word(const ColArgs& a, int b) { return a.fused_max + 2 * (size_t)b + 1; }
SLM_DEV unsigned* plane_timeout_flag(const ColArgs& a) { return a.fused_max + 2 * (size_t)a.max_planes; }
// -> true when every tile of the plane has contributed; max_bits then holds the plane's max
SLM_DEV bool plane_complete(const ColArgs& a, int b, int tiles, unsigned& max_bits) {
    const unsigned long long w = ld_acquire_u64(reinterpret_cast<const unsigned long long*>(plane_max_word(a, b)));
    max_bits = (unsigned)w;
    return (unsigned)(w >> 32) >= (unsigned)tiles;
}

// What the sequencer tells the other warps about the tile in a buffer.
struct TileDesc { long long g; double scale, imax, norm; };      // g < 0: no more tiles

// f(b): byte offset (inside the 1 KB that 16 rows x one 16-byte chunk span) of element b of a 32-element
// run, laid out as 16-byte units on consecutive rows of the 64B-swizzled image.  XOR-linear in b.
SLM_HOSTDEV constexpr unsigned xch_f(unsigned b) { return ((b >> 1) << 6) | (((b >> 2) & 3u) << 4) | ((b & 1u) << 3); }

// ---- 24-point DFT on registers: natural order in, position 8 k1 + k2 holds X[k1 + 3 k2] on exit -------------
// multiply by exp(DIR * 2 pi i * M / 24)
template <int DIR, int M, typename R> SLM_DEV cpx<R> mul_w24(cpx<R> a) {
    constexpr int m = ((M % 24) + 24) % 24;
    if constexpr (m % 3 == 0) return mul_w16<DIR, 2 * (m / 3)>(a);          // multiples of 45 degrees
    else {
        constexpr double C24[24] = {1.0, 0.96592582628906828675, 0.86602540378443864676, 0.70710678118654752440, 0.5,
                                    0.25881904510252076235, 0.0, -0.25881904510252076235, -0.5, -0.70710678118654752440,
                                    -0.86602540378443864676, -0.96592582628906828675, -1.0, -0.96592582628906828675,
                                    -0.86602540378443864676, -0.70710678118654752440, -0.5, -0.25881904510252076235, 0.0,
                                    0.25881904510252076235, 0.5, 0.70710678118654752440, 0.86602540378443864676,
                                    0.96592582628906828675};
        constexpr double sn = C24[(m + 18) % 24];                            // sin(x) = cos(x - pi/2)
        return cmul(a, mk<R>((R)C24[m], (R)(DIR < 0 ? -sn : sn)));
    }
}
template <int DIR, int N2, typename R> struct Dft24Twiddle {                // position 8 k1 + n2 *= W24^(n2 k1), k1 = 1, 2
    static SLM_DEV void run(cpx<R>* v) {
        v[8 + N2] = mul_w24<DIR, N2>(v[8 + N2]);
        v[16 + N2] = mul_w24<DIR, 2 * N2>(v[16 + N2]);
        if constexpr (N2 + 1 < 8) Dft24Twiddle<DIR, N2 + 1, R>::run(v);
    }
};
template <int DIR, typename R> SLM_DEV void dft24(cpx<R>* v) {
    // n = 8 n1 + n2, k = k1 + 3 k2:  X[k1 + 3 k2] = sum_n2 W8^(n2 k2) W24^(n2 k1) sum_n1 W3^(n1 k1) x[8 n1 + n2]
#pragma unroll
    for (int n2 = 0; n2 < 8; ++n2) dft3<DIR>(v[n2], v[8 + n2], v[16 + n2]);
    Dft24Twiddle<DIR, 1, R>::run(v);
    dft8<DIR>(v); dft8<DIR>(v + 8); dft8<DIR>(v + 16);
}

// Side-A register transform of a column of H = 32 RA points and the index its position p holds afterwards.
template <int RA> SLM_HOSTDEV constexpr int side_a_index(int p) { return RA == 32 ? p : (p / 8 + 3 * (p % 8)); }
template <int RA> SLM_HOSTDEV constexpr int side_a_position(int q) { return RA == 32 ? q : (8 * (q % 3) + q / 3); }
template <int RA, int DIR, typename R> SLM_DEV void dft_side_a(cpx<R>* v) {
    if constexpr (RA == 32) dft_small<32, DIR>(v); else dft24<DIR>(v);
}

// v[pos(q)] *= w1^q, q = 1..RA-1 (pos = side_a_position when PERMUTED, else identity); the powers are formed in
// blocks of four so few of them are live at a time.
template <int RA, bool PERMUTED, int Q, typename R> struct TwiddleRun {
    static SLM_DEV void run(cpx<R>* v, const cpx<R>* w, cpx<R> W) {      // w[1..3] = w1^1..3, w[4] = w1^4, W = w1^(4 floor(Q/4))
        constexpr int pos = PERMUTED ? side_a_position<RA>(Q) : Q;
        if constexpr (Q % 4 == 0) { if constexpr (Q > 4) W = cmul(W, w[4]); v[pos] = cmul(v[pos], W); }
        else if constexpr (Q < 4) v[pos] = cmul(v[pos], w[Q]);
        else v[pos] = cmul(v[pos], cmul(W, w[Q % 4]));
        if constexpr (Q + 1 < RA) TwiddleRun<RA, PERMUTED, Q + 1, R>::run(v, w, W);
    }
};
template <int RA, bool PERMUTED, typename R> SLM_DEV void twiddle_run(cpx<R>* v, cpx<R> w1) {
    cpx<R> w[5];
    w[1] = w1; w[2] = cmul(w1, w1); w[3] = cmul(w[2], w1); w[4] = cmul(w[2], w[2]);
    TwiddleRun<RA, PERMUTED, 1, R>::run(v, w, w[4]);
}

// Exchange accesses: address = (lane base ^ X) + OFF with X, OFF compile-time.  The XOR is issued inside the asm
// statement so the addresses of a transform are formed where they are used (one LOP3 each); left to the
// optimiser they are computed once per tile, kept across the two transforms and spilled to local memory.
#if defined(__CUDA_ARCH__) && !defined(SLM_EMULATE)
using XchBase = unsigned;                                        // shared-window address
SLM_DEV XchBase xch_base(unsigned char* buf, unsigned off) { return smem_addr(buf) + off; }
template <unsigned X, unsigned OFF> SLM_DEV void xch_store(XchBase base, cpx<float> v) {
    asm volatile("{\n.reg .u32 a;\nxor.b32 a, %0, %1;\nst.shared.v2.f32 [a+%2], {%3, %4};\n}"
                 ::"r"(base), "n"(X), "n"(OFF), "f"(v.x), "f"(v.y) : "memory");
}
template <unsigned X, unsigned OFF> SLM_DEV cpx<float> xch_load(XchBase base) {
    cpx<float> v;
    asm volatile("{\n.reg .u32 a;\nxor.b32 a, %2, %3;\nld.shared.v2.f32 {%0, %1}, [a+%4];\n}"
                 : "=f"(v.x), "=f"(v.y) : "r"(base), "n"(X), "n"(OFF) : "memory");
    return v;
}
#else
struct XchBase { unsigned char* buf; unsigned off; };
inline XchBase xch_base(unsigned char* buf, unsigned off) { return XchBase{buf, off}; }
template <unsigned X, unsigned OFF, typename R> inline void xch_store(XchBase b, cpx<R> v) { *reinterpret_cast<cpx<R>*>(b.buf + ((b.off ^ X) + OFF)) = v; }
template <unsigned X, unsigned OFF> inline cpx<float> xch_load(XchBase b) { return *reinterpret_cast<const cpx<float>*>(b.buf + ((b.off ^ X) + OFF)); }
#endif
// The warp's exchange region holds a [32][32] array of slots (fewer rows or columns used for RA = 24); slot
// (i, j) lives at element 32 i + (j ^ i), which makes a warp's access conflict free whether its lanes run over
// i (LANE-major: address = lane base ^ f(j)) or over j (STEP-major: address = (lane base ^ f(i)) + 1024 i).
template <int P, int N, int RA, bool PERMUTED> struct XchRun {
    static constexpr unsigned C = (unsigned)(PERMUTED ? side_a_index<RA>(P) : P);        // the index position P holds
    template <typename R> static SLM_DEV void store_step_major(XchBase b, const cpx<R>* v) {
        xch_store<xch_f(C), 1024u * C>(b, v[P]);
        if constexpr (P + 1 < N) XchRun<P + 1, N, RA, PERMUTED>::store_step_major(b, v);
    }
    template <typename R> static SLM_DEV void store_lane_major(XchBase b, const cpx<R>* v) {
        xch_store<xch_f(C), 0u>(b, v[P]);
        if constexpr (P + 1 < N) XchRun<P + 1, N, RA, PERMUTED>::store_lane_major(b, v);
    }
    template <typename R> static SLM_DEV void load_step_major(XchBase b, cpx<R>* v) {
        v[P] = xch_load<xch_f(C), 1024u * C>(b);
        if constexpr (P + 1 < N) XchRun<P + 1, N, RA, PERMUTED>::load_step_major(b, v);
    }
    template <typename R> static SLM_DEV void load_lane_major(XchBase b, cpx<R>* v) {
        v[P] = xch_load<xch_f(C), 0u>(b);
        if constexpr (P + 1 < N) XchRun<P + 1, N, RA, PERMUTED>::load_lane_major(b, v);
    }
};

// Forward transform of a column of H = 32 RA points held by a warp.
//   in : side A, v[p] = x[lane + 32 p], p < RA
//   out: side B, v[k] = X[lane + RA k], k < 32, in lanes < RA
// lm / sm: this lane's LANE-major / STEP-major base inside the warp's exchange region (1 KB aligned region).
template <int RA, typename R>
SLM_DEV void warp_fft_forward(cpx<R>* v, unsigned char* buf, unsigned lm, unsigned sm, cpx<R> w1) {
    dft_side_a<RA, -1>(v);                                       // over n2 = p: Y[n1 = lane][k2 = idx(p)]
    opaque(w1);                                                  // (or the powers are hoisted out of the tile loop and spilled)
    twiddle_run<RA, true>(v, w1);                                // * W_H^(lane k2)
    sync_warp();                                                 // earlier reads of the region are complete
    XchRun<0, RA, RA, true>::store_step_major(xch_base(buf, sm), v);     // slot (k2, lane)
    sync_warp();
    XchRun<0, 32, RA, false>::load_lane_major(xch_base(buf, lm), v);     // slot (lane, r) = Y[n1 = r][k2 = lane]
    dft_small<32, -1>(v);                                        // over n1 = r: X[lane + RA k1]
}
// Inverse transform (unnormalised): side B in, side A out with position p holding y[lane + 32 idx(p)].
template <int RA, typename R>
SLM_DEV void warp_fft_inverse(cpx<R>* v, unsigned char* buf, unsigned lm, unsigned sm, cpx<R> w1, bool active) {
    dft_small<32, +1>(v);                                        // over n2' = k: Z[n1' = lane][k2' = k]
    sync_warp();
    if (active) XchRun<0, 32, RA, false>::store_lane_major(xch_base(buf, lm), v);        // slot (lane, k2'), lanes < RA
    sync_warp();
    XchRun<0, RA, RA, false>::load_step_major(xch_base(buf, sm), v);     // slot (r, lane) = Z[n1' = r][k2' = lane]
    w1.y = -w1.y;
    opaque(w1);
    twiddle_run<RA, false>(v, w1);                               // * conj(W_H)^(r lane)
    dft_side_a<RA, +1>(v);                                       // over n1' = r: y[lane + 32 k1'], k1' = idx(p)
}

// Declared in col_groups.cuh: when a one-pass GD form closes a plane, every tile of the plane has used the plane's max --
// record it and re-arm the plane's words for the next pass.
SLM_DEV void close_fused_max(const ColArgs& a, int b, double norm) {
    PlaneStats* st = a.stats + b;
    const double pm = (double)__uint_as_float(ld_cg(plane_max_word(a, b)));
    st->imax = pm; st->scale = norm / pm;
    *plane_max_word(a, b) = 0u; *plane_count_word(a, b) = 0u;
}

// The one-pass GD forms' share of a plane's max |F|^2 (algorithms.py:86).  A column's max on side B, in every lane.
template <typename R> SLM_DEV R side_b_max(const cpx<R>* v, bool active) {
    R m = 0;
#pragma unroll
    for (int r = 0; r < 32; ++r) m = fmax(m, cnorm2(v[r]));
    if (!active) m = 0;                                          // lanes outside side B hold no points
#pragma unroll
    for (int sh = 16; sh >= 1; sh >>= 1) m = fmax(m, shfl_xor(m, sh));
    return m;
}
// A tile's column maxima fmx[0..TC) -> its plane's max word, then its arrival count.
template <int TC> SLM_DEV void add_tile_max(const ColArgs& a, int b, const float* fmx) {
    float mm = fmx[0];
#pragma unroll
    for (int i = 1; i < TC; ++i) mm = fmax(mm, fmx[i]);
    atomic_max_u32(plane_max_word(a, b), __float_as_uint(mm));  // |F|^2 >= 0: ordered like its bit pattern
    fence_device();
    atomic_add_u32(plane_count_word(a, b), 1u);
}

// One lane waits until every tile of plane b has contributed; -> the bits of the plane's max.  Should the other tiles not
// come (the CTAs of the launch not all resident: a foreign kernel holding SMs for good), it gives up after ~2 s with the
// time-out flag set instead of hanging the device.  PAUSE: back off between polls (the pipelined form's waiting lane).
template <bool PAUSE> SLM_DEV unsigned wait_plane_max(const ColArgs& a, int b, int tiles) {
    const long long t0 = clock_now();
    unsigned max_bits;
    while (!plane_complete(a, b, tiles, max_bits)) {
        if (PAUSE) spin_pause();
        if (clock_now() - t0 > (1ll << 32)) { atomic_max_u32(plane_timeout_flag(a), 1u); break; }
    }
    return max_bits;
}

// The targets of side-B rows lane + RA (r0 + i), i < 8, of a column: grey level and table entry from the tile's grey rows
// (gsrc: the lane's first), or T and the second plane from global memory at goff (zero in lanes outside side B).
template <int RA, int TC, typename R>
SLM_DEV void side_b_targets(const ColArgs& a, bool use_t8, bool active, const uint8_t* gsrc, const R* lut_s, size_t goff, int r0,
                            R* tv, R* aux) {
    if (use_t8) {
#pragma unroll
        for (int i = 0; i < 8; ++i) { const int gl = gsrc[(size_t)(r0 + i) * RA * TC]; tv[i] = (R)gl; aux[i] = lut_s[gl]; }
    } else {
        const R* T = static_cast<const R*>(a.Treal) + goff;
        const R* Q = static_cast<const R*>(a.plane2) + goff;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            tv[i] = active ? ld_ro(T + (size_t)(r0 + i) * RA * a.W) : (R)0;
            aux[i] = active ? ld_ro(Q + (size_t)(r0 + i) * RA * a.W) : (R)0;
        }
    }
}

template <typename R, int H, int MODE>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((ColWarpGeom<R, H>::THREADS), 1)
col_warp_kernel(ColGroupArgs ga, const SLM_GRID_CONSTANT TileMap tm_in, const SLM_GRID_CONSTANT TileMap tm_out) {
    using G = ColWarpGeom<R, H>;
    constexpr int TC = G::TC, ROWB = G::ROWB, NBUF = G::NBUF;
    constexpr bool FUSED = MODE == CGM_GD_FUSED;
    constexpr bool PIPE = MODE == CGM_GD_PIPE;                      // group 0 transforms forward, group 1 does the rest of the tile
    constexpr int STOPS = PIPE ? 1 : G::GROUPS;                     // stop markers that end the kernel (PIPE: both groups see every item)
    constexpr bool HAS_T = cgm_has_target(MODE);
    constexpr bool HAS_OUT = MODE != CGM_STATS;
    constexpr bool IS_GD = cgm_is_gd(MODE);
    constexpr bool IS_STATS = cgm_is_stats(MODE);
    constexpr bool HAS_STATS = MODE != CGM_COMPLEX;
    constexpr int FIELDS = close_fields(cgm_close(MODE));
    const ColArgs& a = ga.c;
    SLM_DYN_SMEM(raw);
    R* const lut_s = reinterpret_cast<R*>(raw + G::OFF_LUT);
    Partial* const red = reinterpret_cast<Partial*>(raw + G::OFF_RED);                 // [NBUF][TC]
    TileDesc* const desc = reinterpret_cast<TileDesc*>(raw + G::OFF_DESC);             // [NBUF]
    TileBarrier* const full = reinterpret_cast<TileBarrier*>(raw + G::OFF_BAR);        // [NBUF] tile (and grey rows) landed
    TileBarrier* const done = reinterpret_cast<TileBarrier*>(raw + G::OFF_BAR + NBUF * 32);     // [NBUF] group is through the tile
    TileBarrier* const taken = reinterpret_cast<TileBarrier*>(raw + G::OFF_BAR + 2 * NBUF * 32); // [NBUF] publisher has the tile's sums
    TileBarrier* const ordered = reinterpret_cast<TileBarrier*>(raw + G::OFF_BAR + 3 * NBUF * 32); // [NBUF] a staging order is posted
    TileBarrier* const fwd = reinterpret_cast<TileBarrier*>(raw + G::OFF_BAR + 4 * NBUF * 32);     // [NBUF] PIPE: the slot holds the transformed field
    auto tile_buf = [&](int s) { return raw + (size_t)s * G::TILE; };
    auto grey_buf = [&](int s) { return raw + G::OFF_GREY + (size_t)s * G::GREY; };
    auto bar = [](TileBarrier* base, int s) { return reinterpret_cast<TileBarrier*>(reinterpret_cast<unsigned char*>(base) + s * 32); };

    const int t = threadIdx.x;
    const int tiles = a.W / TC;
    const long long total = (long long)a.B * tiles;
    const bool use_t8 = HAS_T && a.T8 != nullptr;
    griddep_launch();
    if (t == 0) {
        for (int s = 0; s < NBUF; ++s) {
            mbar_init(bar(full, s), use_t8 ? 2u : 1u);
            mbar_init(bar(done, s), (unsigned)G::GROUP_THREADS);
            mbar_init(bar(taken, s), 1u);
            mbar_init(bar(ordered, s), 1u);
            mbar_init(bar(fwd, s), (unsigned)G::GROUP_THREADS);
        }
        mbar_fence_init();
    }
    if (use_t8) {
        const R* lut = static_cast<const R*>(a.lut);
        for (int i = t; i < 256; i += G::THREADS) lut_s[i] = ld_ro(lut + i);
    }
    griddep_wait();
    sync_cta();

    // Register budget: 640 threads launch with 96 registers each; the service warpgroup gives most of its share
    // back and the four compute warpgroups take it (32 points per lane need ~110 registers).
    if (t >= G::COMPUTE) reg_dealloc<64>(); else reg_alloc<104>();
    if (t >= G::COMPUTE + 96) {
        // ================= publisher warp =================
        if (!HAS_STATS) return;
        const int lane = t - G::COMPUTE - 96;
        if constexpr (PIPE) {
            // Two duties, polled in turn so neither holds the other up: (i) a tile that group 0 has transformed hands its
            // max |F|^2 to its plane (atomic max, then the plane's arrival count) -- kept off the compute warps' path: a
            // round trip to L2 is a quarter of a tile's transform; (ii) the sums of a finished tile, as in the other modes.
            // (Watching the planes' arrival counts here as well, to spare group 1 its polling, made both duties late:
            //  measured 0.251 instead of 0.238 ms per pass.  Handing the tiles out on demand from a device counter instead
            //  of the fixed order -- in case some CTAs were simply slower -- changed nothing: 0.2422 / 0.2445 against
            //  0.2423 / 0.2444 ms; the CTAs drift apart by jitter, not by speed.)
            float* const fmx = reinterpret_cast<float*>(raw + G::OFF_FMX);
            unsigned kf = 0, kd = 0;             // next tile to hand its max over / to publish
            bool fend = false;                   // group 0 has reached the stop marker
            for (;;) {
                // lane 0 looks at the barriers; every lane acts on what IT saw
                enum { EV_FSTOP = 1, EV_FWD = 2, EV_DSTOP = 8, EV_DONE = 16 };
                unsigned ev = 0;
                if (lane == 0) {
                    if (!fend) {
                        const int s = (int)(kf % NBUF);
                        const unsigned par = (kf / NBUF) & 1u;
                        if (mbar_test(bar(full, s), par)) {
                            if (desc[s].g < 0) ev |= EV_FSTOP;
                            else if (mbar_test(bar(fwd, s), par)) ev |= EV_FWD;
                        }
                    }
                    if (kd < kf || fend) {
                        const int s = (int)(kd % NBUF);
                        const unsigned par = (kd / NBUF) & 1u;
                        if (mbar_test(bar(full, s), par)) {
                            if (desc[s].g < 0) ev |= EV_DSTOP;
                            else if (mbar_test(bar(done, s), par)) ev |= EV_DONE;
                        }
                    }
                }
                ev = shfl_idx(ev, 0);
                if (ev & EV_FSTOP) fend = true;
                if (ev & EV_FWD) {
                    const int s = (int)(kf % NBUF);
                    if (lane == 0) add_tile_max<TC>(a, (int)(desc[s].g / tiles), fmx + s * (TC + 2));
                    ++kf;
                }
                if (ev & EV_DSTOP) break;
                if (ev & EV_DONE) {
                    const int s = (int)(kd % NBUF);
                    const TileDesc d = desc[s];
                    const int b = (int)(d.g / tiles), tile = (int)(d.g % tiles);
                    Partial q; q.mx = 0; q.a = 0; q.b = 0; q.c = 0;
                    if (lane < TC) q = red[s * TC + lane];
                    q = warp_reduce<FIELDS>(q);
                    if (lane == 0) mbar_arrive(bar(taken, s));
                    publish_tile<R, H, MODE>(ga, b, tile, tiles, lane, q, d.scale, d.norm);
                    ++kd;
                }
                if (!(ev & (EV_FWD | EV_DONE | EV_FSTOP))) spin_pause();
            }
            return;
        }
        for (unsigned k = 0;; ++k) {
            const int s = (int)(k % NBUF);
            const unsigned par = (k / NBUF) & 1u;
            mbar_wait(bar(full, s), par);
            const TileDesc d = desc[s];
            if (d.g < 0) break;
            const int b = (int)(d.g / tiles), tile = (int)(d.g % tiles);
            mbar_wait(bar(done, s), par);                    // the group's sums of this tile are in shared memory
            Partial q; q.mx = 0; q.a = 0; q.b = 0; q.c = 0;
            if (lane < TC) q = red[s * TC + lane];
            q = warp_reduce<FIELDS>(q);                      // (also: every lane holds its copy before the slot is released)
            if (lane == 0) mbar_arrive(bar(taken, s));
            publish_tile<R, H, MODE>(ga, b, tile, tiles, lane, q, d.scale, d.norm);
        }
        return;
    }

    long long* const order = reinterpret_cast<long long*>(raw + G::OFF_ORDER);       // [NBUF] tile whose target rows slot s wants
    if (t >= G::COMPUTE + 32) {
        // ================= staging helpers: the 8-bit target rows of every posted tile -> its grey buffer =================
        // (off the sequencer's path: a tile's rows are requested as soon as its slot's previous tile is done,
        //  and land while that tile's store drains and the new tile's TMA load is in flight)
        if (!use_t8) return;
        const int who = t - G::COMPUTE - 32;
        int stops = 0;
        for (unsigned k = 0; stops < STOPS; ++k) {
            const int s = (int)(k % NBUF);
            mbar_wait(bar(ordered, s), (k / NBUF) & 1u);
            const long long g = order[s];
            if (g < 0) { ++stops; continue; }
            const int b = (int)(g / tiles), tile = (int)(g % tiles);
            copy_grey_tile<TC, H, G::COPIERS>(a.T8 + (size_t)b * H * a.W + (size_t)tile * TC, (size_t)a.W, grey_buf(s), who);
            sync_named(15, G::COPIERS);
            if (who == 0) mbar_arrive(bar(full, s));
        }
        return;
    }
    if (t >= G::COMPUTE) {
        // ================= sequencer warp: tile order, TMA, target staging =================
        const int lane = t - G::COMPUTE;
        // A candidate tile and its plane's scalars; the loads are issued here and looked at later (resolve).
        struct Peek { long long g; int done; double scale, imax, norm; };
        auto peek = [&](long long g) {
            Peek p; p.g = g; p.done = 0; p.scale = 0; p.imax = 0; p.norm = 0;
            if (g < total && MODE != CGM_COMPLEX) {
                const int b = (int)(g / tiles);
                const PlaneStats* ps = a.stats + b;
                p.done = ga.all_planes ? 0 : ld_cg(&ps->done); p.scale = ld_cg(&ps->scale); p.imax = ld_cg(&ps->imax); p.norm = ld_ro(a.norm + b);
            }
            return p;
        };
        // -> descriptor of the first tile at or after the candidate whose plane is still iterating (g = -1: none)
        auto resolve = [&](Peek p) {
            while (p.g < total && p.done) p = peek(p.g + gridDim.x);      // finished planes rest (tolerance > 0 only)
            TileDesc d; d.g = p.g < total ? p.g : -1; d.scale = p.scale; d.imax = p.imax; d.norm = p.norm;
            return d;
        };
        // tell the helpers which tile's target rows slot s needs next (its grey buffer is free: the slot's tile is done)
        auto stage_grey = [&](int s, const TileDesc& d) {
            if (!use_t8 || lane != 0) return;
            order[s] = d.g;
            mbar_arrive(bar(ordered, s));
        };
        // the buffer is free (its last tile stored and drained, its sums and descriptor taken): hand it over
        auto post = [&](int s, const TileDesc& d) {
            if (lane != 0) return;
            desc[s] = d;
            if (d.g < 0) {                                   // stop marker: complete the phase without data
                mbar_arrive(bar(full, s));
                if (use_t8) mbar_arrive(bar(full, s));       // (the helpers do not arrive for a stop marker)
                return;
            }
            const int b = (int)(d.g / tiles), tile = (int)(d.g % tiles);
            tile_load(tm_in, tile_buf(s), bar(full, s), (long long)b * H, H, (long long)tile * ROWB, ROWB, (int)sizeof(R));
        };
        // the tile that will be loaded when the next buffer frees: have L2 fetch it now, so that load is an L2 hit
        // (A/B on one box: GS pass +2 %; the light max passes, which run near the memory system's limits, lose 4 %
        //  to the extra requests and do without)
        auto prefetch = [&](const TileDesc& d) {
            if (IS_STATS || lane != 0 || d.g < 0) return;
            const int b = (int)(d.g / tiles), tile = (int)(d.g % tiles);
            tile_prefetch(tm_in, (long long)b * H, H, (long long)tile * ROWB, (int)sizeof(R));
        };
        TileDesc cur = resolve(peek(blockIdx.x));
        unsigned k = 0;                                      // next item (tile or stop marker) to issue
        int stops = 0;                                       // stop markers issued: one per group ends the kernel
        while (k < (unsigned)NBUF && stops < STOPS) {
            const int s = (int)(k % NBUF);
            stage_grey(s, cur);
            sync_warp();
            post(s, cur);
            ++k;
            if (cur.g < 0) ++stops; else cur = resolve(peek(cur.g + gridDim.x));
            prefetch(cur);
        }
        // retire tile kd (store it), then reuse its buffer for item kd + NBUF
        for (unsigned kd = 0; kd < k - (unsigned)stops; ++kd) {              // k - stops = tiles issued so far
            const int s = (int)(kd % NBUF);
            const unsigned par = (kd / NBUF) & 1u;
            mbar_wait(bar(done, s), par);
            SLM_STAMP(lane == 0, kd, 10);
            if (HAS_OUT && lane == 0) {
                const TileDesc d = desc[s];
                const int b = (int)(d.g / tiles), tile = (int)(d.g % tiles);
                tile_store(tm_out, tile_buf(s), (long long)b * H, H, (long long)tile * ROWB, ROWB, (int)sizeof(R));
                tile_store_commit();
            }
            if (stops < STOPS) {
                const Peek ahead = peek(cur.g < 0 ? total : cur.g + gridDim.x);   // in flight during the staging below
                stage_grey(s, cur);                                       // the group is through this slot's grey rows
                if (HAS_STATS) mbar_wait(bar(taken, s), par);            // the publisher has this slot's descriptor and sums
                SLM_STAMP(lane == 0, kd, 11);
                if (lane == 0) tile_store_wait_read();                   // the store has drained the buffer
                SLM_STAMP(lane == 0, kd, 12);
                sync_warp();
                post(s, cur);
                ++k;
                if (cur.g < 0) ++stops; else cur = resolve(ahead);
                prefetch(cur);
            }
        }
        if (lane == 0) tile_store_wait_all();
        return;
    }

    // ================= compute warps: one column each =================
    constexpr int RA = G::RA;
    const int grp = t / G::GROUP_THREADS;
    const int c = (t % G::GROUP_THREADS) / 32, lane = t % 32;
    const int pair = c >> 1, half = c & 1;
    const bool active = RA == 32 || lane < RA;                      // side B lives in the first RA lanes
    const int pair_bar = 1 + grp * (TC / 2) + pair;                  // named barrier of the column pair (64 threads)
    // byte offset of (row, column c) in the swizzled tile image: side A row lane + 32 p -> my + 2048 p;
    // side B row lane + RA k -> my + 64 RA k (RA is a multiple of 8, so the swizzle term is the lane's in both)
    const unsigned my = (unsigned)lane * 64u + (((unsigned)c * 8u) ^ ((((unsigned)lane >> 1) & 3u) << 4));
    // exchange region of this warp: its half of the rows of the pair's 16-byte chunk
    const unsigned region = (unsigned)(H / 2) * 64u * half;
    const unsigned lm = region + 1024u * lane + (xch_f((unsigned)lane) ^ ((unsigned)pair << 4));
    const unsigned sm = region + (xch_f((unsigned)lane) ^ ((unsigned)pair << 4));
    const cpx<R> w1 = ld_const(static_cast<const cpx<R>*>(a.tw) + lane);       // exp(-2 pi i lane / H)
    // (a run-time 0 the assembler cannot see through: the exchange addresses of the second transform are formed
    //  afresh instead of being kept -- in local memory -- from the first one)
    const unsigned zero = (unsigned)a.B >> 31;
    constexpr bool IN_B = MODE == CGM_GD_POST;                       // the tile already holds a transformed field
    constexpr bool OUT_B = MODE == CGM_STATS_KEEP;                   // the transformed field goes back as it is
    cpx<R> v[32];
    if constexpr (PIPE) {
        // ================= CGM_GD_PIPE: the two groups share every tile =================
        // group 0: tile -> med_output = fft2(...) columns (algorithms.py:84), left in the buffer in side-B order, its eight
        //          column maxima beside it (the publisher warp adds them to the plane's max and arrival count) -- and on
        //          to the next tile;
        // group 1: once every tile of the plane has arrived (they are in flight on the other SMs, at most NBUF items
        //          away), output = |F|^2 * norm / max, the error sum, mask * F * (output - T) and the inverse transform
        //          (algorithms.py:85-88,92).  Same arithmetic, same bits as the two-pass and the fused forms.
        float* const fmx = reinterpret_cast<float*>(raw + G::OFF_FMX);
        if (grp == 0) {
            for (unsigned k = 0;; ++k) {
                const int s = (int)(k % NBUF);
                const unsigned par = (k / NBUF) & 1u;
                unsigned char* const buf = tile_buf(s);
                SLM_STAMP(t == 0, k, 0);
                mbar_wait(bar(full, s), par);
                const TileDesc d = desc[s];
                if (d.g < 0) break;
                SLM_STAMP(t == 0, k, 1);
#pragma unroll
                for (int p = 0; p < RA; ++p) v[p] = *reinterpret_cast<const cpx<R>*>(buf + my + 2048u * p);
                sync_named(pair_bar, 64);                    // the partner holds its column too: the pair's chunk is free
                warp_fft_forward<RA>(v, buf, lm, sm, w1);
                SLM_STAMP(t == 0, k, 2);
                const R m = side_b_max(v, active);
                if (lane == 0) fmx[s * (TC + 2) + c] = m;
                sync_named(pair_bar, 64);                    // the partner is through its exchange: its rows of my column are free
                if (active) {
#pragma unroll
                    for (int q = 0; q < 32; ++q) *reinterpret_cast<cpx<R>*>(buf + my + 64u * RA * q) = v[q];
                }
                mbar_arrive(bar(fwd, s));                    // the publisher warp takes the eight column maxima to the plane's
                SLM_STAMP(t == 0, k, 3);
            }
            return;
        }
        for (unsigned k = 0;; ++k) {
            const int s = (int)(k % NBUF);
            const unsigned par = (k / NBUF) & 1u;
            unsigned char* const buf = tile_buf(s);
            mbar_wait(bar(full, s), par);
            const TileDesc d = desc[s];
            if (d.g < 0) break;
            const int b = (int)(d.g / tiles), tile = (int)(d.g % tiles);
            SLM_STAMP(t == G::GROUP_THREADS, k, 4);
            mbar_wait(bar(fwd, s), par);
            SLM_STAMP(t == G::GROUP_THREADS, k, 5);
#pragma unroll
            for (int q = 0; q < 32; ++q) v[q] = *reinterpret_cast<const cpx<R>*>(buf + my + 64u * RA * q);
            // the plane's other tiles: counted already, or being transformed on other SMs right now (cooperative launch:
            // every CTA is resident).  The time-out only guards against a broken launch.
            if (c == 0 && lane == 0) fmx[s * (TC + 2) + TC] = __uint_as_float(wait_plane_max<true>(a, b, tiles));
            sync_named(10, G::GROUP_THREADS);
            SLM_STAMP(t == G::GROUP_THREADS, k, 6);
            const double pmax = (double)fmx[s * (TC + 2) + TC];
            const R gdk = (R)(d.norm / pmax);
            sync_named(pair_bar, 64);                        // the partner holds its column too: the pair's chunk is free
            R sa = 0;
            const uint8_t* gsrc = grey_buf(s) + (size_t)lane * TC + c;
            const size_t goff = (size_t)b * H * a.W + (size_t)lane * a.W + tile * TC + c;
#pragma unroll
            for (int r0 = 0; r0 < 32; r0 += 8) {
                R tv[8], aux[8];
                side_b_targets<RA, TC>(a, use_t8, active, gsrc, lut_s, goff, r0, tv, aux);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = r0 + i;
                    v[r] = gd_point(v[r], gd_output(cnorm2(v[r]), gdk, d.norm, pmax), tv[i], aux[i], sa);
                }
            }
            if (!active) sa = 0;                             // lanes outside side B hold no points
            Partial p; p.mx = 0; p.a = (double)sa; p.b = 0; p.c = 0;
            p = warp_reduce<FIELDS>(p);
            if (lane == 0) red[s * TC + c] = p;              // (the sequencer reissued this slot only after its sums were taken)
            SLM_STAMP(t == G::GROUP_THREADS, k, 7);
            warp_fft_inverse<RA>(v, buf, lm, sm, w1, active);
            SLM_STAMP(t == G::GROUP_THREADS, k, 8);
            sync_named(pair_bar, 64);                        // the partner is through its exchange: its rows of my column are free
#pragma unroll
            for (int p2 = 0; p2 < RA; ++p2) *reinterpret_cast<cpx<R>*>(buf + my + 2048u * side_a_index<RA>(p2)) = v[p2];
            fence_async_smem();
            mbar_arrive(bar(done, s));
            SLM_STAMP(t == G::GROUP_THREADS, k, 9);
        }
        return;
    }
    for (unsigned k = (unsigned)grp;; k += G::GROUPS) {
        const int s = (int)(k % NBUF);
        const unsigned par = (k / NBUF) & 1u;
        unsigned char* const buf = tile_buf(s);
        mbar_wait(bar(full, s), par);
        const TileDesc d = desc[s];
        if (d.g < 0) break;
        const int b = (int)(d.g / tiles), tile = (int)(d.g % tiles);
        const bool inverse_only = MODE == CGM_COMPLEX && ga.mode_inverse;
        if (IN_B || inverse_only) {
#pragma unroll
            for (int q = 0; q < 32; ++q) v[q] = *reinterpret_cast<const cpx<R>*>(buf + my + 64u * RA * q);
        } else {
#pragma unroll
            for (int p = 0; p < RA; ++p) v[p] = *reinterpret_cast<const cpx<R>*>(buf + my + 2048u * p);
        }
        sync_named(pair_bar, 64);                            // the partner holds its column too: the pair's chunk is free
        if (!IN_B && !inverse_only) warp_fft_forward<RA>(v, buf, lm, sm, w1);

        // ---- CGM_GD_FUSED: max |F|^2 of the whole plane (algorithms.py:86), across the CTAs holding its tiles ----
        double plane_max = d.imax;
        if (FUSED) {
            const R m = side_b_max(v, active);
            float* const fmx = reinterpret_cast<float*>(raw + G::OFF_FMX) + s * (TC + 2);
            if (lane == 0) fmx[c] = m;
            sync_named(9 + grp, G::GROUP_THREADS);
            if (c == 0 && lane == 0) {
                add_tile_max<TC>(a, b, fmx);
                fmx[TC] = __uint_as_float(wait_plane_max<false>(a, b, tiles));   // the plane's other tiles are in flight on other SMs
            }
            sync_named(9 + grp, G::GROUP_THREADS);
            plane_max = (double)fmx[TC];
#pragma unroll
            for (int r = 0; r < 32; ++r) opaque(v[r]);       // (or the 32 |F|^2 above are kept -- spilled -- for the step below)
        }
        // ---- pointwise step and per-thread sums on side B (see col_group_kernel) ----
        R mx = 0, sa = 0, sb = 0, sc = 0;
        if (MODE == CGM_GS || IS_GD) {
            const R s0r = (R)d.scale;
            const R gdk = (R)(d.norm / plane_max);
            const uint8_t* gsrc = grey_buf(s) + (size_t)lane * TC + c;
            const size_t goff = (size_t)b * H * a.W + (size_t)lane * a.W + tile * TC + c;
#pragma unroll
            for (int r0 = 0; r0 < 32; r0 += 8) {
                R tv[8], aux[8];
                side_b_targets<RA, TC>(a, use_t8, active, gsrc, lut_s, goff, r0, tv, aux);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = r0 + i;
                    const R m2 = cnorm2(v[r]);
                    if (MODE == CGM_GS) {
                        gs_sums(m2, tv[i], s0r, mx, sa, sb, sc);
                        replace_amplitude(v[r], m2, aux[i]);
                    } else {
                        v[r] = gd_point(v[r], gd_output(m2, gdk, d.norm, plane_max), tv[i], aux[i], sa);
                    }
                }
            }
        } else if (IS_STATS) {
#pragma unroll
            for (int r = 0; r < 32; ++r) mx = fmax(mx, cnorm2(v[r]));
        } else {
            const R sc_out = (R)ga.scale;
#pragma unroll
            for (int r = 0; r < 32; ++r) v[r] = cscale(v[r], sc_out);
        }
        if (HAS_STATS) {                                     // this column's sums -> shared memory, for the publisher
            if (!active) { mx = 0; sa = 0; sb = 0; sc = 0; }             // lanes outside side B hold no points
            Partial p; p.mx = (double)mx; p.a = (double)sa; p.b = (double)sb; p.c = (double)sc;
            p = warp_reduce<FIELDS>(p);
            if (lane == 0) red[s * TC + c] = p;             // (the sequencer reissued this slot only after its sums were taken)
        }
        constexpr bool SECOND = MODE == CGM_GS || IS_GD;
        if (SECOND) warp_fft_inverse<RA>(v, buf, lm + zero, sm + zero, w1, active);
        else if (inverse_only) warp_fft_inverse<RA>(v, buf, lm, sm, w1, active);
        if (HAS_OUT) {
            sync_named(pair_bar, 64);                        // the partner is through its exchange: its rows of my column are free
            if (OUT_B || (MODE == CGM_COMPLEX && !inverse_only)) {
                if (active) {
#pragma unroll
                    for (int q = 0; q < 32; ++q) *reinterpret_cast<cpx<R>*>(buf + my + 64u * RA * q) = v[q];
                }
            } else {
#pragma unroll
                for (int p = 0; p < RA; ++p) *reinterpret_cast<cpx<R>*>(buf + my + 2048u * side_a_index<RA>(p)) = v[p];
            }
            fence_async_smem();
        }
        mbar_arrive(bar(done, s));
    }
}

}  // namespace slm
