// Warp-specialised persistent column kernels (sm_100a).
//
// One resident CTA per SM walks the column tiles ([H rows][TC columns]) round-robin:
//   * a PRODUCER warp streams tiles in and out with TMA (tma.cuh): the next tile's field data is
//     loaded (32B/64B-swizzled) while the current one is transformed, the tile's 8-bit target rows
//     are staged beside it, and finished tiles are written back with a TMA store;
//   * the COMPUTE warps own whole columns: the M = H/E threads of a column are consecutive, so a
//     column's transform synchronises on a named barrier over its own warps only.  Column groups
//     run out of phase with each other, which hides barrier, shared-memory and reduction latency
//     that a CTA-wide lock-step exposes (ncu: profiles/).
// Hand-over is by mbarriers: full[s] (tile s landed), done[s] (every compute thread has written its
// results into tile s and fenced them for the async proxy).  A tile's buffer is reused for its own
// output, so two tile buffers suffice.
#pragma once
#include "passes.cuh"

namespace slm {

// Optional device timeline (-DSLM_TRACE): lane 0 of compute warp 0 / of the producer warp stamps
// globaltimer at the phase boundaries of each tile into slm_trace_buf[cta][tile][event].
#if defined(SLM_TRACE) && !defined(SLM_EMULATE)
SLM_DEV void trace_stamp(unsigned long long* buf, bool who, unsigned k, int ev) {
    if (buf && who && k < 64) {
        unsigned long long tns;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tns));
        buf[((size_t)blockIdx.x * 64 + k) * 16 + ev] = tns;
    }
}
#define SLM_STAMP(who, k, ev) trace_stamp(ga.trace, who, k, ev)
#else
#define SLM_STAMP(who, k, ev)
#endif

constexpr int lines_per_group(int m) { return m % 32 == 0 ? 1 : (m % 16 == 0 ? 2 : (m % 8 == 0 ? 4 : 8)); }

template <typename R, int H> struct ColGroupGeom {
    using P = ColPlan<H>;
    using CG = ColGeom<R, H>;
    static constexpr int E = P::E, M = P::M, TC = CG::TC;
    static constexpr int COMPUTE = TC * M;                        // compute threads
    static constexpr int NW = COMPUTE / 32;                       // compute warps
    // producer warp-group (4 warps): lane 0 drives TMA, warps 0-2 stage the 8-bit target rows, warp 3 is the
    // PUBLISHER: it takes each finished tile's partial sums to global memory and closes a plane's iteration
    static constexpr int PRODUCERS = 128;
    static constexpr int COPIERS = 96;
    static constexpr int THREADS = COMPUTE + PRODUCERS;
    static constexpr int ROWB = TC * (int)sizeof(cpx<R>);         // bytes of one tile row
    // PAIRED: a warp covers 16 rows x 2 adjacent columns (lanes 0-15 / 16-31).  With 64-byte swizzled tile rows
    // that makes the tile reads/writes and the grey-level reads bank-conflict free (one column alone is 2-way:
    // 16-byte swizzle chunks cannot separate the two 8-byte halves); the sync group is then the column pair.
    static constexpr bool PAIRED = (M % 16 == 0) && (TC % 2 == 0);
    static constexpr int LPG = PAIRED ? 2 : lines_per_group(M);
    static constexpr int GROUPS = TC / LPG;
    static constexpr int GROUP_THREADS = LPG * M;
    static constexpr size_t TILE = (size_t)H * ROWB;
    static constexpr size_t XCH = (size_t)TC * P::NP * sizeof(cpx<R>);
    static constexpr size_t GREY = (size_t)H * TC;
    // [tile0][tile1][exchange][grey0][grey1][lut][red 2 x NW][counters][barriers]
    static constexpr size_t OFF_XCH = 2 * TILE;
    static constexpr size_t OFF_GREY = OFF_XCH + XCH;
    static constexpr size_t OFF_LUT = OFF_GREY + 2 * GREY;
    static constexpr size_t OFF_RED = OFF_LUT + 256 * sizeof(R);
    static constexpr size_t OFF_CNT = OFF_RED + 2 * 32 * sizeof(Partial);
    static constexpr size_t OFF_TOT = OFF_CNT + 16;                // Partial tile_total[2]
    static constexpr size_t OFF_BAR = OFF_TOT + 2 * sizeof(Partial);
    static constexpr size_t OFF_TW = OFF_BAR + 6 * 32;             // column twiddle table, when it fits
    static constexpr size_t TW_BYTES = (size_t)H * sizeof(cpx<R>);
    static constexpr bool TW_SHARED = OFF_TW + TW_BYTES <= 232448; // 227 KB of shared memory per CTA
    static constexpr size_t SMEM = OFF_TW + (TW_SHARED ? TW_BYTES : 0);
    // P::ONE_STAGE: the radix-5 and composite middle stages (1152, 1280, 1920) hold up to QMAX x radix points per thread
    // beside the tile's grey levels and sums; under this kernel's register cap (128 at 448 threads, 96 at 608) they
    // spilled 200-700 bytes per thread, so those lengths take the spill-free one-CTA-per-tile kernel instead.
    static constexpr bool OK = (ROWB == 64 || ROWB == 32) && COMPUTE % 32 == 0 && TC % LPG == 0 && GROUPS <= 14 &&
                               H % 32 == 0 && NW <= 32 && OFF_TW <= 232448 &&   // (two tile buffers + exchange must fit)
                               P::ONE_STAGE;
    using Sync = GroupSync<GROUP_THREADS>;
};

// One lane's share of a tile of the 8-bit target: rows lane, lane+32, ... (TC bytes each).  Every
// load is issued before the first store so the whole tile is one DRAM round trip.
template <int TC> struct GreyWord;
template <> struct GreyWord<8> { using type = uint2; };
template <> struct GreyWord<4> { using type = unsigned; };
template <> struct GreyWord<2> { using type = unsigned short; };
template <> struct GreyWord<1> { using type = unsigned char; };
template <int TC, int H, int NT, int CHMAX = 16> SLM_DEV void copy_grey_tile(const uint8_t* src, size_t pitch, uint8_t* dst, int lane) {
    using Wd = typename GreyWord<TC>::type;
    constexpr int ROWS = (H + NT - 1) / NT, CH = ROWS < CHMAX ? ROWS : CHMAX;
#pragma unroll 1
    for (int r0 = 0; r0 < ROWS; r0 += CH) {
        Wd w[CH];
#pragma unroll
        for (int i = 0; i < CH; ++i) {
            const int row = lane + NT * (r0 + i);
            if (row < H) w[i] = ld_ro(reinterpret_cast<const Wd*>(src + (size_t)row * pitch));
        }
#pragma unroll
        for (int i = 0; i < CH; ++i) {
            const int row = lane + NT * (r0 + i);
            if (row < H) *reinterpret_cast<Wd*>(dst + (size_t)row * TC) = w[i];
        }
    }
}

template <typename R, int H, int MODE>
SLM_GLOBAL void SLM_LAUNCH_BOUNDS((ColGroupGeom<R, H>::THREADS), 1)
col_group_kernel(ColGroupArgs ga, const SLM_GRID_CONSTANT TileMap tm_in, const SLM_GRID_CONSTANT TileMap tm_out) {
    using G = ColGroupGeom<R, H>;
    using P = ColPlan<H>;
    constexpr int E = G::E, M = G::M, TC = G::TC, ROWB = G::ROWB, CS = (int)sizeof(cpx<R>);
    constexpr bool HAS_T = MODE == CGM_GS || MODE == CGM_GD || MODE == CGM_GD_POST;
    constexpr bool HAS_OUT = MODE != CGM_STATS;
    constexpr bool IS_GD = MODE == CGM_GD || MODE == CGM_GD_POST;
    constexpr bool IS_STATS = MODE == CGM_STATS || MODE == CGM_STATS_KEEP;
    const ColArgs& a = ga.c;
    SLM_DYN_SMEM(raw);
    unsigned char* const tile0 = raw;
    unsigned char* const tile1 = raw + G::TILE;
    uint8_t* const grey0 = raw + G::OFF_GREY;
    uint8_t* const grey1 = grey0 + G::GREY;
    R* const lut_s = reinterpret_cast<R*>(raw + G::OFF_LUT);
    Partial* const red = reinterpret_cast<Partial*>(raw + G::OFF_RED);
    unsigned* const cnt = reinterpret_cast<unsigned*>(raw + G::OFF_CNT);
    TileBarrier* const full = reinterpret_cast<TileBarrier*>(raw + G::OFF_BAR);       // [2]
    TileBarrier* const done = full + 2;                                                // [2]
    TileBarrier* const pubfree = full + 4;                                             // [2] tile_total[s] has been taken
    Partial* const tile_total = reinterpret_cast<Partial*>(raw + G::OFF_TOT);          // [2]

    const int t = threadIdx.x;
    const int tiles = a.W / TC;
    const long long total = (long long)a.B * tiles;
    const bool use_t8 = HAS_T && a.T8 != nullptr;
    griddep_launch();                                 // programmatic dependent launch: see griddep_wait below
    if (t == 0) {
        mbar_init(full + 0, use_t8 ? 1u + G::COPIERS : 1u); mbar_init(full + 1, use_t8 ? 1u + G::COPIERS : 1u);
        mbar_init(pubfree + 0, 1u); mbar_init(pubfree + 1, 1u);
        mbar_init(done + 0, (unsigned)G::COMPUTE); mbar_init(done + 1, (unsigned)G::COMPUTE);
        cnt[0] = 0; cnt[1] = 0;
        mbar_fence_init();
    }
    if (use_t8) {
        const R* lut = static_cast<const R*>(a.lut);
        for (int i = t; i < 256; i += G::THREADS) lut_s[i] = ld_ro(lut + i);
    }
    if (G::TW_SHARED) {                                     // twiddles next to the data: no global round trip inside the transforms
        cpx<R>* tws = reinterpret_cast<cpx<R>*>(raw + G::OFF_TW);
        const cpx<R>* twg = static_cast<const cpx<R>*>(a.tw);
        for (int i = t; i < H; i += G::THREADS) tws[i] = ld_const(twg + i);
    }
    // everything above (barriers, tables: constant inputs) overlapped the tail of the previous pass; from here
    // on the field, the per-plane state and the partial sums of that pass are read
    griddep_wait();
    sync_cta();
    auto rests = [&](int b) { return MODE != CGM_COMPLEX && !ga.all_planes && ld_cg(&a.stats[b].done) != 0; };

    constexpr bool HAS_STATS = MODE != CGM_COMPLEX;
    constexpr int FIELDS = MODE == CGM_GS ? F_ALL : (IS_GD ? F_A : F_MX);
    if (t >= G::COMPUTE + G::COPIERS) {
        // ================= publisher warp =================
        if (!HAS_STATS) return;
        const int lane = t - G::COMPUTE - G::COPIERS;
        const double hw = (double)H * (double)a.W;
        unsigned k = 0;
        for (long long g = blockIdx.x; g < total; g += gridDim.x) {
            const int b = (int)(g / tiles), tile = (int)(g % tiles);
            if (rests(b)) continue;
            const int s = (int)(k & 1u);
            PlaneStats* st = a.stats + b;
            // values the closing formulas need, read before this launch can change them
            const double s0 = ld_cg(&st->scale), norm = ld_ro(a.norm + b);
            mbar_wait(done + s, (k >> 1) & 1u);              // every compute thread is through tile k (totals are in shared memory)
            Partial q = tile_total[s];
            shfl_idx(0u, 0);                                 // all lanes hold their copy before the slot is released
            if (lane == 0) mbar_arrive(pubfree + s);
            Partial* plane_partials = a.partial + (size_t)b * tiles;
            if (ga.defer_close) {                            // the closing kernel behind this launch sums the tiles (col_warp.cuh)
                if (lane == 0) plane_partials[tile] = q;
                ++k;
                continue;
            }
            unsigned ticket = 0;
            if (lane == 0) ticket = publish_partial(q, plane_partials, tile, tiles, a.counter + b);
            Partial tot;
            if (collect_if_last<FIELDS>(ticket, lane, plane_partials, tiles, tot) && lane == 0) {
                if (IS_STATS) {
                    st->imax = tot.mx; st->scale = norm / tot.mx;
                } else {
                    double err;
                    if (MODE == CGM_GS) {
                        const double sN = norm / tot.mx;                 // algorithms.py:37
                        const double s0u = (double)(R)s0;                // the scale the tiles actually used
                        const double dl = (s0u != 0.0) ? sN / s0u - 1.0 : 0.0;
                        err = (tot.a + 2.0 * dl * tot.b + dl * dl * tot.c) / hw;   // == sum((s*I - T)^2)/HW, :38,:162
                        st->imax = tot.mx; st->scale = sN;
                    } else {
                        err = tot.a / hw;                                // algorithms.py:92
                    }
                    const int it = st->iters;
                    a.err_curve[(size_t)b * a.max_loops + it] = err;
                    st->err = err; st->iters = it + 1;
                    st->done = !(err > a.tolerance);                     // loop condition, algorithms.py:29,83
                }
            }
            ++k;
        }
        return;
    }
    if (t >= G::COMPUTE) {
        // ================= producer warps (TMA + target staging) =================
        const int lane = t - G::COMPUTE;
        auto issue = [&](long long g, int s, unsigned kk) {
            const int b = (int)(g / tiles), tile = (int)(g % tiles);
            if (lane == 0) {
                SLM_STAMP(true, kk, 8);
                tile_store_wait_read();          // the store that last read this buffer has drained it
                SLM_STAMP(true, kk, 9);
                tile_load(tm_in, s ? tile1 : tile0, full + s, (long long)b * H, H, (long long)tile * ROWB, ROWB, (int)sizeof(R));
            }
            if (use_t8) {
                sync_named(15, G::COPIERS);      // lane 0's wait (the store has drained) covers the grey buffer too
                const uint8_t* src = a.T8 + (size_t)b * H * a.W + (size_t)tile * TC;
                uint8_t* dst = s ? grey1 : grey0;
                copy_grey_tile<TC, H, G::COPIERS>(src, (size_t)a.W, dst, lane);
                mbar_arrive(full + s);
                SLM_STAMP(lane == 0, kk, 10);
            }
        };
        long long g = blockIdx.x;
        while (g < total && rests((int)(g / tiles))) g += gridDim.x;
        if (g < total) issue(g, 0, 0);
        unsigned k = 0;
        while (g < total) {
            long long gn = g + gridDim.x;
            while (gn < total && rests((int)(gn / tiles))) gn += gridDim.x;
            const int s = (int)(k & 1u);
            if (gn < total) issue(gn, s ^ 1, k + 1);
            SLM_STAMP(lane == 0, k, 11);
            mbar_wait(done + s, (k >> 1) & 1u);
            SLM_STAMP(lane == 0, k, 12);
            if (HAS_OUT && lane == 0) {
                const int b = (int)(g / tiles), tile = (int)(g % tiles);
                tile_store(tm_out, s ? tile1 : tile0, (long long)b * H, H, (long long)tile * ROWB, ROWB, (int)sizeof(R));
                tile_store_commit();
                SLM_STAMP(true, k, 13);
            }
            g = gn;
            ++k;
        }
        if (lane == 0) tile_store_wait_all();
        return;
    }

    // ================= compute warps =================
    const int lane = t % 32, warp = t / 32;
    int c, j;
    if (G::PAIRED) {                                   // pair group pg: M/16 warps, each 16 rows x 2 columns
        const int pg = t / (2 * M), w = (t % (2 * M)) / 32;
        c = 2 * pg + (lane >> 4);
        j = 16 * w + (lane & 15);
    } else {
        c = t / M; j = t % M;
    }
    const typename G::Sync sync{1 + c / G::LPG};
    cpx<R>* const line = reinterpret_cast<cpx<R>*>(raw + G::OFF_XCH) + (size_t)c * P::NP;
    const cpx<R>* tw = G::TW_SHARED ? reinterpret_cast<const cpx<R>*>(raw + G::OFF_TW) : static_cast<const cpx<R>*>(a.tw);
    using Sy = typename G::Sync;
    cpx<R> v[E];
    unsigned k = 0;
    // Per-plane scalars (rest flag, previous scale, max, norm) of a tile are requested ONE TILE AHEAD and
    // only looked at in the next trip of the loop, so their L2 round trips overlap a whole tile of work.
    struct PlaneInfo { int done; double scale, imax, norm; };
    auto fetch_info = [&](long long gg) {
        PlaneInfo pi; pi.done = 1; pi.scale = 0; pi.imax = 0; pi.norm = 0;
        if (gg < total) {
            const int bb = (int)(gg / tiles);
            pi.done = 0;
            if (MODE != CGM_COMPLEX) {
                const PlaneStats* ps = a.stats + bb;
                pi.done = ga.all_planes ? 0 : ld_cg(&ps->done);
                if (MODE == CGM_GS || IS_GD) { pi.scale = ld_cg(&ps->scale); pi.imax = ld_cg(&ps->imax); pi.norm = ld_ro(a.norm + bb); }
            }
        }
        return pi;
    };
    PlaneInfo nxt = fetch_info(blockIdx.x);
    for (long long g = blockIdx.x; g < total; g += gridDim.x) {
        const int b = (int)(g / tiles), tile = (int)(g % tiles);
        const PlaneInfo info = nxt;
        nxt = fetch_info(g + gridDim.x);
        if (info.done) continue;
        const int s = (int)(k & 1u);
        unsigned char* const buf = s ? tile1 : tile0;
        const double s0 = info.scale, imax = info.imax, norm = info.norm;
        SLM_STAMP(t == 0, k, 0);
        mbar_wait(full + s, (k >> 1) & 1u);
        SLM_STAMP(t == 0, k, 1);
#pragma unroll
        for (int r = 0; r < E; ++r)
            v[r] = *reinterpret_cast<const cpx<R>*>(buf + tile_swizzle<ROWB>((unsigned)((j + r * M) * ROWB + c * CS)));
        R tv[E], aux[E];
        if (HAS_T && !use_t8) {                                   // real-valued targets: planes in global memory
            const size_t off = (size_t)b * H * a.W + (size_t)j * a.W + tile * TC + c;
            const R* T = static_cast<const R*>(a.Treal) + off;
            const R* Q = static_cast<const R*>(a.plane2) + off;
#pragma unroll
            for (int r = 0; r < E; ++r) { tv[r] = ld_ro(T + (size_t)r * M * a.W); aux[r] = ld_ro(Q + (size_t)r * M * a.W); }
        }
        if (MODE == CGM_COMPLEX && ga.mode_inverse) line_fft<R, H, +1, 1, Sy, G::TW_SHARED, column_points(H)>(v, line, j, tw, sync);
        else if (MODE != CGM_GD_POST) line_fft<R, H, -1, 1, Sy, G::TW_SHARED, column_points(H)>(v, line, j, tw, sync);

        SLM_STAMP(t == 0, k, 2);
        // ---- pointwise step and per-thread sums ----
        R mx = 0, sa = 0, sb = 0, sc = 0;
        const R s0r = (R)s0;
        if (MODE == CGM_GS || IS_GD) {
            if (use_t8) {                                          // grey level and its table entry, both from shared memory
                const uint8_t* gsrc = (s ? grey1 : grey0) + (size_t)j * TC + c;
#pragma unroll
                for (int r = 0; r < E; ++r) { const int gl = gsrc[(size_t)r * M * TC]; tv[r] = (R)gl; aux[r] = lut_s[gl]; }
            }
            const R gdk = sizeof(R) == 8 ? (R)0 : (R)(norm / imax);
#pragma unroll
            for (int r = 0; r < E; ++r) {
                const R m2 = cnorm2(v[r]);
                if (MODE == CGM_GS) {                                 // algorithms.py:33,36-38 (see col_pass_tile)
                    const R u = s0r * m2, d = u - tv[r];
                    mx = fmax(mx, m2); sa += d * d; sb += d * u; sc += u * u;
                    v[r] = (m2 == (R)0) ? mk<R>(copysign(aux[r], v[r].x), (R)0) : cscale(v[r], aux[r] * rsqrt_fast(m2));
                } else {                                              // algorithms.py:85-88,92
                    R I;
                    if (sizeof(R) == 8) I = (R)(((double)m2 * norm) / imax);
                    else I = m2 * gdk;
                    const R d = I - tv[r];
                    sa += d * d;
                    v[r] = cscale(cscale(v[r], aux[r]), d);
                }
            }
        } else if (IS_STATS) {
#pragma unroll
            for (int r = 0; r < E; ++r) mx = fmax(mx, cnorm2(v[r]));
        } else {
            const R sc_out = (R)ga.scale;
#pragma unroll
            for (int r = 0; r < E; ++r) v[r] = cscale(v[r], sc_out);
        }

        SLM_STAMP(t == 0, k, 3);
        // ---- tile reduction without a CTA barrier: the last warp to arrive sums the warps' partials and leaves
        //      the tile total in shared memory for the publisher warp (nothing global on the compute path) ----
        if (HAS_STATS) {
            Partial p; p.mx = (double)mx; p.a = (double)sa; p.b = (double)sb; p.c = (double)sc;
            p = warp_reduce<FIELDS>(p);
            unsigned arrived = 0;
            if (lane == 0) {
                red[s * 32 + warp] = p;
                fence_block();
                arrived = atomic_add_shared(cnt + s, 1u);
            }
            arrived = shfl_idx(arrived, 0);
            if (arrived == (unsigned)G::NW - 1) {
                fence_block();
                Partial q; q.mx = 0; q.a = 0; q.b = 0; q.c = 0;
                if (lane < G::NW) q = red[s * 32 + lane];
                q = warp_reduce<FIELDS>(q);
                if (lane == 0) {
                    cnt[s] = 0;
                    if (k >= 2) mbar_wait(pubfree + s, ((k >> 1) - 1u) & 1u);   // the publisher has taken this slot's previous total
                    tile_total[s] = q;
                }
            }
        }

        SLM_STAMP(t == 0, k, 4);
        if (MODE == CGM_GS || IS_GD) line_fft<R, H, +1, 1, Sy, G::TW_SHARED, column_points(H)>(v, line, j, tw, sync);
        SLM_STAMP(t == 0, k, 5);
        if (HAS_OUT) {
#pragma unroll
            for (int r = 0; r < E; ++r)
                *reinterpret_cast<cpx<R>*>(buf + tile_swizzle<ROWB>((unsigned)((j + r * M) * ROWB + c * CS))) = v[r];
            fence_async_smem();
        }
        mbar_arrive(done + s);
        SLM_STAMP(t == 0, k, 6);
        ++k;

    }
}

}  // namespace slm
