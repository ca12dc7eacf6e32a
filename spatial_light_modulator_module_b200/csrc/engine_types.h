// Types shared by the pass kernels (passes.cuh), their per-line-length instantiations
// (gen/line_*.cu) and the engine (engine.cu).
#pragma once
#include "cuda_compat.h"

namespace slm {

enum Precision { PREC_F32 = 0, PREC_F64 = 1 };
// ALG_GSW: weighted GS (per-pixel amplitude feedback, DESIGN.md); ALG_GSW_STATS selects its iteration-0 pre-pass
// (col_gsw_stats_kernel) in LineTable::col_pass.  ALG_MP / ALG_MPGD: the SLM-plane pass of multi-plane GS / GD
// (row_multiplane_kernel) in LineTable::row_pass; their Fourier-plane side is GS's / GD's.
enum Algorithm { ALG_GS = 0, ALG_GD = 1, ALG_GSW = 2, ALG_GSW_STATS = 3, ALG_MP = 4, ALG_MPGD = 5 };

// ---- per-plane loop state, device resident --------------------------------------------------
// Written only by the last column tile of a plane to finish a Fourier-plane pass.
struct PlaneStats {
    double imax;     // max |C|^2 of the most recent Fourier-plane pass (algorithms.py:37,86)
    double scale;    // norm / imax of that pass
    double err;      // last error value (algorithms.py:38,92)
    int iters;       // completed iterations == len(error_evolution)
    int done;        // loop condition `error > tolerance` has failed (algorithms.py:29,83)
};

// Per-tile reduction record (deterministic two-stage reduce: tile -> plane).
struct Partial { double mx, a, b, c; };

// What the last tile of a plane closes (close_plane, passes.cuh): the max and the scale only, or a GS / GD iteration.
enum PlaneClose { CLOSE_MAX = 0, CLOSE_GS = 1, CLOSE_GD = 2 };

// ---- SLM-plane (row) pass ----------------------------------------------------------------------
enum RowSource {
    ROW_FROM_Y = 0,      // rows of Y hold the column-inverse-transformed field: finish the ifft2
    ROW_FROM_A32 = 1,    // complex64 field A (reference's first ifft2, algorithms.py:27): phasor in fp32
    ROW_FROM_FIELD = 2,  // caller-supplied B of iteration 0 (GS) / x itself (GD first pass)
    ROW_FROM_A = 3,      // complex<R> field A: phasor in R (targets whose first ifft2 is complex128)
};

struct RowArgs {
    int B, H;
    int source;              // RowSource
    int final_pass;          // 1: emit the hologram (phase) and stop; no forward transform
    const void* Y;           // complex<R> [B][H][W]
    void* X;                 // complex<R> [B][H][W]
    const void* field;       // complex<R> [B][H][W]   (ROW_FROM_FIELD, GS)
    const void* A32;         // complex<float> [B][H][W] (ROW_FROM_A32)
    void* x;                 // GD: complex<R> [B][H][W], updated in place
    const void* inc;         // real<R> [H][W] illumination amplitude or null (uniform)
    const double* lr;        // GD: learning rate of iteration k at lr[k]
    double inv_hw;           // 1/(H*W): scipy's ifft2 normalisation (read by GD only); multi-plane GD: 1/(K*H*W)
    const PlaneStats* stats;
    double* hologram;        // [B][H][W], final pass
    const void* tw;          // complex<R> [W] row twiddles exp(-2 pi i q / W)
    // multi-plane GS and GD (ALG_MP, ALG_MPGD); appended so that the offsets the other kernels read stay where they
    // were.  B counts holograms, plane k of hologram g is plane g * planes + k of Y, X and stats; field (ROW_FROM_FIELD),
    // x (GD) and hologram hold one plane per hologram.
    int planes;              // K, 1..8
    int lens_mask;           // bit k: plane k has a defocus (alpha_k != 0); a clear bit skips the products with L_k
    const void* lens_y;      // complex<R> [K][H]: exp(i alpha_k (y - H/2)^2)
    const void* lens_x;      // complex<R> [K][W]: exp(i alpha_k (x - W/2)^2);  L_k(y, x) = lens_y[k][y] * lens_x[k][x]
};

// ---- Fourier-plane (column) pass -----------------------------------------------------------------
struct ColArgs {
    int B, W;
    const void* X;           // complex<R> [B][H][W]
    void* Y;                 // complex<R> [B][H][W]
    const uint8_t* T8;       // uint8 target [B][H][W] or null
    const void* Treal;       // real<R> target (when T8 == null)
    const void* plane2;      // real<R>: GS |sqrt(T)| plane, GD mask plane (when T8 == null)
    const void* lut;         // R[256]: GS amplitude / GD mask by grey level (when T8 != null)
    const double* norm;      // [B] amax(T)
    PlaneStats* stats;       // [B]
    Partial* partial;        // [B][W / TC]
    unsigned* counter;       // [B] zero before first use; self-resetting
    double* err_curve;       // [B][max_loops]
    int max_loops;
    double tolerance;
    double inv_hw;
    const void* tw;          // complex<R> [H] column twiddles
    int skip_forward;        // col_pass_kernel<GD>: X already holds the column-transformed field (max pass with `keep`)
    unsigned* fused_max;     // one-pass GD forms: [max_planes] pairs {bit pattern of the plane's running max |F|^2, tiles that have
                             // contributed} (8-byte aligned, 0 between launches) + the time-out flag behind them (col_warp.cuh)
    int max_planes;
    // weighted GS (ALG_GSW, ALG_GSW_STATS); appended so that the offsets the other kernels read stay where they were
    void* weights;           // real<R> [B][H][W]: w_{k-1} in, w_k out
    const double* target_sum;   // [B] sum(T), the signal energy S_T
    double* signal_sum;      // [B] P = sum of |C|^2 over {T > 0} of the latest Fourier-plane pass (written by the last tile)
    double* signal_partial;  // [B][W / TC] per-tile partial sums of P
    double weight_limit;     // c >= 1: weights are clamped to [1/c, c]
};

// ---- warp-specialised persistent column kernel (col_groups.cuh) ---------------------------------------
enum ColGroupMode {
    CGM_GS = 0,       // Fourier-plane step of GS      (== col_pass_kernel<GS>)
    CGM_STATS = 2,    // forward transform, max |C|^2  (== col_plain_kernel OUT_STATS)
    CGM_COMPLEX = 3,  // plain transform, complex out  (== col_plain_kernel OUT_COMPLEX)
    CGM_STATS_KEEP = 4,  // CGM_STATS that also writes the transformed field back (GD: F = fft2(b) kept in X)
    CGM_GD_POST = 5,     // Fourier-plane step of GD on an already transformed field (== col_pass_kernel<GD> with skip_forward)
    CGM_GD_FUSED = 6,    // the GD step that takes the plane's max ITSELF: every tile of a plane is in flight at once (grid = a
                         // multiple of the tiles per plane, all CTAs resident), tiles meet at a per-plane counter between
                         // the forward transform and the pointwise step (warp-per-column kernel only)
    CGM_GD_PIPE = 7,     // CGM_GD_FUSED for any batch, on every SM: the CTA's two compute groups split the tile's work -- one
                         // forward-transforms tile after tile (and feeds the planes' maxima), the other takes each tile on once
                         // its plane's maximum is complete -- so nobody idles while a plane's tiles meet.  Cooperative launch.
};
SLM_HOSTDEV constexpr bool cgm_is_gd(int m) { return m == CGM_GD_POST || m == CGM_GD_FUSED || m == CGM_GD_PIPE; }
SLM_HOSTDEV constexpr bool cgm_is_stats(int m) { return m == CGM_STATS || m == CGM_STATS_KEEP; }
SLM_HOSTDEV constexpr bool cgm_has_target(int m) { return m == CGM_GS || cgm_is_gd(m); }      // reads the target and its table
SLM_HOSTDEV constexpr int cgm_close(int m) { return m == CGM_GS ? CLOSE_GS : (cgm_is_gd(m) ? CLOSE_GD : CLOSE_MAX); }
struct ColGroupArgs {
    int mode_inverse;        // CGM_COMPLEX: transform direction
    int all_planes;          // 1: also planes whose loop has ended (the transform kept for the final intensity pass)
    int defer_close;         // 1: the pass only stores its tiles' partial sums; a one-warp-per-plane kernel launched behind it
                             // closes the planes' iteration (warp-per-column kernel, large batches: keeps fences and atomics
                             // out of the tile pipeline)
    double scale;            // CGM_COMPLEX: output scale
    unsigned long long* trace;   // -DSLM_TRACE builds: [ctas][64 tiles][16 events] globaltimer stamps, else null
    ColArgs c;               // loop arguments; B, W, stats, partial, counter, norm, tw are used by every mode
};

// ---- plain transforms / setup / preview ------------------------------------------------------
enum PlainRowInput {
    IN_COMPLEX = 0,          // complex<R> plane
    IN_LUT_U8 = 1,           // real: lut[T8]   (GS setup: float16-rounded sqrt, SURVEY A.1)
    IN_REAL = 2,             // real<R> plane
    IN_PHASE = 3,            // exp(i * phase), phase double plane (generate_hologram.py:25)
};
struct PlainRowArgs {
    int B, H;
    int input;               // PlainRowInput
    int inverse;
    int block_in, block_out; // 0: plain [row][W] layout; else the slab-exchange layout of width block_* (slab.cuh)
    const void* in;          // complex<R> / real<R> / double, by `input`
    const uint8_t* T8;
    const void* lut;         // R[256]
    void* out;               // complex<R> [B][H][W]
    const void* tw;
};
enum PlainColOutput {
    OUT_COMPLEX = 0,         // write the transformed plane (scaled by `scale`)
    OUT_STATS = 1,           // only max |C|^2 -> stats[b].imax / .scale
    OUT_INTENSITY_GS = 2,    // |C|^2 * stats.scale                        (algorithms.py:36-37)
    OUT_INTENSITY_GD = 3,    // (|C|^2 * norm) / imax                      (algorithms.py:85-86)
    OUT_INTENSITY_PREVIEW = 4,  // (|C|^2 / imax) * norm                  (generate_hologram.py:26-29)
};
struct PlainColArgs {
    int B, W;
    int output;              // PlainColOutput
    int inverse;
    int skip_fft;            // intensity outputs: `in` already holds the column-transformed field
    int keep;                // OUT_STATS: also write the transformed field to `out` (GD: the gradient pass starts from it)
    double scale;            // OUT_COMPLEX: multiply results (1/(HW) for ifft2)
    const void* in;          // complex<R> [B][H][W]
    void* out;               // complex<R> [B][H][W] or double [B][H][W]
    const double* norm;      // [B]
    PlaneStats* stats;
    Partial* partial;
    unsigned* counter;
    const void* tw;
};

enum RowFourierMode {
    RF_GS = 0,               // GS: finish fft2, amplitude replacement + error sums, start ifft2 (algorithms.py:31-38)
    RF_GD_MAX = 1,           // GD: finish fft2 (kept, written to `out`), max |F|^2 per line (algorithms.py:84-86)
    RF_GD_POST = 2,          // GD: on the kept transform: output, error sum, mask*F*(output-T), start ifft2 (algorithms.py:85-88,92)
};
// ---- Fourier-plane step on ROWS of a transposed slab (slab-decomposed 2-D transform, slab.cuh) -----------
struct RowFourierArgs {
    int rows;                // local lines (columns of the global plane owned by this rank)
    int block_w;             // exchange-layout block width (0: plain [rows][W])
    const void* in;          // complex<R>: lines after the first transform + exchange
    void* out;               // complex<R>: lines ready for the return exchange
    const uint8_t* T8;       // target, same layout as `in`
    const void* lut;         // R[256] amplitude by grey level
    const PlaneStats* stats; // the context's loop state (slm_rows_close): RF_GS reads the previous iteration's scale
                             // (algorithms.py:37), RF_GD_POST this iteration's norm / max and max
    int mode;                // RowFourierMode
    double norm;             // RF_GD_POST: amax(T) (algorithms.py:74)
    double* partial;         // device [rows][4]: max |C|^2, sum r^2, sum r*u, sum u^2 per line
    double* intensity;       // device double, same layout, or null: |C|^2 (final expected_outcome, unscaled)
    const void* tw;
};

// ---- launch table: one entry per (line length, precision), see gen_lines.py ----------------------
struct LineTable {
    int L, prec;
    int rows_per_cta, row_threads; size_t row_smem;     // when L is the row length W
    int cols_per_cta, col_threads; size_t col_smem;     // when L is the column length H
    void (*prepare)();                                   // per-device function attributes
    int (*row_pass)(int alg, const RowArgs&, cudaStream_t);
    int (*row_plain)(const PlainRowArgs&, cudaStream_t);
    int (*col_pass)(int alg, const ColArgs&, cudaStream_t);
    int (*col_plain)(const PlainColArgs&, cudaStream_t);
    // warp-specialised persistent column kernel (col_groups.cuh); group_ok == 0: not built for this length
    int group_ok, group_row_bytes;
    int group_fused;         // CGM_GD_FUSED is available (col_warp.cuh serves this length and precision)
    int (*col_group)(int mode, const ColGroupArgs&, const void* map_in, const void* map_out, int ctas, cudaStream_t);
    int (*row_fourier)(const RowFourierArgs&, cudaStream_t);     // fp32/fp64 GS Fourier-plane step on rows
    int rows_only;                                               // long lines (>= 8192): no column kernels
};
const LineTable* find_line_table(int L, int prec);
int supported_lengths(int* out, int cap);

}  // namespace slm
