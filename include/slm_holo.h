/* libslmholo -- C ABI of the B200 hologram-synthesis engine.
 *
 * Drop-in boundary for the Gerchberg-Saxton / gradient-descent phase-retrieval path of
 * pranislav/Spatial_Light_Modulator_Module.  The reference has no FFI: its "operator API" is
 * the Python functions of src/algorithms.py and their helpers.  Each entry point below names the
 * reference code it replaces (paths relative to the reference root); the Python package
 * spatial_light_modulator_module_b200 binds them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - return 0 on success, a negative code otherwise; slm_last_error() describes the failure.
 *     Nothing is thrown across the ABI.
 *   - "device" pointers are valid on the context's device; "host" pointers are ordinary memory
 *     read before the call returns.  Planes are row-major [batch][H][W].
 *   - complex<R>/real<R>: R = float for SLM_PREC_F32 contexts, double for SLM_PREC_F64 ones.
 *   - all work is enqueued on the context's stream; only slm_read_curves and slm_rows_state synchronise.
 *   - a context is not thread-safe; no device allocation happens after slm_ctx_create.
 */
#ifndef SLM_HOLO_H
#define SLM_HOLO_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct slm_ctx slm_ctx;

enum { SLM_PREC_F32 = 0, SLM_PREC_F64 = 1 };
enum { SLM_OK = 0, SLM_ERR_ARG = -1, SLM_ERR_SHAPE = -2, SLM_ERR_CUDA = -3, SLM_ERR_ALLOC = -4 };
/* 8-bit conversions of the reference (SURVEY.md 8a Q1-Q4) */
enum { SLM_QUANT_ROUND_WRAP = 1,   /* wavefront_correction.py:458-459 convert_2pi_hologram_to_int_hologram */
       SLM_QUANT_PIL_FLOAT = 2,    /* display_holograms.py:253-258,265 mask_hologram (.npy branch)         */
       SLM_QUANT_FLOOR = 3,        /* move_traps.py:135-138 display_hologram; show_hologram.py:9-11         */
       SLM_QUANT_PREVIEW = 5 };    /* generate_hologram_sequence.py:29 fromarray(expected).convert("L")    */

const char* slm_last_error(void);
int slm_version(void);
/* Line lengths (H and W) the kernels are built for; returns the count, fills up to `cap`. */
int slm_supported_lengths(int* out, int cap);

/* One context per (device, stream, plane shape, precision); owns twiddles and the two field
 * workspaces for up to `max_batch` planes and `max_loops_hint` iterations (grown on demand
 * before any launch).  `cuda_stream` is a cudaStream_t (NULL = default stream). */
int slm_ctx_create(slm_ctx** out, int device, int H, int W, int max_batch, int precision, void* cuda_stream);
void slm_ctx_destroy(slm_ctx* ctx);
size_t slm_ctx_workspace_bytes(const slm_ctx* ctx);
/* number of kernels this context has launched since creation (bench.py's gpu_launches) */
long long slm_ctx_launch_count(const slm_ctx* ctx);

/* Per-launch device timing for bench.py's roofline: while enabled every kernel launch is bracketed
 * by CUDA events on the context's stream.  slm_ctx_profile_read synchronises, accumulates and
 * clears them: ms[k] / count[k], k = 0 SLM-plane (row) pass, 1 Fourier-plane (column) pass,
 * 2 column max pre-pass, 3 plain row transform, 4 plain column transform, 5 elementwise. */
int slm_ctx_profile(slm_ctx* ctx, int enable);
int slm_ctx_profile_read(slm_ctx* ctx, double* ms, long long* count);

/* scipy.fft.fft2 / ifft2 (algorithms.py:2; forward unnormalised, inverse scaled 1/(H*W)).
 * in/out: device complex<R> [batch][H][W]; may alias. */
int slm_fft2(slm_ctx* ctx, int batch, const void* in, void* out, int inverse);

/* gerchberg_saxton(demanded_output, args) -- algorithms.py:10-49.
 *   target_u8      device uint8 target, or NULL when the target is not 8-bit, in which case
 *   target_real    device real<R> target and
 *   amp_real       device real<R> |sqrt(target)| (algorithms.py:21,33) are used
 *   amp_lut        host double[256]: np.sqrt(np.arange(256,dtype=uint8)) (float16-rounded, SURVEY A.1)
 *   norm           host double[batch]: np.amax(target) per plane (algorithms.py:23)
 *   inc_amp        device real<R> [H][W] sqrt(illumination) or NULL = uniform (algorithms.py:14-19)
 *   phasor0        device complex<R> B of iteration 0 (algorithms.py:30) or NULL = compute
 *                  A = ifft2(amplitude) on the device (algorithms.py:27), in complex64 when
 *                  setup_c64 != 0 (what numpy does for <=16-bit / float32 targets), else in R
 *   hologram_out   device double: angle(A) (algorithms.py:48)
 *   expected_out   device double or NULL: expected_outcome (algorithms.py:36-37)
 * Error curves / iteration counts stay in the context until slm_read_curves. */
int slm_gs_run(slm_ctx* ctx, int batch, const uint8_t* target_u8, const void* target_real, const void* amp_real,
               const double* amp_lut, const double* norm, const void* inc_amp, const void* phasor0, int setup_c64,
               int max_loops, double tolerance, double* hologram_out, double* expected_out);

/* Weighted Gerchberg-Saxton (GSW; Di Leonardo, Ianni & Ruocco, Opt. Express 15, 1913 (2007)): GS with per-pixel
 * weights w on the target amplitude, so that the reconstructed intensity follows the target's levels (uniform trap
 * arrays).  Per iteration k, on the signal set {T > 0} where I_k = |C_k|^2 > 0:
 *     w_k = clamp(w_{k-1} * amp / sqrt(sigma_k * I_k), 1/weight_limit, weight_limit),   D_k = (amp * w_k) * C_k / |C_k|
 * with sigma_k = target_sum / P_{k-1}, P = sum of I over the signal set (P_0 for k = 0); elsewhere w_k = w_{k-1}.
 * Scale, error curve, tolerance stop, expected outcome and hologram are GS's; weight_limit = 1 gives GS's bits.
 * Arguments as slm_gs_run, plus
 *   target_sum     host double[batch]: sum(T) per plane
 *   weights        device real<R> [batch][H][W]: initial weights in (ones for plain GSW), final weights out
 *   weight_limit   c >= 1 (else SLM_ERR_ARG) */
int slm_gsw_run(slm_ctx* ctx, int batch, const uint8_t* target_u8, const void* target_real, const void* amp_real,
                const double* amp_lut, const double* norm, const void* inc_amp, const void* phasor0, int setup_c64,
                int max_loops, double tolerance, double* hologram_out, double* expected_out,
                const double* target_sum, void* weights, double weight_limit);

/* Multi-plane Gerchberg-Saxton (Haist et al., Opt. Commun. 140, 299 (1997)): one phase hologram for K target planes at
 * different focus, plane k being the plane a lens of phase alpha_k * rho^2 brings into focus (rho^2 = (y - H/2)^2 +
 * (x - W/2)^2 in pixels^2; alpha_k = -pi px^2 / (lambda f_k), 0 for the Fourier plane).  With L_k = exp(i alpha_k rho^2):
 *     setup      A = sum_k ifft2(amp_k) conj(L_k)               (ifft2 as slm_gs_run's setup)
 *     iteration  B = inc exp(i angle(A));  per plane C_k = fft2(B L_k), D_k = amp_k C_k/|C_k|, error and expected
 *                outcome of plane k as GS's;  A = sum_k ifft2(D_k) conj(L_k)
 *     hologram   angle(A) after the last iteration
 * A hologram iterates until the error of EVERY one of its planes is <= tolerance (or max_loops): its K error curves
 * have the same length.  planes = 1 with alpha = 0 is slm_gs_run, bit for bit.
 * Arguments as slm_gs_run, with the batch made of `holograms` x `planes` planes, plane k of hologram g at g*planes + k:
 *   holograms, planes   1 <= planes <= 8, holograms * planes <= max_batch (else SLM_ERR_ARG)
 *   target_u8 / target_real / amp_real / norm / expected_out   per plane
 *   defocus        host double[planes]: alpha_k in radians per pixel^2, finite (else SLM_ERR_ARG), shared by the holograms
 *   phasor0        device complex<R> [holograms][H][W] or NULL: B of iteration 0
 *   hologram_out   device double [holograms][H][W]
 * Error curves: slm_read_curves over holograms * planes planes. */
int slm_gs_multiplane_run(slm_ctx* ctx, int holograms, int planes, const uint8_t* target_u8, const void* target_real,
                          const void* amp_real, const double* amp_lut, const double* norm, const double* defocus,
                          const void* inc_amp, const void* phasor0, int setup_c64, int max_loops, double tolerance,
                          double* hologram_out, double* expected_out);

/* gradient_descent(demanded_output, args) -- algorithms.py:60-112 (+ dEdX_complex :179-185).
 *   x              device complex<R> [batch][H][W]: the initial guess (algorithms.py:75), updated in place
 *   mask_lut       host double[256]: 1 + white_attention*g/255 for g = 0..255 as numpy computes it
 *                  (uint8 wrap for an int white_attention, SURVEY A.2); mask_real for non-8-bit targets
 *   lr_schedule    host double[max_loops]: args.learning_rate in force during iteration k
 *                  (doubling rule algorithms.py:103-104 applied by the caller) */
int slm_gd_run(slm_ctx* ctx, int batch, const uint8_t* target_u8, const void* target_real, const void* mask_real,
               const double* mask_lut, const double* norm, const void* inc_amp, void* x, const double* lr_schedule,
               int max_loops, double tolerance, double* hologram_out, double* expected_out);

/* make_initial_guess("fourier", ...) -- algorithms.py:154-157: inc_amp * exp(1j*angle(ifft2(sqrt(T)))) */
int slm_fourier_guess(slm_ctx* ctx, int batch, const uint8_t* target_u8, const void* amp_real, const double* amp_lut,
                      const void* inc_amp, int setup_c64, void* x_out);

/* Multi-plane gradient descent: one phase hologram for K target planes at different focus (plane k and L_k as in
 * slm_gs_multiplane_run), by gradient descent on the mean of the planes' errors.  Each iteration:
 *     B = x/|x| inc;  per plane F_k = fft2(B L_k), out_k = |F_k|^2 norm_k / max |F_k|^2,
 *                     G_k = ifft2(mask_k F_k (out_k - T_k)), error and expected outcome of plane k as GD's
 *     dEdF = (sum_k G_k conj(L_k)) inc / K;  x -= lr_i dEdX_complex(dEdF, x)
 *     hologram   angle(x) after the last update
 * A hologram iterates until the error of EVERY one of its planes is <= tolerance (or max_loops); the update of the
 * iteration that ends the loop is applied.  planes = 1 with alpha = 0 runs slm_gd_run's passes: its results, bit for bit.
 * Arguments as slm_gd_run, with the batch made of `holograms` x `planes` planes (g*planes + k), and as
 * slm_gs_multiplane_run for holograms, planes and defocus (same refusals):
 *   target_u8 / target_real / mask_real / norm / expected_out   per plane
 *   x              device complex<R> [holograms][H][W]: one initial guess per hologram, updated in place
 *   lr_schedule    host double[max_loops], shared by the holograms
 *   hologram_out   device double [holograms][H][W]
 * Error curves: slm_read_curves over holograms * planes planes. */
int slm_gd_multiplane_run(slm_ctx* ctx, int holograms, int planes, const uint8_t* target_u8, const void* target_real,
                          const void* mask_real, const double* mask_lut, const double* norm, const double* defocus,
                          const void* inc_amp, void* x, const double* lr_schedule, int max_loops, double tolerance,
                          double* hologram_out, double* expected_out);

/* "fourier" initial guess of multi-plane GD: x = inc exp(i angle(sum_k ifft2(sqrt(T_k)) conj(L_k))), the setup sum of
 * slm_gs_multiplane_run (ifft2 as slm_fourier_guess's).  Arguments as slm_fourier_guess per plane, and holograms,
 * planes, defocus as slm_gs_multiplane_run (same refusals); x_out: device complex<R> [holograms][H][W]. */
int slm_multiplane_fourier_guess(slm_ctx* ctx, int holograms, int planes, const uint8_t* target_u8, const void* amp_real,
                                 const double* amp_lut, const double* defocus, const void* inc_amp, int setup_c64,
                                 void* x_out);

/* make_initial_guess("random" | "zeros", ...) -- algorithms.py:118-124,145-151: exp(1j*2*pi*u) / divide_by
 * from the MT19937 stream `u` (device double[n], drawn on the host exactly as random.random() does);
 * x_out: device complex<R>[n]. */
int slm_random_phasor(slm_ctx* ctx, const double* u, void* x_out, long long n, double divide_by);

/* n successive random.random() values (algorithms.py:121,129,139,147) on the device: MT19937 continued from
 * `state` (host uint32[624], random.getstate()[1][:624]) at read position `pos` (even; 624 right after
 * random.seed).  u: device double[n].  state_out: host uint32[625] = final state words + final position,
 * so the caller can leave the module-level generator where the reference's loop would.  Synchronises. */
int slm_mt19937_uniform(slm_ctx* ctx, const uint32_t* state, int pos, double* u, long long n, uint32_t* state_out);

/* inc_amp * exp(1j*phase): B of algorithms.py:30 from a hologram angle(A), to continue a GS run (used for the
 * per-iteration GIF snapshots, algorithms.py:40-41).  phase: device double[n]; inc_amp: device real<R>[plane] or NULL. */
int slm_phase_phasor(slm_ctx* ctx, const double* phase, const void* inc_amp, void* x_out, long long n, long long plane);

/* move_traps.update_hologram -- move_traps.py:64-68: np.angle(ifft2(one_hot(row, col))) in closed form. */
int slm_single_trap_phase(slm_ctx* ctx, int H, int W, int row, int col, double* out);

/* traps_images.make_traps_image / dot -- traps_images.py:10-16,87-91, batched: zero `frames`
 * (device uint8 [n_frames][H][W]) and set the pixels listed in frame_y_x (device int[n_dots][3]) to 255. */
int slm_trap_frames(slm_ctx* ctx, uint8_t* frames, int n_frames, int H, int W, const int* frame_y_x, int n_dots);

/* ---- one very large plane split by rows over the ranks (BASELINE config 5): slab-decomposed 2-D transform ----
 * Rank p owns `rows` = N/P rows of the N x N field.  A 2-D transform is: line transforms on the row slab,
 * exchange (pack -> all-to-all -> the peers' blocks side by side = the "exchange layout"), line transforms
 * on the received columns (now contiguous lines), exchange back.  The library supplies the kernels.  The
 * all-to-all and the 4-scalar all-gather are either the caller's collectives (NCCL through torch.distributed in
 * slab.py) or this library's stores into the peers' memory (slm_transpose_blocks_peer, slm_rows_reduce with peers),
 * ordered by the caller's device-side barriers.
 * GS does not depend on the transform's scale (only angle(A) is used), so these transforms are unnormalised. */
int slm_rows_create(slm_ctx** out, int device, int rows, int W, int precision, void* cuda_stream);
/* plain line transforms of every row: `in` complex<R> (or in_u8 + host lut[256] -> real input, algorithms.py:21,27);
 * block_in/block_out = 0 for [rows][W], else the exchange layout's block width (= rows). */
int slm_rows_fft(slm_ctx* ctx, const void* in, const uint8_t* in_u8, const double* lut, void* out, int inverse,
                 int block_in, int block_out);
/* SLM-plane step on a row slab (algorithms.py:30,34): in_is_field = 0: finish ifft2 along the rows first;
 * 1: `in` is the field A itself (complex<R>); 2: A as complex64 whatever the context's precision (the
 * reference's first ifft2 runs in complex64 for 8-bit targets, SURVEY A.1) -- phasor taken in fp32.
 * final_pass: write angle(A) to `hologram` (device double [rows][W]) instead of starting the next fft2. */
int slm_rows_gs_row_pass(slm_ctx* ctx, const void* in, void* out, const void* inc_amp, int in_is_field, int final_pass,
                         double* hologram);
/* Fourier-plane step on received columns in the exchange layout (block_w: the block width), by `mode`:
 *   0 (GS, algorithms.py:31-38): finish fft2, replace the amplitude (lut: host double[256], amplitude by grey level),
 *     start ifft2; per-line sums max |C|^2, sum r^2, sum r*u, sum u^2 against the scale of the previous iteration;
 *   1 (GD max, :84-86): finish fft2, keep the transform (out), max |F|^2 per line into partial[.][0];
 *   2 (GD step on the kept transform, after slm_rows_close kind 0 has closed mode 1's maxima: :85-88,92): output,
 *     error sum into partial[.][1], mask * F * (output - T) (lut: the mask by grey level), first half of ifft2.
 * Modes 0 and 2 need target_u8 and lut; norm = amax(T) (read by mode 2).  Scale and max come from the context's loop
 * state (slm_rows_close), which stays on the device.  partial: device double[rows][4]; intensity (nullable, device
 * double, same layout as `in`; modes 0 and 2) receives |C|^2 (GD: the expected outcome = that * norm / max). */
int slm_rows_fourier_pass(slm_ctx* ctx, int mode, const void* in, void* out, int block_w, const uint8_t* target_u8,
                          const double* lut, double norm, double* partial, double* intensity);
/* partial[rows][4] -> out4 (device double[4]: max, three sums) by one CTA in a fixed order.  With n_peers > 0 the four
 * numbers are also stored into every peer's gathered[self] (peer_gathered[r] = rank r's device double[n_peers][4],
 * mapped into this process: peer memory over NVLink) -- otherwise the caller all-gathers out4. */
int slm_rows_reduce(slm_ctx* ctx, const double* partial, int rows, double* out4, const void* const* peer_gathered,
                    int n_peers, int self);
/* Close a Fourier-plane pass of the distributed plane from every rank's four numbers (gathered: device double[world][4],
 * added in rank order) into the context's loop state.  kind 0: the max and the scale norm / max only (the exact scale
 * of GS iteration 0, the max pass of a GD iteration); 1: a GS iteration (scale, error algorithms.py:37-38,162);
 * 2: a GD iteration (error = sum (output - T)^2 / HW, :92).  Kinds 1 and 2 append the error to err_curve (device
 * double[max_loops]), count the iteration and set the loop-ended flag (algorithms.py:29,83). */
int slm_rows_close(slm_ctx* ctx, const double* gathered, int world, double norm, double hw, int kind, double tolerance,
                   double* err_curve);
/* The context's loop state, read back (synchronises the stream; every output nullable): scale and max of the latest
 * closing, iterations closed, loop-ended flag. */
int slm_rows_state(slm_ctx* ctx, double* scale, double* imax, int* iters, int* done);
/* Gradient descent (algorithms.py:60-112) on the distributed plane, same exchange as GS and two Fourier-plane passes
 * (modes 1 and 2, each closed by slm_rows_close: kind 0, then kind 2) per iteration:
 *   slm_rows_reset           zero the context's loop state before a run;
 *   slm_rows_gd_row_pass     SLM-plane pass on this rank's rows: finish ifft2 along the rows (in: lines back from the exchange),
 *                            dEdX + update of x in place with lr_dev[iteration] (:87-91,179-185), x/|x| and the row half of fft2
 *                            (:84) into out; first != 0: no update yet (the run's first pass); final_pass != 0: the last update,
 *                            then angle(x) into hologram (:111) instead of a transform. */
int slm_rows_reset(slm_ctx* ctx);
int slm_rows_gd_row_pass(slm_ctx* ctx, const void* in, void* x, void* out, const double* lr_dev, int first, int final_pass, double* hologram);
/* row slab [rows][W] <-> exchange layout [W/rows][rows][rows] (each block transposed); elem_bytes 1, 8 or 16. */
int slm_transpose_blocks(slm_ctx* ctx, const void* in, void* out, int rows, int W, int elem_bytes, int from_exchange);

/* The transposing copy AS the all-to-all: block q goes straight into rank q's memory (peers[q], mapped into this
 * process -- CUDA peer memory over NVLink), so the blocks cross the links while they are being transposed and no
 * send/receive staging exists.  from_exchange = 0: peers[q] is rank q's receive buffer (exchange layout), block `self`
 * of it is written; from_exchange = 1: peers[q] is rank q's row slab, columns [self*rows, (self+1)*rows) are written.
 * The caller orders the ranks (a device-side barrier before the consumers run and before the buffers are reused). */
int slm_transpose_blocks_peer(slm_ctx* ctx, const void* in, const void* const* peers, int n_peers, int self, int rows, int W,
                              int elem_bytes, int from_exchange);

/* error_evolution and its length per plane (algorithms.py:25,39,93) of the last run.
 * err: host double[batch][max_loops]; iters: host int[batch].  Synchronises the stream. */
int slm_read_curves(slm_ctx* ctx, int batch, int max_loops, double* err, int* iters);

/* show_expected_outcome numeric part -- generate_hologram.py:24-29:
 * |fft2(exp(1j*h))|^2 / max * norm.  hologram/out: device double; norm: host double[batch]. */
int slm_expected_outcome(slm_ctx* ctx, int batch, const double* hologram, const double* norm, double* out);

/* wfc.deflect_2pi -- wavefront_correction.py:440-449: (konst*(sy*i + sx*j)) % 2pi,
 * konst = 2*pi*px/lambda, sy = sin(y_angle*u), sx = sin(x_angle*u) evaluated by the caller. */
int slm_deflect_phase(slm_ctx* ctx, int H, int W, double konst, double sy, double sx, double* out);
/* lens -- generate_hologram.py:189-203: k*(1-sqrt(1+r^2/f2)) % 2pi, k = 2*pi*f/lambda, f2 = f**2;
 * trunc_u8 reproduces the reference's uint8 store (values 0..6). */
int slm_lens_phase(slm_ctx* ctx, int H, int W, double px, double k, double f2, int trunc_u8, double* out);
/* deflect_hologram / add_lens -- generate_hologram.py:178-186: (a + b) % 2pi; b is one plane of
 * `plane` elements broadcast over the n elements of a. */
int slm_add_mod2pi(slm_ctx* ctx, const double* a, const double* b, double* out, long long n, long long plane);
/* mask add + 8-bit conversion, mode = SLM_QUANT_*; mask (one plane, broadcast) may be NULL. */
int slm_quantize(slm_ctx* ctx, const double* phase, const double* mask, double ct2pi, int mode, uint8_t* out,
                 long long n, long long plane);
/* mask_hologram image branch -- display_holograms.py:259-265 */
int slm_quantize_grey(slm_ctx* ctx, const uint8_t* grey, const double* mask, double ct2pi, uint8_t* out,
                      long long n, long long plane);

/* ---- host memory ------------------------------------------------------------------------------------------
 * Page-lock / release a HOST array in place, so that copies from it are plain DMA (the reference hands the same
 * numpy arrays -- the wavefront-correction mask, display_holograms.py:189-204 -- to every frame).  A range that
 * cannot be locked (already locked pages, limits) returns SLM_ERR_CUDA and leaves no pending CUDA error. */
int slm_host_register(void* ptr, size_t bytes);
int slm_host_unregister(void* ptr);

#ifdef __cplusplus
}
#endif
#endif
