// libslmholo: context, pass scheduling and the C ABI (include/slm_holo.h).
//
// Scheduling of one run (all launches on the context's stream, no host synchronisation):
//   GS  (algorithms.py:10-49):  setup -> row pass -> max pre-pass -> { col pass, row pass } * loops
//                               -> final row pass (hologram) -> intensity pass (expected_outcome)
//   GD  (algorithms.py:60-112): row pass -> { max pre-pass, col pass, row pass } * loops
//                               -> final row pass (last update + hologram) -> intensity pass
// Planes whose loop condition has failed (tolerance) are skipped by every later pass, so a batch
// needs no host round trip per iteration.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cmath>
#include <string>
#include <vector>

#include "../../include/slm_holo.h"
#include "elementwise.cuh"
#include "engine_types.h"

using namespace slm;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define SLM_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) return fail(SLM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)
#define SLM_TRY(expr)                                                                           \
    do {                                                                                        \
        int r_ = (expr);                                                                        \
        if (r_ != 0) return r_ < -1000 ? fail(SLM_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString((cudaError_t)(-r_ - 1000))) : r_; \
    } while (0)

struct slm_ctx {
    int device = 0, H = 0, W = 0, max_batch = 0, prec = 0;
    cudaStream_t stream = nullptr;
    const LineTable *row = nullptr, *col = nullptr;       // precision of the context
    const LineTable *row32 = nullptr, *col32 = nullptr;   // complex64 setup path (SURVEY A.1)
    void *X = nullptr, *Y = nullptr;
    void *tw_row = nullptr, *tw_col = nullptr, *tw_row32 = nullptr, *tw_col32 = nullptr;
    PlaneStats* stats = nullptr;
    Partial* partial = nullptr;
    unsigned* counter = nullptr;
    unsigned* fused = nullptr;                            // [max_batch] pairs {plane max bits, tile count} of the one-pass GD forms + time-out flag
    int fused_ctas = 0;                                   // grid of the fused GD column pass (0: two passes)
    bool pipe_ok = false;                                 // CGM_GD_PIPE may be used (warp-per-column kernel, a plane's tiles fit the CTAs' buffers)
    double *err_curve = nullptr, *lr = nullptr, *norm = nullptr;
    // weighted GS, allocated by the first slm_gsw_run: [max_batch] S_T, [max_batch] P, [max_batch][tiles] partials of P
    double *target_sum = nullptr, *signal_sum = nullptr, *signal_partial = nullptr;
    // multi-plane GS, allocated by the first slm_gs_multiplane_run: defocus tables [kMaxPlanes][H] and [kMaxPlanes][W]
    // complex<R>, the alphas they hold, and their host staging (lives as long as the context, like lut_host_f)
    void *lens_y = nullptr, *lens_x = nullptr;
    std::vector<double> lens_alpha;
    std::vector<double> lens_host_d;
    std::vector<float> lens_host_f;
    void* lut = nullptr;
    float* lut32 = nullptr;
    double lut_host[256];                                 // the table the device copies hold (upload_lut)
    float lut_host_f[256];                                // ... narrowed: staging for the copies (lives as long as the context)
    bool lut_valid = false;
    unsigned* mt_buf = nullptr;                           // [624 state in][625 state out] of slm_mt19937_uniform
    int loops_cap = 0, tiles = 0;
    size_t bytes = 0;
    long long launches = 0;
    std::vector<void*> owned;
    // TMA tile maps over X and Y for the warp-specialised column kernel (context precision), its grid
    TileMap map_x, map_y;
    bool use_groups = false;
    int persist_ctas = 1;
    // optional per-launch device timing (slm_ctx_profile): event pairs on the context's stream
    bool profiling = false;
    struct Timed { int kind; cudaEvent_t a, b; };
    std::vector<Timed> timed;
#ifndef SLM_EMULATE
    // graphs of one loop iteration, replayed (see replay_iterations); destroyed once their last launch has run
    struct Replay { cudaGraphExec_t exec; cudaGraph_t graph; cudaEvent_t done; };
    std::vector<Replay> replays;
    cudaStream_t capture_stream = nullptr;                // (the context's stream may be the legacy default stream, which cannot capture)
    // whole loops of small runs, kept per argument set (see replay_iterations)
    struct Kept { std::string key; cudaGraphExec_t exec; cudaGraph_t graph; long long launches; unsigned long long stamp; };
    std::vector<Kept> kept;
    std::vector<std::string> seen;                        // argument sets met once (the last few)
    unsigned long long kept_clock = 0;
#endif
};

// launch kinds reported by slm_ctx_profile_read
enum { K_ROW_PASS = 0, K_COL_PASS = 1, K_COL_STATS = 2, K_ROW_PLAIN = 3, K_COL_PLAIN = 4, K_ELEMENTWISE = 5, K_KINDS = 6 };

#ifndef SLM_EMULATE
struct LaunchTimer {
    slm_ctx* c; int kind; cudaEvent_t a = nullptr, b = nullptr;
    LaunchTimer(slm_ctx* c_, int k) : c(c_), kind(k) {
        c->launches++;
        if (!c->profiling) return;
        cudaEventCreate(&a); cudaEventCreate(&b);
        cudaEventRecord(a, c->stream);
    }
    ~LaunchTimer() {
        if (!a) return;
        cudaEventRecord(b, c->stream);
        c->timed.push_back({kind, a, b});
    }
};
#else
struct LaunchTimer { LaunchTimer(slm_ctx* c, int) { c->launches++; } };
#endif
#define SLM_TIMED(kind, expr) do { LaunchTimer t_(c, kind); SLM_TRY(expr); } while (0)


static size_t real_size(int prec) { return prec == PREC_F64 ? 8 : 4; }

static int dev_alloc(slm_ctx* c, void** p, size_t n) {
    SLM_CUDA(cudaMalloc(p, n ? n : 16));
    c->owned.push_back(*p);
    c->bytes += n;
    return 0;
}

// exp(-2 pi i q / N), q in [0, N), evaluated in extended precision
static int make_twiddles(slm_ctx* c, int N, int prec, void** out) {
    std::vector<double> td(2 * (size_t)N);
    std::vector<float> tf(2 * (size_t)N);
    const long double two_pi = 6.283185307179586476925286766559005768L;
    for (int q = 0; q < N; ++q) {
        // exact octant symmetry is not needed; long double sin/cos are accurate to < 1 ulp of double
        const long double ang = -two_pi * (long double)q / (long double)N;
        td[2 * q] = (double)cosl(ang); td[2 * q + 1] = (double)sinl(ang);
        tf[2 * q] = (float)cosl(ang); tf[2 * q + 1] = (float)sinl(ang);
    }
    const size_t bytes = 2 * (size_t)N * real_size(prec);
    SLM_TRY(dev_alloc(c, out, bytes));
    SLM_CUDA(cudaMemcpy(*out, prec == PREC_F64 ? (const void*)td.data() : (const void*)tf.data(), bytes, cudaMemcpyHostToDevice));
    return 0;
}

// Describe a field plane stack ([rows][W complex columns]) to the TMA unit: 2-D tensor of real
// elements, box = TC complex columns x up to 256 rows, 32B/64B-swizzled shared-memory image.  A tile is
// H / box_rows whole boxes, so box_rows divides H (a box that ran past the tile would land in the next buffer
// and overshoot the barrier's byte count); 256 for every length the column-group kernel serves now.
static int tile_box_rows(int H) {
    int b = H < 256 ? H : 256;
    while (H % b != 0) --b;
    return b;
}
static int make_tile_map(slm_ctx* c, void* base, long long rows, TileMap* out) {
    const size_t cs = 2 * real_size(c->prec);
    const int row_bytes = c->col->group_row_bytes;
    const int box_rows = tile_box_rows(c->H);
#ifdef SLM_EMULATE
    (void)rows;
    out->base = static_cast<unsigned char*>(base);
    out->pitch_bytes = (size_t)c->W * cs;
    out->box_rows = box_rows;
    out->row_bytes = row_bytes;
    return 0;
#else
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        SLM_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
        if (!fn || q != cudaDriverEntryPointSuccess) return fail(SLM_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
        encode = reinterpret_cast<EncodeFn>(fn);
    }
    const cuuint64_t dims[2] = {(cuuint64_t)2 * c->W, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)c->W * cs};
    const cuuint32_t box[2] = {(cuuint32_t)(row_bytes / real_size(c->prec)), (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(&out->map, c->prec == PREC_F64 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                              base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B,
                              CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(SLM_ERR_CUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r));
    out->box_rows = box_rows;
    out->row_bytes = row_bytes;
    return 0;
#endif
}

static int setup_groups(slm_ctx* c) {
    c->use_groups = false;
    if (!c->col->group_ok || getenv("SLM_NO_GROUPS")) return 0;
    SLM_TRY(make_tile_map(c, c->X, (long long)c->max_batch * c->H, &c->map_x));
    SLM_TRY(make_tile_map(c, c->Y, (long long)c->max_batch * c->H, &c->map_y));
#ifdef SLM_EMULATE
    c->persist_ctas = 3;
#else
    int sms = 0;
    SLM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, c->device));
    c->persist_ctas = sms > 0 ? sms : 1;
#endif
    c->use_groups = true;
    {
        // The pipelined one-pass form: a tile waits (in a buffer) for the other tiles of its plane, which sit in at most
        // ceil(tiles / CTAs) buffers of every other CTA -- that many must exist (three per CTA), or the planes could not
        // complete.  The warp-per-column kernel only.
        const char* ck = getenv("SLM_COL_KERNEL");
        const int tiles = c->W / c->col->cols_per_cta;
        c->pipe_ok = c->col->group_fused && !(ck && ck[0] == 'g') && tiles <= 3 * c->persist_ctas;
    }
#ifndef SLM_EMULATE
    // One fused Fourier-plane pass per GD iteration needs every tile of a plane on an SM at the same time: grid = a
    // whole number of planes' tiles, all CTAs resident (one per SM).  Worth it when that grid fills most of the device.
    // (The host emulation runs one CTA at a time and keeps the two-pass form.)
    const char* ck = getenv("SLM_COL_KERNEL");
    const int tiles = c->W / c->col->cols_per_cta;
    if (c->col->group_fused && !(ck && ck[0] == 'g') && !getenv("SLM_NO_FUSED_GD") && tiles <= c->persist_ctas) {
        const int grid = tiles * (c->persist_ctas / tiles);
        if (5 * grid >= 4 * c->persist_ctas) c->fused_ctas = grid;
    }
#endif
    return 0;
}

#ifdef SLM_TRACE
// developer tooling (trace builds only): arm / read the column kernel's device timeline
static unsigned long long* g_trace = nullptr;
static int g_trace_mode = -1;
extern "C" int slm_trace_arm(int mode) {
    if (!g_trace) cudaMalloc((void**)&g_trace, 148 * 64 * 16 * sizeof(unsigned long long));
    cudaMemset(g_trace, 0, 148 * 64 * 16 * sizeof(unsigned long long));
    g_trace_mode = mode;
    return 0;
}
extern "C" int slm_trace_read(unsigned long long* out) {
    cudaDeviceSynchronize();
    return (int)cudaMemcpy(out, g_trace, 148 * 64 * 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
}
#endif
// Launch one mode of the warp-specialised column kernel over X (in) -> map_out.
static int launch_group(slm_ctx* c, int mode, int batch, const ColArgs* loop, const TileMap* map_out, int inverse, double scale,
                        int all_planes = 0) {
    ColGroupArgs ga{};
    if (loop) ga.c = *loop;
    ga.mode_inverse = inverse; ga.scale = scale; ga.all_planes = all_planes;
    // large batches: the planes are closed by a kernel behind the pass (see ColGroupArgs::defer_close); a few planes
    // keep the in-kernel closing, which costs no extra launch
    ga.defer_close = (mode != CGM_COMPLEX && mode != CGM_GD_FUSED && !getenv("SLM_NO_DEFER_CLOSE") &&
                      (long long)batch * (c->W / c->col->cols_per_cta) > 4LL * c->persist_ctas) ? 1 : 0;
#ifdef SLM_TRACE
    if (mode == g_trace_mode) { ga.trace = g_trace; g_trace_mode = -1; }      // trace the next launch of that mode only
#endif
    ga.c.B = batch; ga.c.W = c->W; ga.c.stats = c->stats; ga.c.partial = c->partial; ga.c.counter = c->counter;
    ga.c.norm = c->norm; ga.c.tw = c->tw_col;
    ga.c.fused_max = c->fused; ga.c.max_planes = c->max_batch;
    int ctas = mode == CGM_GD_FUSED ? c->fused_ctas : c->persist_ctas;
    if (mode == CGM_GD_PIPE) {
        static const char* pc = getenv("SLM_PIPE_CTAS");         // developer switch (A/B measurements)
        if (pc && atoi(pc) > 0 && atoi(pc) <= c->persist_ctas) ctas = atoi(pc);
    }
    const int kind = (mode == CGM_STATS || mode == CGM_STATS_KEEP) ? K_COL_STATS : (mode == CGM_COMPLEX ? K_COL_PLAIN : K_COL_PASS);
    SLM_TIMED(kind, c->col->col_group(mode, ga, &c->map_x, map_out ? map_out : &c->map_x, ctas, c->stream));
    if (ga.defer_close) c->launches++;               // the closing kernel behind the pass
    return 0;
}

static int ensure_loops(slm_ctx* c, int max_loops) {
    if (max_loops <= c->loops_cap) return 0;
    int cap = c->loops_cap ? c->loops_cap : 256;
    while (cap < max_loops) cap *= 2;
    SLM_CUDA(cudaStreamSynchronize(c->stream));
    for (void* old : {(void*)c->err_curve, (void*)c->lr}) {           // the smaller buffers are not needed any more
        if (!old) continue;
        for (size_t i = 0; i < c->owned.size(); ++i)
            if (c->owned[i] == old) { c->owned.erase(c->owned.begin() + i); break; }
        cudaFree(old);
    }
    c->err_curve = nullptr; c->lr = nullptr;
    SLM_TRY(dev_alloc(c, (void**)&c->err_curve, (size_t)c->max_batch * cap * sizeof(double)));
    SLM_TRY(dev_alloc(c, (void**)&c->lr, (size_t)cap * sizeof(double)));
    c->loops_cap = cap;
    return 0;
}

// `times` identical iterations of a loop: the launches of up to kReplayChunk iterations (issued by `body` on the
// context's stream) are captured into a CUDA graph and the graph is launched times / chunk times -- one driver call
// per 20 iterations instead of three to five kernel launches per iteration, which the HOST could not always keep up
// with (measured on a slow box of the pool: GS 43.6 instead of 32.1 ms per 100 iterations of 32 planes).  One graph
// per iteration was tried first: the device-side start-up gap between graph launches cost the five-kernel two-pass GD
// form more (53.4 ms) than the host saved (44.9 ms without graphs).  Every iteration-dependent quantity (iteration count, learning rate, scale, loop condition)
// lives in device memory, so the captured arguments are the same for all iterations (SURVEY 7, step 4).
// Falls back to plain launches when capture is not possible; SLM_NO_GRAPH=1 disables it.
static const int kReplayChunk = 20;          // iterations per graph: a graph launch has a start-up gap of its own on the device

#ifndef SLM_EMULATE
// Record `n` iterations (issued by `body` on the context's stream) into an instantiated graph.  The iterations are
// recorded from a stream of the context's own (the caller's may be the legacy default stream, which cannot capture).
// Returns false -- with the context untouched -- when the driver refuses; launches_out: kernels in the graph.
template <class F> static bool record_iterations(slm_ctx* c, int n, F& body, cudaGraph_t* graph, cudaGraphExec_t* exec, long long* launches_out,
                                                 int* rc_out) {
    *rc_out = 0;
    cudaGetLastError();
    if (!c->capture_stream && cudaStreamCreateWithFlags(&c->capture_stream, cudaStreamNonBlocking) != cudaSuccess) {
        c->capture_stream = nullptr; cudaGetLastError(); return false;
    }
    if (cudaStreamBeginCapture(c->capture_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return false; }
    const long long before = c->launches;
    cudaStream_t callers = c->stream;
    c->stream = c->capture_stream;
    // Recorded without programmatic dependent launch: in a graph the kernels follow each other without the host in
    // between, and a dependent kernel that starts early only takes SM slots from the tail of its predecessor
    // (measured, one 1024^2 plane x 100 iterations from a kept graph: GD 2.39 ms without, 2.67 ms with; GS 2.11 / 2.30).
    const bool pdl = tl_pdl;
    tl_pdl = false;
    int rc = 0;
    for (int i = 0; i < n && rc == 0; ++i) rc = body();
    tl_pdl = pdl;
    c->stream = callers;
    *graph = nullptr; *exec = nullptr;
    const cudaError_t e = cudaStreamEndCapture(c->capture_stream, graph);
    *launches_out = c->launches - before;
    c->launches = before;
    if (rc == 0 && e == cudaSuccess && *graph && cudaGraphInstantiate(exec, *graph, 0) == cudaSuccess) return true;
    if (*graph) cudaGraphDestroy(*graph);
    cudaGetLastError();                                           // (e.g. an attribute the driver cannot capture): plain launches
    if (rc != 0 && rc != SLM_ERR_CUDA) *rc_out = rc;
    return false;
}
#endif

// `times` identical iterations of a loop.  Every iteration-dependent quantity (iteration count, learning rate, scale,
// loop condition) lives in device memory, so the launches of all iterations of a run have the same arguments
// (SURVEY 7, step 4) and can be replayed from a CUDA graph instead of being launched one by one:
//   * LARGE runs (batches): up to kReplayChunk iterations are recorded and the graph is launched times / chunk times --
//     one driver call per 20 iterations instead of three to five launches per iteration, which the HOST could not
//     always keep up with (a slow box of the pool: GS 43.6 instead of 32.1 ms, GD 50.4 instead of 41.9 ms per 100
//     iterations of 32 planes).  One graph per iteration was tried first: the device-side start-up gap between graph
//     launches cost the five-kernel two-pass GD form more (53.4 ms) than the host saved (44.9 ms without graphs).
//   * SMALL runs (one SLM-size plane: latency bound, ~200 launches in under 3 ms): recording a graph per run costs more
//     than it saves (3.0 instead of 2.8 ms), so the whole loop is recorded once per distinct argument set -- `key`: the
//     bytes of every launch argument -- when that set is seen the SECOND time, kept (four per context), and later runs
//     are ONE graph launch.  The drop-in calls meet this in practice: holograms of one shape made one after the other
//     get the same buffers from the allocator.
// Falls back to plain launches whenever capture is not possible; SLM_NO_GRAPH=1 disables all of it.
template <class F> static int replay_iterations(slm_ctx* c, int batch, int times, const std::string& key, F body) {
#ifndef SLM_EMULATE
    static const bool on = !getenv("SLM_NO_GRAPH");
    for (size_t i = 0; i < c->replays.size();) {               // retire one-shot graphs whose last launch has run
        if (cudaEventQuery(c->replays[i].done) == cudaSuccess) {
            cudaGraphExecDestroy(c->replays[i].exec); cudaGraphDestroy(c->replays[i].graph); cudaEventDestroy(c->replays[i].done);
            c->replays.erase(c->replays.begin() + i);
        } else ++i;
    }
    cudaGetLastError();
    const bool large = (long long)batch * c->H * c->W > (1ll << 21);
    if (on && !c->profiling && times >= 4 && large) {
        const int chunk = times < kReplayChunk ? times : kReplayChunk;
        cudaGraph_t graph; cudaGraphExec_t exec; long long launches = 0; int rc = 0;
        if (record_iterations(c, chunk, body, &graph, &exec, &launches, &rc)) {
            for (int i = 0; i < times / chunk; ++i) SLM_CUDA(cudaGraphLaunch(exec, c->stream));
            c->launches += launches * (times / chunk);
            slm_ctx::Replay r{exec, graph, nullptr};
            SLM_CUDA(cudaEventCreateWithFlags(&r.done, cudaEventDisableTiming));
            SLM_CUDA(cudaEventRecord(r.done, c->stream));
            c->replays.push_back(r);
            for (int i = 0; i < times % chunk; ++i) SLM_TRY(body());     // the remainder: plain launches
            return 0;
        }
        if (rc) return rc;
    } else if (on && !c->profiling && times >= 4 && times <= 512 && !key.empty()) {
        for (auto& k : c->kept) {
            if (k.key == key) {                                           // seen before and recorded: one launch
                SLM_CUDA(cudaGraphLaunch(k.exec, c->stream));
                c->launches += k.launches;
                k.stamp = ++c->kept_clock;
                return 0;
            }
        }
        bool met = false;
        for (auto& k : c->seen) met = met || k == key;
        if (met) {                                                        // second sighting: record the whole loop and keep it
            cudaGraph_t graph; cudaGraphExec_t exec; long long launches = 0; int rc = 0;
            if (record_iterations(c, times, body, &graph, &exec, &launches, &rc)) {
                if (c->kept.size() >= 4) {                                // drop the least recently used (not in flight: launches are stream ordered,
                    size_t old = 0;                                       //  and destroying an exec waits for nothing it still needs)
                    for (size_t i = 1; i < c->kept.size(); ++i) if (c->kept[i].stamp < c->kept[old].stamp) old = i;
                    SLM_CUDA(cudaStreamSynchronize(c->stream));
                    cudaGraphExecDestroy(c->kept[old].exec); cudaGraphDestroy(c->kept[old].graph);
                    c->kept.erase(c->kept.begin() + old);
                }
                SLM_CUDA(cudaGraphLaunch(exec, c->stream));
                c->launches += launches;
                c->kept.push_back({key, exec, graph, launches, ++c->kept_clock});
                return 0;
            }
            if (rc) return rc;
        } else {
            if (c->seen.size() >= 4) c->seen.erase(c->seen.begin());
            c->seen.push_back(key);
        }
    }
    cudaGetLastError();
#else
    (void)batch; (void)key;
#endif
    for (int i = 0; i < times; ++i) SLM_TRY(body());
    return 0;
}

extern "C" const char* slm_last_error(void) { return g_err.c_str(); }
extern "C" int slm_version(void) { return 104; }
extern "C" int slm_supported_lengths(int* out, int cap) { return supported_lengths(out, cap); }

extern "C" void slm_ctx_destroy(slm_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
#ifndef SLM_EMULATE
    for (auto& r : c->replays) { cudaGraphExecDestroy(r.exec); cudaGraphDestroy(r.graph); cudaEventDestroy(r.done); }
    for (auto& k : c->kept) { cudaGraphExecDestroy(k.exec); cudaGraphDestroy(k.graph); }
    if (c->capture_stream) cudaStreamDestroy(c->capture_stream);
#endif
    for (void* p : c->owned) cudaFree(p);
    delete c;
}

extern "C" int slm_ctx_create(slm_ctx** out, int device, int H, int W, int max_batch, int precision, void* stream) {
    if (!out || max_batch < 1 || (precision != PREC_F32 && precision != PREC_F64)) return fail(SLM_ERR_ARG, "slm_ctx_create: bad argument");
    const LineTable* row = find_line_table(W, precision);
    const LineTable* col = find_line_table(H, precision);
    if (!row || !col) {
        char buf[160];
        snprintf(buf, sizeof buf, "unsupported plane shape %dx%d: rows and columns must be one of the built line lengths (", H, W);
        std::string both, rows;
        int lens[64];
        const int n = supported_lengths(lens, 64);
        for (int i = 0; i < n && i < 64; ++i) {
            std::string& s = find_line_table(lens[i], precision)->rows_only ? rows : both;
            s += (s.empty() ? "" : ", ") + std::to_string(lens[i]);
        }
        return fail(SLM_ERR_SHAPE, buf + both + (rows.empty() ? "" : "; row length only: " + rows) + ")");
    }
    if (H % row->rows_per_cta != 0 || W % col->cols_per_cta != 0) return fail(SLM_ERR_SHAPE, "plane shape not divisible by the CTA tile");
    SLM_CUDA(cudaSetDevice(device));
    slm_ctx* c = new slm_ctx;
    c->device = device; c->H = H; c->W = W; c->max_batch = max_batch; c->prec = precision;
    c->stream = (cudaStream_t)stream;
    c->row = row; c->col = col;
    c->row32 = find_line_table(W, PREC_F32); c->col32 = find_line_table(H, PREC_F32);
    row->prepare(); col->prepare(); c->row32->prepare(); c->col32->prepare();
    const size_t plane = (size_t)H * W, cs = 2 * real_size(precision);
    int rc = 0;
    auto A = [&](void** p, size_t n) { if (!rc) rc = dev_alloc(c, p, n); };
    A(&c->X, (size_t)max_batch * plane * cs);
    A(&c->Y, (size_t)max_batch * plane * cs);
    c->tiles = W / col->cols_per_cta;
    const int tiles32 = W / c->col32->cols_per_cta;
    const int tmax = c->tiles > tiles32 ? c->tiles : tiles32;
    A((void**)&c->stats, (size_t)max_batch * sizeof(PlaneStats));
    A((void**)&c->partial, (size_t)max_batch * tmax * sizeof(Partial));
    A((void**)&c->counter, (size_t)max_batch * sizeof(unsigned));
    A((void**)&c->fused, 3 * (size_t)max_batch * sizeof(unsigned));
    A((void**)&c->norm, (size_t)max_batch * sizeof(double));
    A(&c->lut, 256 * real_size(precision));
    A((void**)&c->lut32, 256 * sizeof(float));
    if (!rc) rc = make_twiddles(c, W, precision, &c->tw_row);
    if (!rc) rc = make_twiddles(c, H, precision, &c->tw_col);
    if (!rc && precision == PREC_F64) { rc = make_twiddles(c, W, PREC_F32, &c->tw_row32); if (!rc) rc = make_twiddles(c, H, PREC_F32, &c->tw_col32); }
    if (!rc && precision == PREC_F32) { c->tw_row32 = c->tw_row; c->tw_col32 = c->tw_col; }
    if (!rc) rc = ensure_loops(c, 256);
    if (!rc) rc = setup_groups(c);
    if (!rc && cudaMemset(c->counter, 0, (size_t)max_batch * sizeof(unsigned)) != cudaSuccess) rc = fail(SLM_ERR_CUDA, "cudaMemset(counter)");
    if (!rc && cudaMemset(c->fused, 0, 3 * (size_t)max_batch * sizeof(unsigned)) != cudaSuccess) rc = fail(SLM_ERR_CUDA, "cudaMemset(fused)");
    if (!rc && cudaMemset(c->stats, 0, (size_t)max_batch * sizeof(PlaneStats)) != cudaSuccess) rc = fail(SLM_ERR_CUDA, "cudaMemset(stats)");
    if (rc) { std::string keep = g_err; slm_ctx_destroy(c); g_err = keep; return rc; }
    *out = c;
    return 0;
}

extern "C" size_t slm_ctx_workspace_bytes(const slm_ctx* c) { return c ? c->bytes : 0; }

extern "C" int slm_ctx_profile(slm_ctx* c, int enable) {
    if (!c) return fail(SLM_ERR_ARG, "slm_ctx_profile: null context");
    c->profiling = enable != 0;
    return 0;
}
// ms[k], count[k] for k < 6: row pass, column pass, column max pre-pass, plain row, plain column, elementwise
extern "C" int slm_ctx_profile_read(slm_ctx* c, double* ms, long long* count) {
    if (!c || !ms || !count) return fail(SLM_ERR_ARG, "slm_ctx_profile_read: null argument");
    for (int k = 0; k < K_KINDS; ++k) { ms[k] = 0; count[k] = 0; }
#ifndef SLM_EMULATE
    SLM_CUDA(cudaSetDevice(c->device));
    SLM_CUDA(cudaStreamSynchronize(c->stream));
    for (auto& t : c->timed) {
        float e = 0;
        cudaEventElapsedTime(&e, t.a, t.b);
        ms[t.kind] += e; count[t.kind]++;
        cudaEventDestroy(t.a); cudaEventDestroy(t.b);
    }
    c->timed.clear();
#endif
    return 0;
}
extern "C" long long slm_ctx_launch_count(const slm_ctx* c) { return c ? c->launches : 0; }

static int check_batch(slm_ctx* c, int batch, const char* who) {
    if (!c) return fail(SLM_ERR_ARG, std::string(who) + ": null context");
    if (!c->col) return fail(SLM_ERR_ARG, std::string(who) + ": this is a row-slab context (slm_rows_create)");
    if (batch < 1 || batch > c->max_batch) return fail(SLM_ERR_ARG, std::string(who) + ": batch exceeds the context's max_batch");
    SLM_CUDA(cudaSetDevice(c->device));
    return 0;
}

// host LUT (double[256]) -> device R[256] and float[256]
static int upload_lut(slm_ctx* c, const double* lut) {
    if (c->lut_valid && memcmp(c->lut_host, lut, sizeof c->lut_host) == 0) return 0;     // unchanged since the last run: no copy, no sync
    // (a copy from pageable memory is staged by the driver before the call returns, and the staging arrays are the
    //  context's own: no synchronisation -- GD and GS alternate their tables in error_evolution_curves)
    memcpy(c->lut_host, lut, sizeof c->lut_host);
    c->lut_valid = true;
    for (int i = 0; i < 256; ++i) c->lut_host_f[i] = (float)lut[i];
    SLM_CUDA(cudaMemcpyAsync(c->lut32, c->lut_host_f, sizeof c->lut_host_f, cudaMemcpyHostToDevice, c->stream));
    if (c->prec == PREC_F64) SLM_CUDA(cudaMemcpyAsync(c->lut, c->lut_host, sizeof c->lut_host, cudaMemcpyHostToDevice, c->stream));
    else SLM_CUDA(cudaMemcpyAsync(c->lut, c->lut_host_f, sizeof c->lut_host_f, cudaMemcpyHostToDevice, c->stream));
    return 0;
}

// Programmatic dependent launch for the passes of this run?  (env SLM_PDL=0/1 overrides.)
static void choose_pdl(slm_ctx* c, int batch) {
#ifndef SLM_EMULATE
    static const char* force = getenv("SLM_PDL");
    tl_pdl = force ? force[0] == '1' : (long long)batch * c->H * c->W <= (1ll << 21);
#else
    (void)c; (void)batch;
#endif
}

static int begin_run(slm_ctx* c, int batch, const double* norm, int max_loops) {
    choose_pdl(c, batch);
    SLM_TRY(ensure_loops(c, max_loops));
    SLM_CUDA(cudaMemsetAsync(c->stats, 0, (size_t)batch * sizeof(PlaneStats), c->stream));
    if (c->fused) SLM_CUDA(cudaMemsetAsync(c->fused, 0, 3 * (size_t)c->max_batch * sizeof(unsigned), c->stream));
    if (norm) SLM_CUDA(cudaMemcpyAsync(c->norm, norm, (size_t)batch * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    return 0;
}

static const int kEwThreads = 256;
static unsigned ew_blocks(long long n) { long long b = (n + kEwThreads - 1) / kEwThreads; return (unsigned)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b)); }

// A = ifft2(amplitude) into c->Y (algorithms.py:27 / :155); returns the RowSource that reads it
static int setup_field(slm_ctx* c, int batch, const uint8_t* T8, const void* amp_real, int setup_c64, int* source) {
    const bool f32path = (c->prec == PREC_F32) || setup_c64;
    const LineTable* row = f32path ? c->row32 : c->row;
    const LineTable* col = f32path ? c->col32 : c->col;
    PlainRowArgs ra{};
    ra.B = batch; ra.H = c->H; ra.inverse = 1; ra.out = c->X;
    ra.tw = f32path ? c->tw_row32 : c->tw_row;
    if (T8) { ra.input = IN_LUT_U8; ra.T8 = T8; ra.lut = f32path ? (const void*)c->lut32 : (const void*)c->lut; }
    else {
        if (!amp_real) return fail(SLM_ERR_ARG, "setup: neither target_u8 nor amp_real given");
        ra.input = IN_REAL; ra.in = amp_real;
        if (f32path && c->prec == PREC_F64) {   // narrow the float64 plane the way scipy's _asfarray does for float32 data
            const long long n = (long long)batch * c->H * c->W;
            { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH((convert_kernel<double, float>), dim3(ew_blocks(n)), dim3(kEwThreads), 0, c->stream,
                       static_cast<const double*>(amp_real), static_cast<float*>(c->Y), n); }
            ra.in = c->Y;
        }
    }
    SLM_TIMED(K_ROW_PLAIN, row->row_plain(ra, c->stream));
    PlainColArgs ca{};
    ca.B = batch; ca.W = c->W; ca.output = OUT_COMPLEX; ca.inverse = 1; ca.scale = 1.0 / ((double)c->H * c->W);
    ca.in = c->X; ca.out = c->Y; ca.tw = f32path ? c->tw_col32 : c->tw_col;
    if (c->use_groups && col == c->col) SLM_TRY(launch_group(c, CGM_COMPLEX, batch, nullptr, &c->map_y, 1, ca.scale));
    else SLM_TIMED(K_COL_PLAIN, col->col_plain(ca, c->stream));
    *source = f32path ? ROW_FROM_A32 : ROW_FROM_A;
    return 0;
}

static PlainColArgs stats_args(slm_ctx* c, int batch, int output, void* out) {
    PlainColArgs a{};
    a.B = batch; a.W = c->W; a.output = output; a.inverse = 0; a.scale = 1.0;
    a.in = c->X; a.out = out; a.norm = c->norm; a.stats = c->stats; a.partial = c->partial; a.counter = c->counter;
    a.tw = c->tw_col;
    return a;
}

// max |C|^2 of the column transform of X -> stats (GS iteration 0 / every GD iteration / preview)
static int run_stats(slm_ctx* c, int batch) {
    if (c->use_groups) return launch_group(c, CGM_STATS, batch, nullptr, nullptr, 0, 1.0);
    SLM_TIMED(K_COL_STATS, c->col->col_plain(stats_args(c, batch, OUT_STATS, nullptr), c->stream));
    return 0;
}

extern "C" int slm_fft2(slm_ctx* c, int batch, const void* in, void* out, int inverse) {
    SLM_TRY(check_batch(c, batch, "slm_fft2"));
    if (!in || !out) return fail(SLM_ERR_ARG, "slm_fft2: null plane");
    PlainRowArgs ra{};
    ra.B = batch; ra.H = c->H; ra.input = IN_COMPLEX; ra.inverse = inverse; ra.in = in; ra.out = c->X; ra.tw = c->tw_row;
    SLM_TIMED(K_ROW_PLAIN, c->row->row_plain(ra, c->stream));
    PlainColArgs ca{};
    ca.B = batch; ca.W = c->W; ca.output = OUT_COMPLEX; ca.inverse = inverse;
    ca.scale = inverse ? 1.0 / ((double)c->H * c->W) : 1.0;
    ca.in = c->X; ca.out = out; ca.tw = c->tw_col;
    if (c->use_groups) {
        TileMap map_out;
        SLM_TRY(make_tile_map(c, out, (long long)batch * c->H, &map_out));
        SLM_TRY(launch_group(c, CGM_COMPLEX, batch, nullptr, &map_out, inverse, ca.scale));
    } else {
        SLM_TIMED(K_COL_PLAIN, c->col->col_plain(ca, c->stream));
    }
    return 0;
}

// The start of a loop run (GS, weighted GS, GD): the checks the three entry points share -- their messages carry the
// entry point's name `who` -- the run's state, the table, and the fields of the row and column arguments that do not
// depend on the algorithm.  `given`: the entry point's own required pointers, which `required` names; `refused`: why
// the entry point refuses one of its own arguments, or null.
static int begin_loop(slm_ctx* c, int batch, const char* who, const char* loops_msg, bool given, const char* required,
                      const char* table_msg, const char* refused, const uint8_t* T8, const void* Treal, const void* plane2, const double* lut,
                      const double* norm, const void* inc_amp, int max_loops, double tolerance, double* hologram_out,
                      RowArgs* ra, ColArgs* ca) {
    const std::string w(who);
    SLM_TRY(check_batch(c, batch, who));
    if (max_loops < 1) return fail(SLM_ERR_ARG, w + ": " + loops_msg);
    if (!given) return fail(SLM_ERR_ARG, w + ": " + required + " are required");
    if (T8 ? !lut : !(Treal && plane2)) return fail(SLM_ERR_ARG, w + ": " + table_msg);
    if (refused) return fail(SLM_ERR_ARG, w + ": " + refused);
    SLM_TRY(begin_run(c, batch, norm, max_loops));
    if (T8) SLM_TRY(upload_lut(c, lut));

    memset(ra, 0, sizeof *ra);                                      // zero padding too: the loop's graph key is made of these bytes
    ra->B = batch; ra->H = c->H; ra->Y = c->Y; ra->X = c->X; ra->inc = inc_amp; ra->stats = c->stats;
    ra->inv_hw = 1.0 / ((double)c->H * c->W); ra->hologram = hologram_out; ra->tw = c->tw_row;
    memset(ca, 0, sizeof *ca);
    ca->B = batch; ca->W = c->W; ca->X = c->X; ca->Y = c->Y; ca->T8 = T8; ca->Treal = Treal; ca->plane2 = plane2;
    ca->lut = c->lut; ca->norm = c->norm; ca->stats = c->stats; ca->partial = c->partial; ca->counter = c->counter;
    ca->err_curve = c->err_curve; ca->max_loops = max_loops; ca->tolerance = tolerance;
    ca->inv_hw = ra->inv_hw; ca->tw = c->tw_col;
    return 0;
}

// Iterations 0 .. max_loops-2 (Fourier-plane step + SLM-plane pass), replayed under a key of `family` (the kernel family)
// and every argument the loop's launches are made of; then the last iteration, which ends with the final pass.
template <class F> static int run_loop(slm_ctx* c, int batch, const char* family, int alg, RowArgs& ra, const ColArgs& ca,
                                       F fourier_step) {
    ra.source = ROW_FROM_Y;
    std::string key(family);
    double* const hologram = ra.hologram;
    ra.hologram = nullptr;                                          // (only the final pass -- outside the loop -- writes the hologram)
    key.append(reinterpret_cast<const char*>(&ra), sizeof ra).append(reinterpret_cast<const char*>(&ca), sizeof ca);
    key.append(reinterpret_cast<const char*>(&batch), sizeof batch);
    ra.hologram = hologram;
    SLM_TRY(replay_iterations(c, batch, ca.max_loops - 1, key, [&]() -> int {
        SLM_TRY(fourier_step());
        SLM_TIMED(K_ROW_PASS, c->row->row_pass(alg, ra, c->stream));
        return 0;
    }));
    SLM_TRY(fourier_step());
    ra.final_pass = 1;
    SLM_TIMED(K_ROW_PASS, c->row->row_pass(alg, ra, c->stream));
    return 0;
}

// GS and weighted GS after begin_loop.  Weighted GS runs the launches of GS's one-CTA-per-tile branch ("gs/plain") at
// every batch size, with the GSW forms of the max pre-pass and of the column pass (col_pass_tile<ALG_GSW>).  The
// persistent column kernels have no room for a weight tile (col_warp.cuh: three 64 KB tile buffers), so the context's
// batch does not choose a kernel for it.
//
// Multi-plane GS (ra.planes > 0) is GS with the multi-plane row pass (ALG_MP): `batch` counts planes, ra.B holograms.
static int gs_loop(slm_ctx* c, int batch, bool weighted, RowArgs& ra, ColArgs& ca, const uint8_t* T8, const void* amp_real,
                   const void* phasor0, int setup_c64, double* expected_out) {
    const bool multiplane = ra.planes > 0;
    const int row_alg = multiplane ? ALG_MP : ALG_GS;
    if (phasor0) { ra.source = ROW_FROM_FIELD; ra.field = phasor0; }
    else {
        int src = 0;
        SLM_TRY(setup_field(c, batch, T8, amp_real, setup_c64, &src));
        ra.source = src; ra.A32 = c->Y; ra.field = c->Y;
    }
    SLM_TIMED(K_ROW_PASS, c->row->row_pass(row_alg, ra, c->stream));
    // Fewer tiles than SMs (one SLM-size plane): the persistent tile pipeline of the column-group kernels has nothing to
    // pipeline, and the plain column kernel -- one CTA per tile, CTA-wide transforms -- has the shorter latency
    // (measured per 100 iterations of one 1024^2 plane: 1.91 against 2.11 ms; 512^2 x 20: 0.35 against 0.39 ms; from
    // two planes on the pipeline wins).  Decided per CONTEXT (its largest batch), not per run: the two kernels round
    // differently, and a plane's result must not depend on how many planes share its batch (the tail of a movie).  One
    // kernel family per run also because the expected outcome below takes its maximum with the arithmetic that made
    // the transform.  SLM_GS_GROUPS=1 keeps the pipeline (tests compare contexts of different sizes bit for bit).
    const bool groups = !weighted && c->use_groups &&
                        ((long long)c->max_batch * (c->W / c->col->cols_per_cta) > c->persist_ctas || getenv("SLM_GS_GROUPS"));
    // exact scale of iteration 0 so the one-pass error of later iterations is well conditioned (weighted: and P_0 for sigma_0)
    if (weighted) SLM_TIMED(K_COL_STATS, c->col->col_pass(ALG_GSW_STATS, ca, c->stream));
    else if (groups) SLM_TRY(run_stats(c, batch));
    else SLM_TIMED(K_COL_STATS, c->col->col_plain(stats_args(c, batch, OUT_STATS, nullptr), c->stream));

    const int col_alg = weighted ? ALG_GSW : ALG_GS;
    const char* family = weighted ? "gsw/plain" : multiplane ? (groups ? "mp/pipeline" : "mp/plain") : (groups ? "gs/pipeline" : "gs/plain");
    SLM_TRY(run_loop(c, batch, family, row_alg, ra, ca, [&]() -> int {
        if (groups) SLM_TRY(launch_group(c, CGM_GS, batch, &ca, &c->map_y, 0, 1.0));
        else SLM_TIMED(K_COL_PASS, c->col->col_pass(col_alg, ca, c->stream));
        return 0;
    }));
    if (expected_out) {
        PlainColArgs ia = stats_args(c, batch, OUT_INTENSITY_GS, expected_out);
        if (groups) {
            // C = fft2(B) of the last iteration once more, by the SAME kernel arithmetic that took its max, kept in X;
            // the intensity pass then only scales |C|^2 (max(expected_outcome) == norm like the reference's, :36-37)
            SLM_TRY(launch_group(c, CGM_STATS_KEEP, batch, nullptr, &c->map_x, 0, 1.0, 1));
            ia.skip_fft = 1;
        }
        SLM_TIMED(K_COL_PLAIN, c->col->col_plain(ia, c->stream));
    }
    return 0;
}

extern "C" int slm_gs_run(slm_ctx* c, int batch, const uint8_t* T8, const void* Treal, const void* amp_real,
                          const double* amp_lut, const double* norm, const void* inc_amp, const void* phasor0,
                          int setup_c64, int max_loops, double tolerance, double* hologram_out, double* expected_out) {
    RowArgs ra; ColArgs ca;
    SLM_TRY(begin_loop(c, batch, "slm_gs_run", "max_loops must be >= 1 (the reference raises UnboundLocalError for 0)",
                       norm && hologram_out, "norm and hologram_out", "give target_u8 + amp_lut, or target_real + amp_real",
                       nullptr, T8, Treal, amp_real, amp_lut, norm, inc_amp, max_loops, tolerance, hologram_out, &ra, &ca));
    return gs_loop(c, batch, false, ra, ca, T8, amp_real, phasor0, setup_c64, expected_out);
}

extern "C" int slm_gsw_run(slm_ctx* c, int batch, const uint8_t* T8, const void* Treal, const void* amp_real,
                           const double* amp_lut, const double* norm, const void* inc_amp, const void* phasor0,
                           int setup_c64, int max_loops, double tolerance, double* hologram_out, double* expected_out,
                           const double* target_sum, void* weights, double weight_limit) {
    RowArgs ra; ColArgs ca;
    SLM_TRY(begin_loop(c, batch, "slm_gsw_run", "max_loops must be >= 1", norm && hologram_out && target_sum && weights,
                       "norm, target_sum, weights and hologram_out", "give target_u8 + amp_lut, or target_real + amp_real",
                       weight_limit >= 1.0 ? nullptr : "weight_limit must be >= 1",
                       T8, Treal, amp_real, amp_lut, norm, inc_amp, max_loops, tolerance, hologram_out, &ra, &ca));
    if (!c->target_sum) {
        SLM_TRY(dev_alloc(c, (void**)&c->target_sum, (size_t)c->max_batch * sizeof(double)));
        SLM_TRY(dev_alloc(c, (void**)&c->signal_sum, (size_t)c->max_batch * sizeof(double)));
        SLM_TRY(dev_alloc(c, (void**)&c->signal_partial, (size_t)c->max_batch * c->tiles * sizeof(double)));
    }
    SLM_CUDA(cudaMemcpyAsync(c->target_sum, target_sum, (size_t)batch * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    ca.weights = weights; ca.target_sum = c->target_sum; ca.signal_sum = c->signal_sum; ca.signal_partial = c->signal_partial;
    ca.weight_limit = weight_limit;
    return gs_loop(c, batch, true, ra, ca, T8, amp_real, phasor0, setup_c64, expected_out);
}

// Multi-plane GS: the defocus tables lens_y[k][i] = exp(i alpha_k (i - H/2)^2) and lens_x[k][j] (W) of `planes` planes, in
// the context's precision.  Phases are evaluated in extended precision and reduced mod 2 pi before sin / cos, as in
// make_twiddles.  Uploaded when the alphas differ from those of the previous run.
static const int kMaxPlanes = 8;
static int upload_lenses(slm_ctx* c, int planes, const double* alpha) {
    const size_t cs = 2 * real_size(c->prec);
    if (!c->lens_y) {
        SLM_TRY(dev_alloc(c, &c->lens_y, (size_t)kMaxPlanes * c->H * cs));
        SLM_TRY(dev_alloc(c, &c->lens_x, (size_t)kMaxPlanes * c->W * cs));
    }
    if (c->lens_alpha.size() == (size_t)planes && memcmp(c->lens_alpha.data(), alpha, planes * sizeof(double)) == 0) return 0;
    c->lens_alpha.assign(alpha, alpha + planes);
    const long double two_pi = 6.283185307179586476925286766559005768L;
    for (int axis = 0; axis < 2; ++axis) {
        const int n = axis == 0 ? c->H : c->W;
        c->lens_host_d.resize(2 * (size_t)planes * n);
        c->lens_host_f.resize(2 * (size_t)planes * n);
        for (int k = 0; k < planes; ++k) {
            for (int i = 0; i < n; ++i) {
                const long double d = (long double)i - (long double)n / 2;        // lens_kernel's centre (elementwise.cuh)
                const long double ph = fmodl((long double)alpha[k] * (d * d), two_pi);
                const size_t q = 2 * ((size_t)k * n + i);
                c->lens_host_d[q] = (double)cosl(ph); c->lens_host_d[q + 1] = (double)sinl(ph);
                c->lens_host_f[q] = (float)cosl(ph); c->lens_host_f[q + 1] = (float)sinl(ph);
            }
        }
        // (a copy from pageable memory is staged by the driver before the call returns, see upload_lut)
        const void* src = c->prec == PREC_F64 ? (const void*)c->lens_host_d.data() : (const void*)c->lens_host_f.data();
        SLM_CUDA(cudaMemcpyAsync(axis == 0 ? c->lens_y : c->lens_x, src, (size_t)planes * n * cs, cudaMemcpyHostToDevice, c->stream));
    }
    return 0;
}

// The multi-plane entry points' own refusals (after the context): `planes` outside 1..kMaxPlanes and `holograms` x
// `planes` above the context's batch fail at once; a missing or non-finite defocus, or a rows-only context, is left
// in `refused` for begin_loop, which names the entry point.
static int check_multiplane(slm_ctx* c, const std::string& who, int holograms, int planes, const double* defocus,
                            std::string* refused) {
    if (!c) return fail(SLM_ERR_ARG, who + ": null context");
    if (planes < 1 || planes > kMaxPlanes) return fail(SLM_ERR_ARG, who + ": planes must be in 1.." + std::to_string(kMaxPlanes));
    if (holograms < 1 || (long long)holograms * planes > c->max_batch)
        return fail(SLM_ERR_ARG, who + ": holograms * planes must be in 1..max_batch of the context");
    if (!defocus) *refused = "defocus is required";
    for (int k = 0; defocus && k < planes && refused->empty(); ++k)
        if (!std::isfinite(defocus[k])) *refused = "defocus[" + std::to_string(k) + "] is not finite";
    if (refused->empty() && c->row && c->row->rows_only) *refused = "no multi-plane pass for rows of " + std::to_string(c->W) + " points";
    return 0;
}

// The defocus tables and the multi-plane fields of the row arguments: ra.B counts holograms from here on.
static int multiplane_rows(slm_ctx* c, RowArgs& ra, int holograms, int planes, const double* defocus) {
    SLM_TRY(upload_lenses(c, planes, defocus));
    ra.B = holograms; ra.planes = planes; ra.lens_y = c->lens_y; ra.lens_x = c->lens_x;
    for (int k = 0; k < planes; ++k)
        if (defocus[k] != 0.0) ra.lens_mask |= 1 << k;
    return 0;
}

extern "C" int slm_gs_multiplane_run(slm_ctx* c, int holograms, int planes, const uint8_t* T8, const void* Treal,
                                     const void* amp_real, const double* amp_lut, const double* norm, const double* defocus,
                                     const void* inc_amp, const void* phasor0, int setup_c64, int max_loops, double tolerance,
                                     double* hologram_out, double* expected_out) {
    const std::string who = "slm_gs_multiplane_run";
    std::string refused;
    SLM_TRY(check_multiplane(c, who, holograms, planes, defocus, &refused));
    RowArgs ra; ColArgs ca;
    SLM_TRY(begin_loop(c, holograms * planes, who.c_str(), "max_loops must be >= 1 (the reference raises UnboundLocalError for 0)",
                       norm && hologram_out, "norm and hologram_out", "give target_u8 + amp_lut, or target_real + amp_real",
                       refused.empty() ? nullptr : refused.c_str(),
                       T8, Treal, amp_real, amp_lut, norm, inc_amp, max_loops, tolerance, hologram_out, &ra, &ca));
    SLM_TRY(multiplane_rows(c, ra, holograms, planes, defocus));
    return gs_loop(c, holograms * planes, false, ra, ca, T8, amp_real, phasor0, setup_c64, expected_out);
}

// GD and multi-plane GD after begin_loop, with ra.x and ra.lr set: the first pass, the choice of the Fourier-plane form,
// the loop and the expected outcome.  Multi-plane GD (ra.planes > 0) is GD with the multi-plane row pass (ALG_MPGD):
// `batch` counts planes, ra.B holograms; its kept graphs have families of their own.
static int gd_loop(slm_ctx* c, int batch, RowArgs& ra, ColArgs& ca, double* expected_out) {
    const bool multiplane = ra.planes > 0;
    const int row_alg = multiplane ? ALG_MPGD : ALG_GD;
    ra.source = ROW_FROM_FIELD;
    SLM_TIMED(K_ROW_PASS, c->row->row_pass(row_alg, ra, c->stream));
    // The fused pass saves a launch and a trip of the field through L2/HBM per iteration, but its CTAs wait for each
    // other once per plane and it leaves the SMs beyond a whole number of planes idle: measured faster for a few
    // planes (latency bound: 2.9 vs 3.3 ms per 100-iteration hologram), slower for a large batch (47.9 vs 46.4 ms).
    // Larger batches: the same single pass with the wait taken out of the SMs' way (CGM_GD_PIPE).  SLM_GD_FORM =
    // fused | pipe | two_pass overrides the choice (tests, A/B measurements); read per call.
    const char* form = getenv("SLM_GD_FORM");
    const bool few = (long long)batch * (c->W / c->col->cols_per_cta) <= 4LL * c->persist_ctas;
    bool fused = c->use_groups && c->fused_ctas && !getenv("SLM_NO_FUSED_GD") && few;
    bool pipe = c->use_groups && c->pipe_ok && !getenv("SLM_NO_FUSED_GD") && !fused;
    if (form && c->use_groups) {
        fused = form[0] == 'f' && c->fused_ctas;
        pipe = form[0] == 'p' && c->pipe_ok;
    }
    // two-pass form without the column groups: the max pass keeps the transformed field in X (below)
    if (!c->use_groups) ca.skip_forward = 1;
    const char* family = multiplane ? (fused ? "mgdf" : (pipe ? "mgdp" : "mgd2")) : (fused ? "gdf" : (pipe ? "gdp" : "gd2"));
    SLM_TRY(run_loop(c, batch, family, row_alg, ra, ca, [&]() -> int {
        if (fused) {
            // one Fourier-plane pass: the tiles of a plane agree on amax(output_unnormed) (algorithms.py:86) between
            // their forward transforms and the gradient step
            SLM_TRY(launch_group(c, CGM_GD_FUSED, batch, &ca, &c->map_y, 0, 1.0));
        } else if (pipe) {
            SLM_TRY(launch_group(c, CGM_GD_PIPE, batch, &ca, &c->map_y, 0, 1.0));
        } else if (c->use_groups) {
            // med_output = fft2(...) is finished in place in X while its max is taken (algorithms.py:84-86),
            // so the gradient pass starts from the transformed field
            SLM_TRY(launch_group(c, CGM_STATS_KEEP, batch, nullptr, &c->map_x, 0, 1.0));
            SLM_TRY(launch_group(c, CGM_GD_POST, batch, &ca, &c->map_y, 0, 1.0));
        } else {
            // amax(output_unnormed), algorithms.py:86; the transformed field is kept in X so the gradient pass need not
            // transform again (ca.skip_forward)
            PlainColArgs sa = stats_args(c, batch, OUT_STATS, c->X);
            sa.keep = 1;
            SLM_TIMED(K_COL_STATS, c->col->col_plain(sa, c->stream));
            SLM_TIMED(K_COL_PASS, c->col->col_pass(ALG_GD, ca, c->stream));
        }
        return 0;
    }));
    if (expected_out) {
        PlainColArgs ia = stats_args(c, batch, OUT_INTENSITY_GD, expected_out);
        // two-pass form: X already holds med_output; one-pass forms: transform X once more (same kernel arithmetic), kept
        if (fused || pipe) SLM_TRY(launch_group(c, CGM_STATS_KEEP, batch, nullptr, &c->map_x, 0, 1.0, 1));
        ia.skip_fft = 1;
        SLM_TIMED(K_COL_PLAIN, c->col->col_plain(ia, c->stream));
    }
    return 0;
}

extern "C" int slm_gd_run(slm_ctx* c, int batch, const uint8_t* T8, const void* Treal, const void* mask_real,
                          const double* mask_lut, const double* norm, const void* inc_amp, void* x,
                          const double* lr_schedule, int max_loops, double tolerance, double* hologram_out,
                          double* expected_out) {
    RowArgs ra; ColArgs ca;
    SLM_TRY(begin_loop(c, batch, "slm_gd_run", "max_loops must be >= 1 (the reference raises UnboundLocalError for 0)",
                       norm && hologram_out && x && lr_schedule, "norm, x, lr_schedule and hologram_out",
                       "give target_u8 + mask_lut, or target_real + mask_real", nullptr,
                       T8, Treal, mask_real, mask_lut, norm, inc_amp, max_loops, tolerance, hologram_out, &ra, &ca));
    SLM_CUDA(cudaMemcpyAsync(c->lr, lr_schedule, (size_t)max_loops * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    ra.x = x; ra.lr = c->lr;
    return gd_loop(c, batch, ra, ca, expected_out);
}

extern "C" int slm_gd_multiplane_run(slm_ctx* c, int holograms, int planes, const uint8_t* T8, const void* Treal,
                                     const void* mask_real, const double* mask_lut, const double* norm, const double* defocus,
                                     const void* inc_amp, void* x, const double* lr_schedule, int max_loops, double tolerance,
                                     double* hologram_out, double* expected_out) {
    const std::string who = "slm_gd_multiplane_run";
    std::string refused;
    SLM_TRY(check_multiplane(c, who, holograms, planes, defocus, &refused));
    RowArgs ra; ColArgs ca;
    SLM_TRY(begin_loop(c, holograms * planes, who.c_str(), "max_loops must be >= 1 (the reference raises UnboundLocalError for 0)",
                       norm && hologram_out && x && lr_schedule, "norm, x, lr_schedule and hologram_out",
                       "give target_u8 + mask_lut, or target_real + mask_real", refused.empty() ? nullptr : refused.c_str(),
                       T8, Treal, mask_real, mask_lut, norm, inc_amp, max_loops, tolerance, hologram_out, &ra, &ca));
    SLM_CUDA(cudaMemcpyAsync(c->lr, lr_schedule, (size_t)max_loops * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    ra.x = x; ra.lr = c->lr;
    // One plane at the Fourier plane is GD itself: it runs GD's row pass, so it gives GD's bits at GD's rate.  (The
    // multi-plane pass at K = 1 ran at 0.70-0.81 of GD's plane rate, DESIGN.md §4, and its fp64 results differed
    // from GD's in the last bit: the same arithmetic, compiled into a different kernel.)
    if (planes > 1 || defocus[0] != 0.0) {
        SLM_TRY(multiplane_rows(c, ra, holograms, planes, defocus));
        // the cost is the mean of the planes' errors: dEdF = sum_k G_k conj(L_k) inc / K
        ra.inv_hw = 1.0 / ((double)planes * c->H * c->W);
    }
    return gd_loop(c, holograms * planes, ra, ca, expected_out);
}

extern "C" int slm_fourier_guess(slm_ctx* c, int batch, const uint8_t* T8, const void* amp_real, const double* amp_lut,
                                 const void* inc_amp, int setup_c64, void* x_out) {
    SLM_TRY(check_batch(c, batch, "slm_fourier_guess"));
    if (!x_out || (T8 && !amp_lut)) return fail(SLM_ERR_ARG, "slm_fourier_guess: bad argument");
    if (T8) SLM_TRY(upload_lut(c, amp_lut));
    int src = 0;
    SLM_TRY(setup_field(c, batch, T8, amp_real, setup_c64, &src));
    const long long plane = (long long)c->H * c->W, n = plane * batch;
    const dim3 grid(ew_blocks(n)), block(kEwThreads);
    {
        LaunchTimer t_(c, K_ELEMENTWISE);
        if (c->prec == PREC_F32)
            SLM_LAUNCH((phasor_field_kernel<float, float>), grid, block, 0, c->stream, static_cast<const cpx<float>*>(c->Y),
                       static_cast<const float*>(inc_amp), static_cast<cpx<float>*>(x_out), n, plane);
        else if (src == ROW_FROM_A32)
            SLM_LAUNCH((phasor_field_kernel<double, float>), grid, block, 0, c->stream, static_cast<const cpx<float>*>(c->Y),
                       static_cast<const double*>(inc_amp), static_cast<cpx<double>*>(x_out), n, plane);
        else
            SLM_LAUNCH((phasor_field_kernel<double, double>), grid, block, 0, c->stream, static_cast<const cpx<double>*>(c->Y),
                       static_cast<const double*>(inc_amp), static_cast<cpx<double>*>(x_out), n, plane);
    }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

// "fourier" initial guess of multi-plane GD: x = inc exp(i angle(sum_k ifft2(amp_k) conj(L_k))), multi-plane GS's setup
// sum.  The setup field of every plane, then the multi-plane row pass in its final form writes the phase of the sum
// into X (G double planes fit in the context's max_batch complex planes), and slm_phase_phasor makes x of it.
extern "C" int slm_multiplane_fourier_guess(slm_ctx* c, int holograms, int planes, const uint8_t* T8, const void* amp_real,
                                            const double* amp_lut, const double* defocus, const void* inc_amp, int setup_c64,
                                            void* x_out) {
    const std::string who = "slm_multiplane_fourier_guess";
    std::string refused;
    SLM_TRY(check_multiplane(c, who, holograms, planes, defocus, &refused));
    SLM_TRY(check_batch(c, holograms * planes, who.c_str()));
    if (!refused.empty()) return fail(SLM_ERR_ARG, who + ": " + refused);
    if (!x_out || (T8 ? !amp_lut : !amp_real)) return fail(SLM_ERR_ARG, who + ": x_out, and target_u8 + amp_lut or amp_real, are required");
    if (T8) SLM_TRY(upload_lut(c, amp_lut));
    RowArgs ra;
    memset(&ra, 0, sizeof ra);
    int src = 0;
    SLM_TRY(setup_field(c, holograms * planes, T8, amp_real, setup_c64, &src));
    SLM_TRY(multiplane_rows(c, ra, holograms, planes, defocus));
    ra.H = c->H; ra.source = src; ra.A32 = c->Y; ra.field = c->Y; ra.tw = c->tw_row;
    ra.hologram = static_cast<double*>(c->X); ra.final_pass = 1;
    SLM_TIMED(K_ROW_PASS, c->row->row_pass(ALG_MP, ra, c->stream));
    const long long plane = (long long)c->H * c->W;
    return slm_phase_phasor(c, static_cast<const double*>(c->X), inc_amp, x_out, plane * holograms, plane);
}

extern "C" int slm_random_phasor(slm_ctx* c, const double* u, void* x_out, long long n, double divide_by) {
    if (!c) return fail(SLM_ERR_ARG, "slm_random_phasor: null context");
    SLM_CUDA(cudaSetDevice(c->device));
    if (!u || !x_out || n < 1 || divide_by == 0.0) return fail(SLM_ERR_ARG, "slm_random_phasor: bad argument");
    const dim3 grid(ew_blocks(n)), block(kEwThreads);
    {
        LaunchTimer t_(c, K_ELEMENTWISE);
        if (c->prec == PREC_F32) SLM_LAUNCH((random_phasor_kernel<float>), grid, block, 0, c->stream, u, static_cast<cpx<float>*>(x_out), n, divide_by);
        else SLM_LAUNCH((random_phasor_kernel<double>), grid, block, 0, c->stream, u, static_cast<cpx<double>*>(x_out), n, divide_by);
    }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int slm_mt19937_uniform(slm_ctx* c, const uint32_t* state, int pos, double* u, long long n, uint32_t* state_out) {
    if (!c) return fail(SLM_ERR_ARG, "slm_mt19937_uniform: null context");
    SLM_CUDA(cudaSetDevice(c->device));
    if (!state || !u || !state_out || n < 1 || pos < 0 || pos > 624 || (pos & 1)) return fail(SLM_ERR_ARG, "slm_mt19937_uniform: bad argument (pos must be even)");
    if (!c->mt_buf) SLM_TRY(dev_alloc(c, (void**)&c->mt_buf, (624 + 625) * sizeof(unsigned)));
    unsigned* dev = c->mt_buf;                       // [624 in][625 out]
    SLM_CUDA(cudaMemcpyAsync(dev, state, 624 * sizeof(unsigned), cudaMemcpyHostToDevice, c->stream));
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(mt19937_uniform_kernel, dim3(1), dim3(kMtThreads), 0, c->stream, dev, pos, u, n, dev + 624); }
    SLM_CUDA(cudaGetLastError());
    SLM_CUDA(cudaMemcpyAsync(state_out, dev + 624, 625 * sizeof(unsigned), cudaMemcpyDeviceToHost, c->stream));
    SLM_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
}

extern "C" int slm_phase_phasor(slm_ctx* c, const double* phase, const void* inc_amp, void* x_out, long long n, long long plane) {
    if (!c) return fail(SLM_ERR_ARG, "slm_phase_phasor: null context");
    SLM_CUDA(cudaSetDevice(c->device));
    if (!phase || !x_out || n < 1 || plane < 1) return fail(SLM_ERR_ARG, "slm_phase_phasor: bad argument");
    const dim3 grid(ew_blocks(n)), block(kEwThreads);
    {
        LaunchTimer t_(c, K_ELEMENTWISE);
        if (c->prec == PREC_F32) SLM_LAUNCH((phase_phasor_kernel<float>), grid, block, 0, c->stream, phase, static_cast<const float*>(inc_amp), static_cast<cpx<float>*>(x_out), n, plane);
        else SLM_LAUNCH((phase_phasor_kernel<double>), grid, block, 0, c->stream, phase, static_cast<const double*>(inc_amp), static_cast<cpx<double>*>(x_out), n, plane);
    }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int slm_single_trap_phase(slm_ctx* c, int H, int W, int row, int col, double* out) {
    if (!c) return fail(SLM_ERR_ARG, "slm_single_trap_phase: null context");
    SLM_CUDA(cudaSetDevice(c->device));
    if (!out || H < 1 || W < 1 || row < 0 || row >= H || col < 0 || col >= W) return fail(SLM_ERR_ARG, "slm_single_trap_phase: bad argument");
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(single_trap_kernel, dim3(ew_blocks((long long)H * W)), dim3(kEwThreads), 0, c->stream, out, H, W, row, col); }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int slm_trap_frames(slm_ctx* c, uint8_t* frames, int n_frames, int H, int W, const int* frame_y_x, int n_dots) {
    if (!c) return fail(SLM_ERR_ARG, "slm_trap_frames: null context");
    SLM_CUDA(cudaSetDevice(c->device));
    if (!frames || n_frames < 1 || H < 1 || W < 1 || n_dots < 0 || (n_dots && !frame_y_x)) return fail(SLM_ERR_ARG, "slm_trap_frames: bad argument");
    SLM_CUDA(cudaMemsetAsync(frames, 0, (size_t)n_frames * H * W, c->stream));
    if (n_dots) {
        LaunchTimer t_(c, K_ELEMENTWISE);
        SLM_LAUNCH(scatter_dots_kernel, dim3((unsigned)((n_dots + 255) / 256)), dim3(256), 0, c->stream, frames, frame_y_x, n_dots, (long long)H * W, W);
    }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

// ---- row-slab API: one very large plane split by rows over the ranks (slab-decomposed transform) ---------
extern "C" int slm_rows_create(slm_ctx** out, int device, int rows, int W, int precision, void* stream) {
    if (!out || rows < 1 || (precision != PREC_F32 && precision != PREC_F64)) return fail(SLM_ERR_ARG, "slm_rows_create: bad argument");
    const LineTable* row = find_line_table(W, precision);
    if (!row) return fail(SLM_ERR_SHAPE, "unsupported line length " + std::to_string(W));
    // the slab Fourier-plane kernel sums a line's partials per warp: a line is either within one warp or whole warps
    const int m = row->row_threads / row->rows_per_cta;
    if (m > 32 && m % 32 != 0)
        return fail(SLM_ERR_SHAPE, "line length " + std::to_string(W) + " is not supported on the slab path (" + std::to_string(m) +
                                       " threads per line: neither within one warp nor whole warps)");
    if (rows % row->rows_per_cta != 0 || rows % 32 != 0) return fail(SLM_ERR_SHAPE, "slab rows must be a multiple of 32 and of the CTA row tile");
    SLM_CUDA(cudaSetDevice(device));
    slm_ctx* c = new slm_ctx;
    c->device = device; c->H = rows; c->W = W; c->max_batch = 1; c->prec = precision;
    c->stream = (cudaStream_t)stream;
    c->row = row; c->col = nullptr;
    row->prepare();
    int rc = 0;
    auto A = [&](void** p, size_t n) { if (!rc) rc = dev_alloc(c, p, n); };
    A((void**)&c->stats, 2 * sizeof(PlaneStats));           // [0] the loop state, [1] stays zero (slm_rows_gs_row_pass)
    A(&c->lut, 256 * real_size(precision));
    A((void**)&c->lut32, 256 * sizeof(float));
    if (!rc) rc = make_twiddles(c, W, precision, &c->tw_row);
    if (!rc && cudaMemset(c->stats, 0, 2 * sizeof(PlaneStats)) != cudaSuccess) rc = fail(SLM_ERR_CUDA, "cudaMemset(stats)");
    if (rc) { std::string keep = g_err; slm_ctx_destroy(c); g_err = keep; return rc; }
    *out = c;
    return 0;
}

// exchange-layout block width the row kernels can address: a power-of-two number of runs of M = threads-per-line points
static bool block_width_ok(const slm_ctx* c, int wb) {
    if (wb == 0) return true;
    const int m = c->row->row_threads / c->row->rows_per_cta;
    if (wb < m || wb % m) return false;
    const int q = wb / m;
    return (q & (q - 1)) == 0;
}

extern "C" int slm_rows_fft(slm_ctx* c, const void* in, const uint8_t* in_u8, const double* lut, void* out, int inverse,
                            int block_in, int block_out) {
    if (!c || !out || (!in && !in_u8) || (in_u8 && !lut)) return fail(SLM_ERR_ARG, "slm_rows_fft: bad argument");
    SLM_CUDA(cudaSetDevice(c->device));
    if (in_u8) SLM_TRY(upload_lut(c, lut));
    PlainRowArgs ra{};
    ra.B = 1; ra.H = c->H; ra.inverse = inverse; ra.block_in = block_in; ra.block_out = block_out; ra.out = out; ra.tw = c->tw_row;
    if (in_u8) { ra.input = IN_LUT_U8; ra.T8 = in_u8; ra.lut = c->lut; } else { ra.input = IN_COMPLEX; ra.in = in; }
    SLM_TIMED(K_ROW_PLAIN, c->row->row_plain(ra, c->stream));
    return 0;
}

extern "C" int slm_rows_gs_row_pass(slm_ctx* c, const void* in, void* out, const void* inc_amp, int in_is_field, int final_pass,
                                    double* hologram) {
    if (!c || !in || (final_pass ? !hologram : !out)) return fail(SLM_ERR_ARG, "slm_rows_gs_row_pass: bad argument");
    SLM_CUDA(cudaSetDevice(c->device));
    RowArgs ra{};
    // A GS run on the slab ends where the caller stops issuing iterations: with tolerance <= 0 it runs them all and cuts
    // the error curve itself.  So its row passes read the record that stays zero, not the loop-ended flag, which an error
    // of exactly 0 sets (one bright pixel at the origin), and which would stop them while the Fourier-plane passes go on.
    ra.B = 1; ra.H = c->H; ra.Y = in; ra.field = in; ra.X = out; ra.inc = inc_amp; ra.stats = c->stats + 1; ra.hologram = hologram;
    ra.inv_hw = 1.0; ra.tw = c->tw_row; ra.final_pass = final_pass;
    ra.A32 = in;
    ra.source = in_is_field == 2 ? ROW_FROM_A32 : (in_is_field ? ROW_FROM_A : ROW_FROM_Y);
    SLM_TIMED(K_ROW_PASS, c->row->row_pass(ALG_GS, ra, c->stream));
    return 0;
}

extern "C" int slm_rows_fourier_pass(slm_ctx* c, int mode, const void* in, void* out, int block_w, const uint8_t* target_u8,
                                     const double* lut, double norm, double* partial, double* intensity) {
    if (!c || !in || !out || !partial || mode < RF_GS || mode > RF_GD_POST) return fail(SLM_ERR_ARG, "slm_rows_fourier_pass: bad argument");
    const bool has_target = mode != RF_GD_MAX;
    if (has_target && (!target_u8 || !lut)) return fail(SLM_ERR_ARG, "slm_rows_fourier_pass: this mode needs the target and its table");
    if (!block_width_ok(c, block_w))
        return fail(SLM_ERR_SHAPE, "slm_rows_fourier_pass: the exchange block width must be a power-of-two multiple of the line's thread count");
    SLM_CUDA(cudaSetDevice(c->device));
    if (has_target) SLM_TRY(upload_lut(c, lut));
    RowFourierArgs fa{};
    fa.rows = c->H; fa.block_w = block_w; fa.in = in; fa.out = out; fa.T8 = target_u8; fa.lut = c->lut; fa.stats = c->stats;
    fa.mode = mode; fa.norm = norm; fa.partial = partial; fa.intensity = intensity; fa.tw = c->tw_row;
    SLM_TIMED(mode == RF_GD_MAX ? K_COL_STATS : K_COL_PASS, c->row->row_fourier(fa, c->stream));
    return 0;
}

static int peer_ptrs(const void* const* peers, int n, PeerPtrs* out, const char* who) {
    if (n < 0 || n > 16 || (n && !peers)) return fail(SLM_ERR_ARG, std::string(who) + ": at most 16 peers");
    for (int i = 0; i < 16; ++i) out->p[i] = i < n ? const_cast<void*>(peers[i]) : nullptr;
    return 0;
}

extern "C" int slm_rows_reduce(slm_ctx* c, const double* partial, int rows, double* out4, const void* const* peer_gathered,
                               int n_peers, int self) {
    if (!c || !partial || !out4 || rows < 1) return fail(SLM_ERR_ARG, "slm_rows_reduce: bad argument");
    SLM_CUDA(cudaSetDevice(c->device));
    PeerPtrs pp;
    SLM_TRY(peer_ptrs(peer_gathered, n_peers, &pp, "slm_rows_reduce"));
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(rows_reduce_kernel, dim3(1), dim3(256), 0, c->stream, partial, rows, out4, pp, n_peers, self); }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int slm_rows_close(slm_ctx* c, const double* gathered, int world, double norm, double hw, int kind, double tolerance,
                              double* err_curve) {
    if (!c || !gathered || world < 1 || kind < CLOSE_MAX || kind > CLOSE_GD || (kind != CLOSE_MAX && !err_curve))
        return fail(SLM_ERR_ARG, "slm_rows_close: bad argument");
    SLM_CUDA(cudaSetDevice(c->device));
    using CloseKernel = void (*)(const double*, int, double, double, double, double*, PlaneStats*);
    static const CloseKernel kernels[2][3] = {     // [precision][kind]
        {rows_close_kernel<float, CLOSE_MAX>, rows_close_kernel<float, CLOSE_GS>, rows_close_kernel<float, CLOSE_GD>},
        {rows_close_kernel<double, CLOSE_MAX>, rows_close_kernel<double, CLOSE_GS>, rows_close_kernel<double, CLOSE_GD>}};
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(kernels[c->prec][kind], dim3(1), dim3(32), 0, c->stream, gathered, world, norm, hw,
                                                    tolerance, err_curve, c->stats); }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int slm_rows_reset(slm_ctx* c) {
    if (!c) return fail(SLM_ERR_ARG, "slm_rows_reset: null context");
    SLM_CUDA(cudaSetDevice(c->device));
    SLM_CUDA(cudaMemsetAsync(c->stats, 0, sizeof(PlaneStats), c->stream));
    return 0;
}

extern "C" int slm_rows_state(slm_ctx* c, double* scale, double* imax, int* iters, int* done) {
    if (!c) return fail(SLM_ERR_ARG, "slm_rows_state: null context");
    SLM_CUDA(cudaSetDevice(c->device));
    PlaneStats st;
    SLM_CUDA(cudaMemcpyAsync(&st, c->stats, sizeof st, cudaMemcpyDeviceToHost, c->stream));
    SLM_CUDA(cudaStreamSynchronize(c->stream));
    if (scale) *scale = st.scale;
    if (imax) *imax = st.imax;
    if (iters) *iters = st.iters;
    if (done) *done = st.done;
    return 0;
}

extern "C" int slm_rows_gd_row_pass(slm_ctx* c, const void* in, void* x, void* out, const double* lr_dev, int first, int final_pass,
                                    double* hologram) {
    if (!c || !x || !lr_dev || (!first && !in) || (final_pass ? !hologram : !out)) return fail(SLM_ERR_ARG, "slm_rows_gd_row_pass: bad argument");
    SLM_CUDA(cudaSetDevice(c->device));
    RowArgs ra{};
    ra.B = 1; ra.H = c->H; ra.Y = in; ra.field = in; ra.X = out; ra.x = x; ra.lr = lr_dev; ra.stats = c->stats; ra.hologram = hologram;
    ra.inv_hw = 1.0 / ((double)c->W * (double)c->W);              // scipy's ifft2 normalisation of the WHOLE (square) plane, algorithms.py:87-89
    ra.tw = c->tw_row; ra.final_pass = final_pass;
    ra.source = first ? ROW_FROM_FIELD : ROW_FROM_Y;
    SLM_TIMED(K_ROW_PASS, c->row->row_pass(ALG_GD, ra, c->stream));
    return 0;
}

extern "C" int slm_transpose_blocks_peer(slm_ctx* c, const void* in, const void* const* peers, int n_peers, int self, int rows, int W,
                                         int elem_bytes, int from_exchange) {
    if (!c || !in || n_peers < 1 || self < 0 || self >= n_peers) return fail(SLM_ERR_ARG, "slm_transpose_blocks_peer: bad argument");
    if (rows < 32 || rows % 32 || W != rows * n_peers) return fail(SLM_ERR_SHAPE, "slm_transpose_blocks_peer: W must be rows * peers, rows a multiple of 32");
    SLM_CUDA(cudaSetDevice(c->device));
    PeerPtrs pp;
    SLM_TRY(peer_ptrs(peers, n_peers, &pp, "slm_transpose_blocks_peer"));
    const int n_x = rows / 32;
    const dim3 grid(n_x * n_peers, rows / 32, 1), block(256);             // x: (tile, destination), destination fastest
    {
        LaunchTimer t_(c, K_ELEMENTWISE);
        if (elem_bytes == 16) SLM_LAUNCH((transpose_blocks_peer_kernel<cpx<double>>), grid, block, 0, c->stream, static_cast<const cpx<double>*>(in), pp, rows, W, from_exchange, self, n_x);
        else if (elem_bytes == 8) SLM_LAUNCH((transpose_blocks_peer_kernel<double>), grid, block, 0, c->stream, static_cast<const double*>(in), pp, rows, W, from_exchange, self, n_x);
        else if (elem_bytes == 1) SLM_LAUNCH((transpose_blocks_peer_kernel<unsigned char>), grid, block, 0, c->stream, static_cast<const unsigned char*>(in), pp, rows, W, from_exchange, self, n_x);
        else return fail(SLM_ERR_ARG, "slm_transpose_blocks_peer: elem_bytes must be 1, 8 or 16");
    }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int slm_transpose_blocks(slm_ctx* c, const void* in, void* out, int rows, int W, int elem_bytes, int from_exchange) {
    if (!c || !in || !out || in == out) return fail(SLM_ERR_ARG, "slm_transpose_blocks: bad argument");
    if (rows < 32 || rows % 32 || W % rows) return fail(SLM_ERR_SHAPE, "slm_transpose_blocks: rows must be a multiple of 32 dividing W");
    SLM_CUDA(cudaSetDevice(c->device));
    const dim3 grid(rows / 32, rows / 32, W / rows), block(256);
    {
        LaunchTimer t_(c, K_ELEMENTWISE);
        if (elem_bytes == 16) SLM_LAUNCH((transpose_blocks_kernel<cpx<double>>), grid, block, 0, c->stream, static_cast<const cpx<double>*>(in), static_cast<cpx<double>*>(out), rows, W, from_exchange);
        else if (elem_bytes == 8) SLM_LAUNCH((transpose_blocks_kernel<double>), grid, block, 0, c->stream, static_cast<const double*>(in), static_cast<double*>(out), rows, W, from_exchange);
        else if (elem_bytes == 1) SLM_LAUNCH((transpose_blocks_kernel<unsigned char>), grid, block, 0, c->stream, static_cast<const unsigned char*>(in), static_cast<unsigned char*>(out), rows, W, from_exchange);
        else return fail(SLM_ERR_ARG, "slm_transpose_blocks: elem_bytes must be 1, 8 or 16");
    }
    SLM_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int slm_read_curves(slm_ctx* c, int batch, int max_loops, double* err, int* iters) {
    SLM_TRY(check_batch(c, batch, "slm_read_curves"));
    if (max_loops < 1 || max_loops > c->loops_cap) return fail(SLM_ERR_ARG, "slm_read_curves: max_loops does not match the last run");
    std::vector<PlaneStats> st(batch);
    SLM_CUDA(cudaMemcpyAsync(st.data(), c->stats, (size_t)batch * sizeof(PlaneStats), cudaMemcpyDeviceToHost, c->stream));
    if (err) SLM_CUDA(cudaMemcpyAsync(err, c->err_curve, (size_t)batch * max_loops * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    unsigned timed_out = 0;
    if (c->fused) SLM_CUDA(cudaMemcpyAsync(&timed_out, c->fused + 2 * (size_t)c->max_batch, sizeof timed_out, cudaMemcpyDeviceToHost, c->stream));   // (the flag behind the pairs)
    SLM_CUDA(cudaStreamSynchronize(c->stream));
    if (timed_out) return fail(SLM_ERR_CUDA, "the fused Fourier-plane pass timed out waiting for the tiles of a plane (its CTAs were not all "
                                             "resident: is another kernel holding SMs?); set SLM_NO_FUSED_GD=1");
    if (iters) for (int b = 0; b < batch; ++b) iters[b] = st[b].iters;
    return 0;
}

extern "C" int slm_expected_outcome(slm_ctx* c, int batch, const double* hologram, const double* norm, double* out) {
    SLM_TRY(check_batch(c, batch, "slm_expected_outcome"));
    if (!hologram || !norm || !out) return fail(SLM_ERR_ARG, "slm_expected_outcome: null argument");
    SLM_TRY(begin_run(c, batch, norm, 1));
    PlainRowArgs ra{};
    ra.B = batch; ra.H = c->H; ra.input = IN_PHASE; ra.inverse = 0; ra.in = hologram; ra.out = c->X; ra.tw = c->tw_row;
    SLM_TIMED(K_ROW_PLAIN, c->row->row_plain(ra, c->stream));
    PlainColArgs ia = stats_args(c, batch, OUT_INTENSITY_PREVIEW, out);
    if (c->use_groups) { SLM_TRY(launch_group(c, CGM_STATS_KEEP, batch, nullptr, &c->map_x, 0, 1.0, 1)); ia.skip_fft = 1; }   // see slm_gs_run
    else SLM_TRY(run_stats(c, batch));
    SLM_TIMED(K_COL_PLAIN, c->col->col_plain(ia, c->stream));
    return 0;
}

extern "C" int slm_host_register(void* ptr, size_t bytes) {
    if (!ptr || !bytes) return fail(SLM_ERR_ARG, "slm_host_register: bad argument");
#ifdef SLM_EMULATE
    return 0;
#else
    const cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterDefault);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(SLM_ERR_CUDA, std::string("cudaHostRegister: ") + cudaGetErrorString(e)); }
    return 0;
#endif
}
extern "C" int slm_host_unregister(void* ptr) {
    if (!ptr) return fail(SLM_ERR_ARG, "slm_host_unregister: bad argument");
#ifdef SLM_EMULATE
    return 0;
#else
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(SLM_ERR_CUDA, std::string("cudaHostUnregister: ") + cudaGetErrorString(e)); }
    return 0;
#endif
}

#define SLM_EW_PROLOGUE(who)                                              \
    if (!c) return fail(SLM_ERR_ARG, who ": null context");              \
    SLM_CUDA(cudaSetDevice(c->device));

extern "C" int slm_deflect_phase(slm_ctx* c, int H, int W, double konst, double sy, double sx, double* out) {
    SLM_EW_PROLOGUE("slm_deflect_phase");
    if (!out || H < 1 || W < 1) return fail(SLM_ERR_ARG, "slm_deflect_phase: bad argument");
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(deflect_kernel, dim3(ew_blocks((long long)H * W)), dim3(kEwThreads), 0, c->stream, out, H, W, konst, sy, sx); }
    SLM_CUDA(cudaGetLastError());
    return 0;
}
extern "C" int slm_lens_phase(slm_ctx* c, int H, int W, double px, double k, double f2, int trunc_u8, double* out) {
    SLM_EW_PROLOGUE("slm_lens_phase");
    if (!out || H < 1 || W < 1) return fail(SLM_ERR_ARG, "slm_lens_phase: bad argument");
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(lens_kernel, dim3(ew_blocks((long long)H * W)), dim3(kEwThreads), 0, c->stream, out, H, W, px, k, f2, trunc_u8); }
    SLM_CUDA(cudaGetLastError());
    return 0;
}
extern "C" int slm_add_mod2pi(slm_ctx* c, const double* a, const double* b, double* out, long long n, long long plane) {
    SLM_EW_PROLOGUE("slm_add_mod2pi");
    if (!a || !b || !out || n < 1 || plane < 1) return fail(SLM_ERR_ARG, "slm_add_mod2pi: bad argument");
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(add_mod2pi_kernel, dim3(ew_blocks(n)), dim3(kEwThreads), 0, c->stream, a, b, out, n, plane); }
    SLM_CUDA(cudaGetLastError());
    return 0;
}
extern "C" int slm_quantize(slm_ctx* c, const double* phase, const double* mask, double ct2pi, int mode, uint8_t* out,
                            long long n, long long plane) {
    SLM_EW_PROLOGUE("slm_quantize");
    if (!phase || !out || n < 1 || plane < 1) return fail(SLM_ERR_ARG, "slm_quantize: bad argument");
    if (mode != QUANT_Q1 && mode != QUANT_Q2 && mode != QUANT_Q3 && mode != QUANT_PREVIEW) return fail(SLM_ERR_ARG, "slm_quantize: unknown mode");
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(quantize_kernel, dim3(ew_blocks(n)), dim3(kEwThreads), 0, c->stream, phase, mask, ct2pi, mode, out, n, plane); }
    SLM_CUDA(cudaGetLastError());
    return 0;
}
extern "C" int slm_quantize_grey(slm_ctx* c, const uint8_t* grey, const double* mask, double ct2pi, uint8_t* out,
                                 long long n, long long plane) {
    SLM_EW_PROLOGUE("slm_quantize_grey");
    if (!grey || !mask || !out || n < 1 || plane < 1) return fail(SLM_ERR_ARG, "slm_quantize_grey: bad argument");
    { LaunchTimer t_(c, K_ELEMENTWISE); SLM_LAUNCH(quantize_grey_kernel, dim3(ew_blocks(n)), dim3(kEwThreads), 0, c->stream, grey, mask, ct2pi, out, n, plane); }
    SLM_CUDA(cudaGetLastError());
    return 0;
}
