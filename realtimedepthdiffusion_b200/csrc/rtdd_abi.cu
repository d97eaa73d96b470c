// Host side of librtdd.so: contexts, the HBM arena, the per-level sweep schedule
// (CUDA graphs), and the extern "C" entry points declared in include/rtdd.h.
//
// ref: src/GPUSolver.cu:33-71 (alloc/free), :264-272 (LUT), :274-316 (level driver),
//      src/main.cpp:95,153,232-295 (pyramid orchestration restated by rtdd_frame_*).

#include "rtdd_internal.h"

#include <math.h>
#include <cmath>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

int rtdd_fail(rtdd_ctx *ctx, int code, const char *where)
{
    if (ctx) {
        char buf[256];
        if (code > 0)
            snprintf(buf, sizeof buf, "%s: %s", where, cudaGetErrorString((cudaError_t)code));
        else
            snprintf(buf, sizeof buf, "%s: %s", where,
                     code == RTDD_E_ARG ? "bad argument" : code == RTDD_E_STATE ? "call-order violation"
                     : code == RTDD_E_NOMEM ? "host allocation failed" : code == RTDD_E_PEER ? "peer set-up failed" : "error");
        ctx->err = buf;
    }
    return code;
}

int rtdd_check(rtdd_ctx *ctx, cudaError_t e, const char *where)
{
    if (e == cudaSuccess) return 0;
    return rtdd_fail(ctx, (int)e, where);
}

#define RTDD_TRY(expr, where)                                   \
    do {                                                        \
        const int _rc = rtdd_check(ctx, (expr), (where));       \
        if (_rc) return _rc;                                    \
    } while (0)

namespace {

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ref: src/GPUSolver.cu:282-285,297-299 -- rho*rho in fp32, the quotient in fp64, stored to fp32.
void omega_schedule(int iterations, std::vector<float> &om)
{
    const int S = 10;
    const float rho = 0.99f;
    float omega = 0.0f;
    om.resize(iterations > 0 ? iterations : 0);
    for (int it = 0; it < iterations; it++) {
        if (it < S) omega = 1.0f;
        else if (it == S) { const float r2 = rho * rho; omega = (float)(2.0 / (2.0 - (double)r2)); }
        else { const float r2 = rho * rho; const float r2w = r2 * omega; omega = (float)(4.0 / (4.0 - (double)r2w)); }
        om[it] = omega;
    }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

bool encode_plane_map(EncodeTiledFn fn, CUtensorMap *map, void *base, bool f32, int widthElems, int rows, int boxW, int boxH)
{
    const cuuint64_t dims[2] = {(cuuint64_t)widthElems, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)widthElems * (f32 ? 4u : 1u)};
    const cuuint32_t box[2] = {(cuuint32_t)boxW, (cuuint32_t)boxH};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

void build_tensor_maps(rtdd_ctx *ctx)
{
    void *fnp = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fnp, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !fnp) {
        cudaGetLastError();
        return;                          // levels keep hasMaps = false: the LDG form of the blocked kernel is used
    }
    EncodeTiledFn fn = (EncodeTiledFn)fnp;
    for (auto &L : ctx->lv) {
        bool ok = true;
        for (int k = 0; k < 4 && ok; k++) ok = encode_plane_map(fn, &L.tmX[k], L.x[k], true, L.pitchF, L.planeRows, 128, 64);
        // byte boxes are 144 wide: see TmaSmem::WB in solver_kernels.cu
        ok = ok && encode_plane_map(fn, &L.tmLinkR, L.linkR, false, L.pitchB, L.planeRows, 144, 64);
        ok = ok && encode_plane_map(fn, &L.tmLinkD, L.linkD, false, L.pitchB, L.planeRows, 144, 64);
        ok = ok && encode_plane_map(fn, &L.tmMask, L.mask, false, L.pitchB, L.planeRows, 144, 64);
        ok = ok && encode_plane_map(fn, &L.tmLinkD1, L.linkD, false, L.pitchB, L.planeRows, 144, 65);
        L.hasMaps = ok;
    }
}

void destroy_graphs(rtdd_ctx *ctx)
{
    for (auto &kv : ctx->graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    ctx->graphs.clear();
}

static int g_zeroCopyOut = 1;           // see host_plane_alias
static int g_passPlanner = 1;           // 1: passes of their own lengths (rtdd::blocked_plan_passes); 0: one length per level (round-2a behaviour)

// Sweep-variant policy (all variants are bit-identical; this only decides speed).
void pick_variant(const rtdd_ctx *ctx, const RtddLevel &L, int iters, int *variant, int *T, int *form = nullptr)
{
    if (form) *form = 0;
    int v = ctx->variant, t = ctx->sweepsPerPass;
    int rR, rC, rB, rW;
    const bool fits = rtdd::resident_plan(L.rows, L.cols, &rR, &rC, &rB, &rW);
    if (v == 3 && !fits) v = 2;          // level too large for one cluster: temporally blocked instead
    // measured (tools/coarse_level_cases.py): 240x135 resident 0.23 ms vs blocked 0.36; 256x256 resident 0.30..0.33 (32 warps per
    // CTA, the 64-register build; two rows per warp no better) vs blocked 0.23..0.26 -- the crossover lies in between
    const bool residentPays = fits && (long)L.rows * L.cols <= 49152;
    if (v == 0) v = (residentPays && iters >= 8) ? 3 : 2;
    if (v == 3) {
        t = 0;
    } else if (v == 2) {
        if (t <= 0) {
            // 128x64-tile levels (>= 2^18 pixels): sweeps per pass and form from the cost model fitted to tools/tune_levels.py;
            // smaller levels: 11 (128x32 tiles, measured in round 1)
            // (a context planned for throughput also takes 128x64 tiles below 2^18 pixels: the flat 128x32 tiles keep 104 x 10 of their
            // 128 x 32 pixels at 11 sweeps per pass -- fine while the GPU is not full anyway, four times the SM time when it is)
            const long px = (long)L.rows * L.cols;
            if (px >= (1L << 18) || ctx->planThroughput) {
                int f = 0;
                rtdd::blocked_plan(L.rows, L.cols, iters, ctx->smCount, &t, &f);
                if (form) *form = f;
            } else {
                t = 11;
                if (form) *form = 2;         // 128x32 tiles; the pass planner may still move the level to another form
            }
        }
        if (t > RTDD_MAX_T) t = RTDD_MAX_T;
        if (t > iters) t = iters > 0 ? iters : 1;
    } else {
        t = 1;
    }
    *variant = v;
    *T = t;
}

int ensure_omega_table(rtdd_ctx *ctx, int iters)
{
    if (iters <= ctx->dOmegaCap) return 0;
    // the schedule is prefix-stable: keep one device copy long enough for the longest level seen
    const int cap = iters > 4096 ? iters : 4096;
    std::vector<float> all;
    omega_schedule(cap, all);
    float *d = nullptr;
    RTDD_TRY(cudaMalloc((void **)&d, (size_t)cap * sizeof(float)), "omega table");
    RTDD_TRY(cudaMemcpy(d, all.data(), (size_t)cap * sizeof(float), cudaMemcpyHostToDevice), "omega table");
    if (ctx->dOmega) {
        RTDD_TRY(cudaDeviceSynchronize(), "omega table");
        destroy_graphs(ctx);         // graphs captured with the old table
        cudaFree(ctx->dOmega);
    }
    ctx->dOmega = d;
    ctx->dOmegaCap = cap;
    return 0;
}

bool target_ok(const float *depth, size_t depthPitch)
{
    return (((uintptr_t)depth | depthPitch) & 15u) == 0;
}

// Enqueue `iters` sweeps of `level` on stream `s`, starting from plane x[0] (prev = implicit zeros).  The last
// pass writes to *target when given (caller's depth plane / u8 map); otherwise *resultPlane tells where x_K is.
int enqueue_sweeps(rtdd_ctx *ctx, cudaStream_t s, int level, int iters, const rtdd::SweepTarget *target, int *kernels, int *resultPlane)
{
    const RtddLevel &L = ctx->lv[level];
    int variant, T, form;
    pick_variant(ctx, L, iters, &variant, &T, &form);
    std::vector<float> om;
    omega_schedule(iters, om);
    const float gamma = 0.99f;
    cudaError_t e = cudaSuccess;
    int n = 0, result = 0;
    if (variant == 3) {
        e = rtdd::launch_sweep_resident(s, L, ctx->dLut, L.x[0], L.x[2], ctx->dOmega, iters, gamma, target);
        n = 1;
        result = 2;
    } else if (variant == 1) {
        // three-plane rotation: x_k in plane k%3, x_{k+1} -> (k+1)%3, x_{k-1} in (k+2)%3
        for (int k = 0; k < iters && e == cudaSuccess; k++) {
            e = rtdd::launch_sweep_single(s, L, ctx->dLut, L.x[k % 3], L.x[(k + 2) % 3], L.x[(k + 1) % 3], om[k], gamma, k == 0,
                                          (k == iters - 1) ? target : nullptr);
            n++;
        }
        result = iters % 3;
    } else {
        // pair A = planes (0,1), pair B = planes (2,3); each pass reads one pair and writes the other
        // Passes: the caller's own list (rtdd_set_pass_plan), else -- 128x64-tile levels without a forced sweeps-per-pass -- the
        // planner's (every pass with the halo of its own length), else `T` sweeps per pass with the halo of T throughout.
        std::vector<int> plan;
        bool ownHalo = false;
        const std::vector<int> &forced = ctx->passPlan[level];
        int forcedSum = 0;
        for (int m : forced) forcedSum += m;
        if (!forced.empty() && forcedSum == iters) {
            plan = forced;
            ownHalo = true;
        } else if (g_passPlanner && ctx->sweepsPerPass <= 0 && form != 0) {
            plan.resize(iters);
            int f2 = form;
            const int np = rtdd::blocked_plan_passes(L.rows, L.cols, iters, ctx->smCount, (target && target->u8b) ? 1 : 0, ctx->planThroughput ? 1 : 0, plan.data(), iters, &f2);
            if (np > 0) { plan.resize(np); form = f2; ownHalo = true; } else plan.clear();
        }
        if (plan.empty())
            for (int k = 0; k < iters; k += T) plan.push_back(iters - k < T ? iters - k : T);
        int cur = 0, k = 0;
        for (size_t i = 0; i < plan.size() && e == cudaSuccess; i++) {
            const int m = plan[i];
            rtdd::OmegaPack pack;
            for (int j = 0; j < RTDD_MAX_T; j++) pack.w[j] = (j < m) ? om[k + j] : 0.0f;
            const int src = cur, dst = cur ^ 2;
            e = rtdd::launch_sweep_blocked(s, L, ctx->dLut, L.x[src], L.x[src + 1], L.x[dst], L.x[dst + 1], pack, ownHalo ? m : T, m, gamma,
                                           k == 0, ctx->smCount, (k + m >= iters) ? target : nullptr, nullptr, form);
            n++;
            cur = dst;
            k += m;
        }
        result = cur;
    }
    *kernels = n;
    *resultPlane = result;
    return rtdd_check(ctx, e, "sweep launch");
}

struct LevelArgs {
    int level, iters;
    float *depth; size_t depthPitch;
    const uint8_t *scribble; size_t scribblePitch;
    const uint8_t *gray; size_t grayPitch;
    uint8_t *u8; size_t u8Pitch;          // optional quantised output (whole-frame path, level 0)
    // whole-frame path, levels below the coarsest: the guess is the prolongation of `coarse` with the level's Dirichlet
    // values re-injected from `edited`; it is produced inside the level set-up instead of being read from `depth`
    const float *coarse; size_t coarsePitch; int coarseRows, coarseCols;
    const uint8_t *edited; size_t editedPitch;
    bool resetBad;                        // clear the level's out-of-range flag first (the whole-frame graph clears all levels' flags at its start)
    uint8_t *u8b = nullptr; size_t u8bPitch = 0;   // optional second 8-bit map: device alias of the caller's pinned host plane
};

// Opt-in (rtdd_set_tuning("fused_prolong", 1)): bit-identical and tested, but measured no faster than the three separate
// kernels inside the frame graph (4K 1.9025 vs 1.8945 ms, 8K UHD 3.081 vs 3.065 ms, 1080p 1.306 vs 1.307 ms): with
// programmatic dependent launch the small kernels already overlap, and the 66 MB saved at 4K are ~1 % of a frame.  Re-measured with
// the final round-2 kernels: 1.751 against 1.740 ms.
static int g_fusedProlong = 0;

// One level on stream `s`: edge-weight pass, sweeps, result into the caller's depth plane.  `capturing` selects
// the event-record flavour that is legal inside a stream capture.
int enqueue_level(rtdd_ctx *ctx, cudaStream_t s, const LevelArgs &a, bool capturing, int *kernels)
{
    RtddLevel &L = ctx->lv[a.level];
    const bool coarsest = (a.level == ctx->levels - 1);
    const int threshold = (a.level == 0) ? 0 : 4;          // ref: src/GPUSolver.cu:201-202
    int n = 0;
    unsigned int *resetResidual = (a.iters > 0) ? L.dResidual : nullptr;     // the set-up kernel zeroes the level's residual word
    if (a.resetBad) RTDD_TRY(cudaMemsetAsync(L.dBad, 0, sizeof(unsigned int), s), "level flags");
    if (a.coarse) {
        // ref: src/main.cpp:272-281 + src/GPUSolver.cu:290-293 in one pass; the guess itself is never stored as a pitched plane
        RTDD_TRY(rtdd::launch_level_prolong_init(s, L, a.coarse, a.coarsePitch, a.coarseRows, a.coarseCols, a.edited, a.editedPitch,
                                                 a.scribble, a.scribblePitch, a.gray, a.grayPitch, threshold, L.x[0], resetResidual), "level prolong+init");
    } else {
        RTDD_TRY(rtdd::launch_level_init(s, L, a.depth, a.depthPitch, a.scribble, a.scribblePitch, a.gray, a.grayPitch, coarsest, threshold, L.x[0],
                                         resetResidual), "level init");
    }
    n++;
    int plane = 0;
    bool direct = false;
    if (a.iters > 0) {
        direct = target_ok(a.depth, a.depthPitch);
        rtdd::SweepTarget tgt = {direct ? a.depth : nullptr, (int)(a.depthPitch / sizeof(float)), direct ? a.u8 : nullptr, (int)a.u8Pitch, L.dResidual,
                                 (direct && a.u8) ? a.u8b : nullptr, (int)a.u8bPitch};
        const unsigned int flags = capturing ? cudaEventRecordExternal : cudaEventRecordDefault;
        RTDD_TRY(cudaEventRecordWithFlags(L.evBegin, s, flags), "level event");
        int k = 0;
        int rc = enqueue_sweeps(ctx, s, a.level, a.iters, &tgt, &k, &plane);
        if (rc) return rc;
        RTDD_TRY(cudaEventRecordWithFlags(L.evEnd, s, flags), "level event");
        L.timed = true; L.lastIters = a.iters; L.lastKernels = k;
        ctx->captureTiming.push_back({a.level, a.iters, k});
        n += k;
    }
    if (!direct) {
        RTDD_TRY(rtdd::launch_copy_out(s, L, L.x[plane], a.depth, a.depthPitch), "copy out");
        n++;
        if (a.u8) {
            RTDD_TRY(rtdd::launch_quantise(s, a.depth, a.depthPitch, a.u8, a.u8Pitch, L.rows, L.cols), "quantise");
            n++;
        }
    }
    *kernels = n;
    return 0;
}

// Capture `body` into a graph (or fetch it from the cache) and launch it on the context stream.
template <class Body>
int run_cached_graph(rtdd_ctx *ctx, const RtddGraphKey &key, Body body)
{
    auto it = ctx->graphs.find(key);
    if (it == ctx->graphs.end()) {
        if (ctx->graphs.size() >= 64) {                      // callers that keep changing planes: start over
            RTDD_TRY(cudaStreamSynchronize(ctx->stream), "graph cache");
            destroy_graphs(ctx);
        }
        cudaStream_t cs = ctx->captureStream;
        RTDD_TRY(cudaStreamBeginCapture(cs, cudaStreamCaptureModeRelaxed), "cudaStreamBeginCapture");
        int kernels = 0;
        ctx->captureTiming.clear();
        const int rc = body(cs, &kernels);
        cudaGraph_t graph = nullptr;
        const cudaError_t e2 = cudaStreamEndCapture(cs, &graph);
        if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
        RTDD_TRY(e2, "cudaStreamEndCapture");
        RtddGraph g;
        const cudaError_t e = cudaGraphInstantiate(&g.exec, graph, 0);
        cudaGraphDestroy(graph);
        RTDD_TRY(e, "cudaGraphInstantiate");
        g.kernels = kernels;
        g.timing = ctx->captureTiming;
        it = ctx->graphs.emplace(key, g).first;
    }
    RTDD_TRY(cudaGraphLaunch(it->second.exec, ctx->stream), "cudaGraphLaunch");
    // the level events now bracket THIS graph's sweeps: rtdd_level_sweep_ms must pair them with this graph's counts
    for (const RtddLevelTiming &t : it->second.timing) {
        RtddLevel &L = ctx->lv[t.level];
        L.timed = true; L.lastIters = t.iters; L.lastKernels = t.kernels;
    }
    ctx->launches += it->second.kernels;
    return 0;
}

int level_dims_ok(const rtdd_ctx *ctx, int level, int rows, int cols)
{
    if (level < 0 || level >= ctx->levels) return 0;
    const RtddLevel &L = ctx->lv[level];
    return rows >= 1 && cols >= 1 && rows <= L.rows && cols <= L.cols;
}

}  // namespace

extern "C" {

int rtdd_pyramid_levels(int rows, int cols)
{
    // ref: src/main.cpp:95 -- int pyrLevels = log2(std::max(std::min(cols, rows) / 45, 1)) + 1;
    int m = (cols < rows ? cols : rows) / 45;
    if (m < 1) m = 1;
    return (int)log2((double)m) + 1;
}

int rtdd_level_iterations(int maxIterations, int levels, int level)
{
    // ref: src/main.cpp:263 -- int CUDAIteration = maxIterations / powf(2.0, (pyrLevels - 1) - level);
    return (int)((float)maxIterations / powf(2.0f, (float)((levels - 1) - level)));
}

// ---- row-strip planning (host only; no reference counterpart: the reference is single-GPU) -----------------------
// Which levels are cut into row strips and who owns which rows.  The coarsest level still worth splitting (at least
// minStripPixels pixels, every strip at least max(halo, 2) rows) is cut evenly; every finer level doubles those
// boundaries, so a rank's fine rows are exactly the prolongation of its own coarse rows.  Levels coarser than that are
// replicated (solved by every rank).
int rtdd_plan_strips(const int *levelRows, const int *levelCols, int levels, int nranks, int halo, long long minStripPixels,
                     int *split, int *ownBegin, int *ownEnd)
{
    if (!levelRows || !levelCols || !split || !ownBegin || !ownEnd || levels < 1 || nranks < 1 || halo < 1) return RTDD_E_ARG;
    for (int l = 0; l < levels; l++) split[l] = 0;
    if (nranks <= 1) return 0;
    int cs = -1;
    const int minRows = halo > 2 ? halo : 2;
    for (int l = 0; l < levels; l++) {
        if ((long long)levelRows[l] * levelCols[l] >= minStripPixels && levelRows[l] / nranks >= minRows) cs = l;
        else break;
    }
    if (cs < 0) return 0;
    std::vector<long long> bounds(nranks + 1);
    for (int r = 0; r < nranks; r++) bounds[r] = ((long long)r * levelRows[cs]) / nranks;
    for (int l = cs; l >= 0; l--) {
        if (l < cs)
            for (int r = 0; r < nranks; r++) bounds[r] *= 2;
        bounds[nranks] = levelRows[l];
        split[l] = 1;
        for (int r = 0; r < nranks; r++) {
            ownBegin[l * nranks + r] = (int)bounds[r];
            ownEnd[l * nranks + r] = (int)bounds[r + 1];
            if (bounds[r + 1] - bounds[r] < halo) return RTDD_E_ARG;          // a strip shorter than its halo
        }
    }
    return 0;
}

// The passes of one split level: `iters` sweeps in passes of at most passSweeps (<= halo) sweeps, with a halo exchange
// whenever `halo` sweeps have gone by since the ghost rows were last fresh, and after the last pass if the level feeds a
// prolongation (level > 0).  Fills sweepsOfPass[i] and exchangeAfter[i]; returns the number of passes (or a negative
// RTDD_E_* when `capacity` is too small).
int rtdd_strip_schedule(int iters, int halo, int passSweeps, int level, int *sweepsOfPass, int *exchangeAfter, int capacity)
{
    if (iters < 0 || halo < 1 || level < 0 || !sweepsOfPass || !exchangeAfter || capacity < 0) return RTDD_E_ARG;
    int T = passSweeps;
    if (T < 1 || T > halo) T = halo;
    int k = 0, since = 0, n = 0;
    while (k < iters) {
        int m = T;
        if (iters - k < m) m = iters - k;
        if (halo - since < m) m = halo - since;
        if (n >= capacity) return RTDD_E_ARG;
        k += m;
        since += m;
        const bool exchange = (since >= halo || k >= iters) && (k < iters || level > 0);
        sweepsOfPass[n] = m;
        exchangeAfter[n] = exchange ? 1 : 0;
        if (exchange) since = 0;
        n++;
    }
    return n;
}

static int create_impl(int rows, int cols, int levels, int device, const int *planeRows, rtdd_ctx **out);

int rtdd_create(int rows, int cols, int levels, int device, rtdd_ctx **out)
{
    return create_impl(rows, cols, levels, device, nullptr, out);
}

// host only: the pass plan of one level solved with the temporally blocked kernels (see rtdd::blocked_plan)
int rtdd_plan_blocked(int rows, int cols, int iterations, int smCount, int *sweepsPerPass, int *clusterForm)
{
    if (rows < 1 || cols < 1 || iterations < 0 || smCount < 1 || !sweepsPerPass || !clusterForm) return RTDD_E_ARG;
    int T = 0, form = 0;
    rtdd::blocked_plan(rows, cols, iterations > 0 ? iterations : 1, smCount, &T, &form);
    *sweepsPerPass = T;
    *clusterForm = (form == 3) ? 1 : 0;
    return 0;
}

// host only: the passes of one level, each with the halo of its own length (see rtdd::blocked_plan_passes).  flags: 1 = the last
// pass also stores the 8-bit map into pinned host memory and is made as long as the tiling allows; 2 = plan for throughput (a
// context of a batch): total SM time instead of the level's latency
int rtdd_plan_passes(int rows, int cols, int iterations, int smCount, int flags, int *sweepsOfPass, int capacity, int *clusterForm)
{
    if (rows < 1 || cols < 1 || iterations < 1 || smCount < 1 || flags < 0 || flags > 3 || !sweepsOfPass || capacity < 1 || !clusterForm) return RTDD_E_ARG;
    int form = 0;
    const int n = rtdd::blocked_plan_passes(rows, cols, iterations, smCount, flags & 1, (flags >> 1) & 1, sweepsOfPass, capacity, &form);
    if (n <= 0) return RTDD_E_ARG;
    *clusterForm = (form == 3) ? 1 : (form == 2) ? 2 : 0;
    return n;
}

// The caller's own passes for one level of the temporally blocked kernels (tuning, tests): npasses lengths of 1..16 sweeps; a level
// solved with a different total falls back to the planner.  npasses = 0 removes the list.
int rtdd_set_pass_plan(rtdd_ctx *ctx, int level, const int *sweepsOfPass, int npasses)
{
    if (!ctx || level < 0 || level >= ctx->levels || level >= 32 || npasses < 0 || (npasses > 0 && !sweepsOfPass)) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_set_pass_plan");
    for (int i = 0; i < npasses; i++)
        if (sweepsOfPass[i] < 1 || sweepsOfPass[i] > RTDD_MAX_T) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_set_pass_plan");
    DeviceGuard guard(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    destroy_graphs(ctx);
    ctx->passPlan[level].assign(sweepsOfPass, sweepsOfPass + npasses);
    return 0;
}

// host only: rows the scratch planes of every level must hold on EVERY rank of a row-strip frame (largest window of the split levels)
int rtdd_plan_strip_planes(const int *levelRows, const int *levelCols, int levels, int nranks, int halo, long long minStripPixels, int *planeRows)
{
    if (!levelRows || !levelCols || !planeRows || levels < 1 || nranks < 1 || halo < 1 || minStripPixels < 1) return RTDD_E_ARG;
    std::vector<int> split(levels), ob((size_t)levels * nranks), oe((size_t)levels * nranks);
    const int rc = rtdd_plan_strips(levelRows, levelCols, levels, nranks, halo, minStripPixels, split.data(), ob.data(), oe.data());
    if (rc) return rc;
    for (int l = 0; l < levels; l++) {
        planeRows[l] = levelRows[l];
        if (nranks > 1 && split[l]) {
            int mx = 0;
            for (int r = 0; r < nranks; r++) {
                const int w0 = ob[l * nranks + r] - halo > 0 ? ob[l * nranks + r] - halo : 0;
                const int w1 = oe[l * nranks + r] + halo < levelRows[l] ? oe[l * nranks + r] + halo : levelRows[l];
                if (w1 - w0 > mx) mx = w1 - w0;
            }
            planeRows[l] = mx;
        }
    }
    return 0;
}

// A context for ONE rank of a row-strip frame: the planes of the levels that rtdd_plan_strips splits hold only the largest row
// window any rank keeps (own rows + ghost rows), not the whole level -- 0.9 GB instead of 6.8 GB per rank for a 16384^2 image on
// 8 GPUs.  All ranks get the same layout (peers address each other's planes by offset).  Whole-level calls on a split level
// (rtdd_solve_level ...) return RTDD_E_STATE; follow with rtdd_strip_frame_setup using the same rank / halo / minStripPixels.
int rtdd_create_strip(int rows, int cols, int levels, int device, int nranks, int halo, long long minStripPixels, rtdd_ctx **out)
{
    if (!out) return RTDD_E_ARG;
    *out = nullptr;
    if (rows < 1 || cols < 1 || levels < 1 || levels > 30 || nranks < 1 || halo < 1 || minStripPixels < 1) return RTDD_E_ARG;
    std::vector<int> lr(levels), lc(levels), plane(levels);
    for (int l = 0; l < levels; l++) {
        lr[l] = (int)((float)rows / powf(2.0f, (float)l)); lc[l] = (int)((float)cols / powf(2.0f, (float)l));
        if (lr[l] < 1) lr[l] = 1;
        if (lc[l] < 1) lc[l] = 1;
    }
    const int rc = rtdd_plan_strip_planes(lr.data(), lc.data(), levels, nranks, halo, minStripPixels, plane.data());
    if (rc) return rc;
    return create_impl(rows, cols, levels, device, plane.data(), out);
}

static int create_impl(int rows, int cols, int levels, int device, const int *planeRows, rtdd_ctx **out)
{
    if (!out) return RTDD_E_ARG;
    *out = nullptr;
    if (rows < 1 || cols < 1 || levels < 1 || levels > 30) return RTDD_E_ARG;
    rtdd_ctx *ctx = new (std::nothrow) rtdd_ctx();
    if (!ctx) return RTDD_E_NOMEM;
    cudaError_t e;
    if (device < 0) { e = cudaGetDevice(&device); if (e != cudaSuccess) { delete ctx; return (int)e; } }
    ctx->device = device;
    ctx->rows = rows; ctx->cols = cols; ctx->levels = levels;
    DeviceGuard guard(device);
    int sm = 0;
    e = cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) { delete ctx; return (int)e; }
    ctx->smCount = sm > 0 ? sm : 148;
    e = cudaStreamCreateWithFlags(&ctx->ownStream, cudaStreamDefault);
    if (e != cudaSuccess) { delete ctx; return (int)e; }
    ctx->stream = ctx->ownStream;
    e = cudaStreamCreateWithFlags(&ctx->captureStream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { cudaStreamDestroy(ctx->ownStream); delete ctx; return (int)e; }

    // one arena: per level 4 float planes + 3 byte planes, each with a guard row above and below
    ctx->lv.resize(levels);
    size_t total = 257 * sizeof(float) + 256 + 256 + 2048;   // LUT + one residual word per level (<= 30 levels) + strip tickets/flags
    for (int l = 0; l < levels; l++) {
        RtddLevel &L = ctx->lv[l];
        // ref: src/GPUSolver.cu:42-43 -- int rowsPerLevel = rows / powf(2, level)
        L.rows = (int)((float)rows / powf(2.0f, (float)l));
        L.cols = (int)((float)cols / powf(2.0f, (float)l));
        if (L.rows < 1 || L.cols < 1) { L.rows = L.rows < 1 ? 1 : L.rows; L.cols = L.cols < 1 ? 1 : L.cols; }
        L.planeRows = planeRows ? planeRows[l] : L.rows;
        L.pitchF = (int)rtdd_round_up((size_t)L.cols + 4, 64);
        L.pitchB = (int)rtdd_round_up((size_t)L.cols + 4, 128);
        total += 4 * rtdd_round_up((size_t)L.pitchF * L.planeRows * sizeof(float), 256);
        total += 3 * rtdd_round_up((size_t)L.pitchB * L.planeRows, 256);
        total += rtdd_round_up((size_t)8 * RTDD_MAX_HALO * L.pitchF * sizeof(float), 256);     // staged peer exchange (rtdd_strip_push)
    }
    e = cudaMalloc(&ctx->arena, total);
    if (e != cudaSuccess) { cudaStreamDestroy(ctx->captureStream); cudaStreamDestroy(ctx->ownStream); delete ctx; return (int)e; }
    ctx->arenaBytes = total;
    cudaMemsetAsync(ctx->arena, 0, total, ctx->stream);
    char *p = (char *)ctx->arena;
    ctx->dLut = (float *)p;
    p += rtdd_round_up(257 * sizeof(float), 256);
    unsigned int *resWords = (unsigned int *)p;
    ctx->dErrWord = resWords + 63;                     // <= 30 levels use words 0..29
    ctx->dPeerBadWord = resWords + 62;
    p += 256;
    unsigned int *stripWords = (unsigned int *)p;      // 16 words per level (same offset in every rank's arena)
    p += 2048;
    for (int l = 0; l < levels; l++) {
        RtddLevel &L = ctx->lv[l];
        L.dResidual = resWords + l;
        L.dBad = resWords + 32 + l;
        L.dStripWords = stripWords + 16 * l;
        for (int k = 0; k < 4; k++) { L.x[k] = (float *)p; p += rtdd_round_up((size_t)L.pitchF * L.planeRows * sizeof(float), 256); }
        L.linkR = (uint8_t *)p; p += rtdd_round_up((size_t)L.pitchB * L.planeRows, 256);
        L.linkD = (uint8_t *)p; p += rtdd_round_up((size_t)L.pitchB * L.planeRows, 256);
        L.mask = (uint8_t *)p;  p += rtdd_round_up((size_t)L.pitchB * L.planeRows, 256);
        L.stage = (float *)p;   p += rtdd_round_up((size_t)8 * RTDD_MAX_HALO * L.pitchF * sizeof(float), 256);
    }
    build_tensor_maps(ctx);
    e = rtdd::configure_kernels();
    if (e == cudaSuccess) e = rtdd::configure_stereo();
    for (int l = 0; l < levels && e == cudaSuccess; l++) {
        e = cudaEventCreate(&ctx->lv[l].evBegin);
        if (e == cudaSuccess) e = cudaEventCreate(&ctx->lv[l].evEnd);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { rtdd_destroy(ctx); return (int)e; }
    *out = ctx;
    return 0;
}

int rtdd_destroy(rtdd_ctx *ctx)
{
    if (!ctx) return RTDD_E_ARG;
    DeviceGuard guard(ctx->device);
    cudaError_t e = cudaDeviceSynchronize();
    destroy_graphs(ctx);
    for (auto &L : ctx->lv) {
        if (L.evBegin) cudaEventDestroy(L.evBegin);
        if (L.evEnd) cudaEventDestroy(L.evEnd);
    }
    for (void *p : ctx->ipcImports) cudaIpcCloseMemHandle(p);
    if (ctx->dOmega) cudaFree(ctx->dOmega);
    if (ctx->arena) cudaFree(ctx->arena);
    if (ctx->frameArena) cudaFree(ctx->frameArena);
    if (ctx->satScratch) cudaFree(ctx->satScratch);
    if (ctx->bandArena) cudaFree(ctx->bandArena);
    if (ctx->captureStream) cudaStreamDestroy(ctx->captureStream);
    if (ctx->ownStream) cudaStreamDestroy(ctx->ownStream);
    delete ctx;
    return (int)e;
}

int rtdd_load_weights(rtdd_ctx *ctx, float beta)
{
    if (!ctx) return RTDD_E_ARG;
    // Deviation: the reference accepts any beta.  A negative one gives weights above 1 (sums above 8, outside the range the
    // sweeps' branch-free division is proven for, which the cluster kernel does not check), a non-finite one NaN weights;
    // neither has an edge-stopping meaning.  Refused before the table is touched, so the previous one stays in force.
    if (!(beta >= 0.0f) || !std::isfinite(beta)) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_load_weights (beta must be finite and >= 0)");
    DeviceGuard guard(ctx->device);
    // ref: src/GPUSolver.cu:266-268 -- host expf, fp32
    for (int w = 0; w < 256; w++) ctx->hLut[w] = expf(-beta * w);
    ctx->hLut[256] = 0.0f;
    RTDD_TRY(cudaMemcpyAsync(ctx->dLut, ctx->hLut, 257 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream), "rtdd_load_weights");
    RTDD_TRY(cudaStreamSynchronize(ctx->stream), "rtdd_load_weights");
    ctx->lutLoaded = true;
    return 0;
}

int rtdd_set_stream(rtdd_ctx *ctx, void *stream)
{
    if (!ctx) return RTDD_E_ARG;
    ctx->stream = stream ? (cudaStream_t)stream : ctx->ownStream;
    return 0;
}

int rtdd_sync(rtdd_ctx *ctx)
{
    if (!ctx) return RTDD_E_ARG;
    DeviceGuard guard(ctx->device);
    RTDD_TRY(cudaStreamSynchronize(ctx->stream), "rtdd_sync");
    RTDD_TRY(cudaGetLastError(), "rtdd_sync");
    if (ctx->peerUp || ctx->peerDn) {
        // strip mode: a halo wait that gave up (spin_timeout_ms) left a mark instead of killing the context
        unsigned int w = 0;
        RTDD_TRY(cudaMemcpy(&w, ctx->dErrWord, sizeof(w), cudaMemcpyDeviceToHost), "rtdd_sync");
        if (w == RTDD_SPIN_TIMED_OUT) {
            cudaMemset(ctx->dErrWord, 0, sizeof(w));
            return rtdd_fail(ctx, RTDD_E_PEER, "rtdd_sync (a halo wait on a neighbouring rank timed out; ghost rows are stale)");
        }
    }
    return 0;
}

const char *rtdd_last_error(const rtdd_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
unsigned long long rtdd_launch_count(const rtdd_ctx *ctx) { return ctx ? ctx->launches : 0ULL; }
int rtdd_levels(const rtdd_ctx *ctx) { return ctx ? ctx->levels : 0; }

int rtdd_set_tuning(rtdd_ctx *ctx, const char *key, int value)
{
    if (!ctx || !key) return RTDD_E_ARG;
    if (strcmp(key, "blocked_tile") == 0 && (value == 0 || value == 32 || value == 34 || value == 64)) {
        rtdd::set_blocked_tile_override(value);
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "resident_warps") == 0 && value >= 1 && value <= 32) {
        rtdd::set_resident_warps(value);
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "resident_r1_max_warps") == 0 && value >= 1 && value <= 32) {
        rtdd::set_resident_r1_max_warps(value);
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "fused_prolong") == 0 && (value == 0 || value == 1)) {
        g_fusedProlong = value;
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "pass_planner") == 0 && (value == 0 || value == 1)) {
        g_passPlanner = value;
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "plan_throughput") == 0 && (value == 0 || value == 1)) {
        ctx->planThroughput = (value != 0);          // this context only
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "zero_copy_out") == 0 && (value == 0 || value == 1)) {
        g_zeroCopyOut = value;          // graphs are keyed by the host alias: nothing to rebuild
        return 0;
    }
    if (strcmp(key, "strip_residual") == 0 && (value == 0 || value == 1)) {
        ctx->stripResidual = (value != 0);
        return 0;
    }
    if (strcmp(key, "spin_timeout_ms") == 0 && value >= 0) {
        ctx->spinTimeoutMs = (unsigned int)value;
        return 0;
    }
    if (strcmp(key, "strip_peer_staging") == 0 && (value == 0 || value == 1)) {
        ctx->peerStaging = (value != 0);
        return 0;
    }
    if (strcmp(key, "pdl") == 0 && (value == 0 || value == 1)) {
        rtdd::set_pdl(value);
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "blocked_grid_cap") == 0 && value >= 0) {
        rtdd::set_blocked_grid_cap(value);
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "blocked_cluster") == 0 && (value == 1 || value == 2 || value == 4 || value == 8)) {
        rtdd::set_blocked_cluster(value);
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    if (strcmp(key, "blocked_tma") == 0 && value >= 0 && value <= 3) {
        rtdd::set_blocked_tma(value);
        DeviceGuard guard(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        destroy_graphs(ctx);
        return 0;
    }
    return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_set_tuning");
}

int rtdd_set_sweep_variant(rtdd_ctx *ctx, int variant, int sweepsPerPass)
{
    if (!ctx || variant < 0 || variant > 3 || sweepsPerPass < 0 || sweepsPerPass > RTDD_MAX_T) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_set_sweep_variant");
    ctx->variant = variant;
    ctx->sweepsPerPass = sweepsPerPass;
    return 0;
}

// ---- the solve ---------------------------------------------------------------

static int edge_pass(rtdd_ctx *ctx, const float *depth, size_t depthPitch, const uint8_t *scribble, size_t scribblePitch,
                     const uint8_t *gray, size_t grayPitch, int rows, int cols, int level, const char *where)
{
    if (!ctx) return RTDD_E_ARG;
    if (!depth || !gray || !level_dims_ok(ctx, level, rows, cols)) return rtdd_fail(ctx, RTDD_E_ARG, where);
    RtddLevel &L = ctx->lv[level];
    if (rows != L.rows || cols != L.cols) return rtdd_fail(ctx, RTDD_E_ARG, where);   // planes are sized per level (ref :42-48)
    if (L.planeRows < L.rows) return rtdd_fail(ctx, RTDD_E_STATE, where);             // a strip context holds only a window of this level
    // ref: src/GPUSolver.cu:201-202 -- threshold 4, 0 at level 0; :196 -- ungated on the coarsest level
    const bool coarsest = (level == ctx->levels - 1);
    const int threshold = (level == 0) ? 0 : 4;
    RTDD_TRY(cudaMemsetAsync(L.dBad, 0, sizeof(unsigned int), ctx->stream), where);
    RTDD_TRY(rtdd::launch_level_init(ctx->stream, L, depth, depthPitch, scribble, scribblePitch, gray, grayPitch, coarsest, threshold, L.x[0]), where);
    ctx->launches++;
    return 0;
}

int rtdd_solve_level(rtdd_ctx *ctx, float *depth, size_t depthPitch, const uint8_t *scribble, size_t scribblePitch,
                     const uint8_t *gray, size_t grayPitch, int rows, int cols, int maxIterations, int level)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->lutLoaded) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_solve_level (rtdd_load_weights not called)");
    if (!depth || !gray || !scribble || maxIterations < 0 || !level_dims_ok(ctx, level, rows, cols))
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_solve_level");
    RtddLevel &L = ctx->lv[level];
    if (rows != L.rows || cols != L.cols) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_solve_level");   // planes are sized per level (ref :42-48)
    if (L.planeRows < L.rows) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_solve_level (a strip context holds only a window of this level)");
    DeviceGuard guard(ctx->device);
    int rc = ensure_omega_table(ctx, maxIterations);
    if (rc) return rc;
    int variant, T;
    pick_variant(ctx, L, maxIterations, &variant, &T);
    RtddGraphKey key{};
    key.kind = 1; key.level = level; key.iters = maxIterations; key.variant = variant; key.T = T;
    key.p[0] = depth; key.p[1] = scribble; key.p[2] = gray;
    key.pitch[0] = depthPitch; key.pitch[1] = scribblePitch; key.pitch[2] = grayPitch;
    const LevelArgs args{level, maxIterations, depth, depthPitch, scribble, scribblePitch, gray, grayPitch, nullptr, 0, nullptr, 0, 0, 0, nullptr, 0, true};
    return run_cached_graph(ctx, key, [&](cudaStream_t cs, int *kernels) { return enqueue_level(ctx, cs, args, true, kernels); });
}

int rtdd_selftest_division(rtdd_ctx *ctx, unsigned long long n, unsigned long long seed, int mode, unsigned long long *mismatches)
{
    if (!ctx) return RTDD_E_ARG;
    if (!mismatches || mode < 0 || mode > 4) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_selftest_division");
    DeviceGuard guard(ctx->device);
    unsigned long long *d = nullptr;
    RTDD_TRY(cudaMalloc((void **)&d, sizeof(*d)), "rtdd_selftest_division");
    cudaError_t e = cudaMemsetAsync(d, 0, sizeof(*d), ctx->stream);
    if (e == cudaSuccess) e = rtdd::launch_division_selftest(ctx->stream, n, seed, mode, d);
    if (e == cudaSuccess) e = cudaMemcpyAsync(mismatches, d, sizeof(*d), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    ctx->launches++;
    return rtdd_check(ctx, e, "rtdd_selftest_division");
}

int rtdd_level_sweep_ms(rtdd_ctx *ctx, int level, float *ms, int *iterations, int *kernels)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels || !ms) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_level_sweep_ms");
    RtddLevel &L = ctx->lv[level];
    if (!L.timed) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_level_sweep_ms (level not solved yet)");
    DeviceGuard guard(ctx->device);
    RTDD_TRY(cudaEventSynchronize(L.evEnd), "rtdd_level_sweep_ms");
    RTDD_TRY(cudaEventElapsedTime(ms, L.evBegin, L.evEnd), "rtdd_level_sweep_ms");
    if (iterations) *iterations = L.lastIters;
    if (kernels) *kernels = L.lastKernels;
    return 0;
}

int rtdd_level_residual(rtdd_ctx *ctx, int level, float *residual)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels || !residual) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_level_residual");
    DeviceGuard guard(ctx->device);
    unsigned int bits = 0;
    RTDD_TRY(cudaMemcpyAsync(&bits, ctx->lv[level].dResidual, sizeof(bits), cudaMemcpyDeviceToHost, ctx->stream), "rtdd_level_residual");
    RTDD_TRY(cudaStreamSynchronize(ctx->stream), "rtdd_level_residual");
    memcpy(residual, &bits, sizeof(bits));
    return 0;
}

int rtdd_solve_level_converge(rtdd_ctx *ctx, float *depth, size_t depthPitch, const uint8_t *scribble, size_t scribblePitch,
                              const uint8_t *gray, size_t grayPitch, int rows, int cols, int maxIterations, float tolerance,
                              int checkEvery, int level, int *iterationsRun, float *finalResidual)
{
    if (!ctx) return RTDD_E_ARG;
    if (maxIterations < 0 || checkEvery < 1 || !(tolerance >= 0.0f)) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_solve_level_converge");
    int rc = rtdd_strip_init(ctx, level, depth, depthPitch, scribble, scribblePitch, gray, grayPitch, rows, cols, 0, rows);
    if (rc) return rc;
    const int T = 8;
    int done = 0;
    float res = INFINITY;
    struct ResidualOn {                                       // the passes of this call fill the residual word
        rtdd_ctx *c; bool old;
        explicit ResidualOn(rtdd_ctx *x) : c(x), old(x->stripResidual) { c->stripResidual = true; }
        ~ResidualOn() { c->stripResidual = old; }
    } residualOn(ctx);
    while (done < maxIterations) {
        int chunk = maxIterations - done < checkEvery ? maxIterations - done : checkEvery;
        while (chunk > 0) {
            const int n = chunk < T ? chunk : T;
            rc = rtdd_strip_pass(ctx, level, done, n, T);
            if (rc) return rc;
            done += n;
            chunk -= n;
        }
        rc = rtdd_level_residual(ctx, level, &res);          // one 4-byte read-back per check
        if (rc) return rc;
        if (res <= tolerance) break;
    }
    if (iterationsRun) *iterationsRun = done;
    if (finalResidual) *finalResidual = res;
    return rtdd_strip_finish(ctx, level, depth, depthPitch, 0, rows);
}

int rtdd_edge_weights(rtdd_ctx *ctx, const float *depth, size_t depthPitch, const uint8_t *gray, size_t grayPitch,
                      int rows, int cols, int level, uint8_t *linkRight, uint8_t *linkDown, size_t outPitch)
{
    if (!ctx) return RTDD_E_ARG;
    DeviceGuard guard(ctx->device);
    // the mask plane is not needed for the links: pass gray as a stand-in scribble plane (any readable u8 plane)
    int rc = edge_pass(ctx, depth, depthPitch, gray, grayPitch, gray, grayPitch, rows, cols, level, "rtdd_edge_weights");
    if (rc) return rc;
    if (linkRight || linkDown) {
        RTDD_TRY(rtdd::launch_export_links(ctx->stream, ctx->lv[level], linkRight, linkDown, outPitch), "rtdd_edge_weights (export)");
        ctx->launches++;
    }
    return 0;
}

// ---- row strips (multi-GPU domain decomposition of one level) -----------------------
//
// A rank owns rows [a, b) of a level and keeps a window [a - H, b + H) (clipped to the image) in the level's
// planes.  Window edges that are not image edges are treated like the inner edges of the blocked kernel's tiles:
// after n sweeps the n rows next to such an edge are stale, so with H >= the sweeps between two halo exchanges
// every owned row has gone through exactly the reference's per-pixel recipe -- bit-identical to one GPU.
// The exchange itself (the (x_k, x_{k-1}) rows next to the strip boundary) is the caller's: NCCL send/recv on
// rtdd_strip_planes' pointers (realtimedepthdiffusion_b200/strips.py).

static int strip_init_impl(rtdd_ctx *ctx, int level, const float *depth, size_t depthPitch, const uint8_t *scribble, size_t scribblePitch,
                           const uint8_t *gray, size_t grayPitch, int rows, int cols, int winBegin, int winEnd, int fixRowA, int fixRowB);

int rtdd_strip_init(rtdd_ctx *ctx, int level, const float *depth, size_t depthPitch, const uint8_t *scribble, size_t scribblePitch,
                    const uint8_t *gray, size_t grayPitch, int rows, int cols, int winBegin, int winEnd)
{
    return strip_init_impl(ctx, level, depth, depthPitch, scribble, scribblePitch, gray, grayPitch, rows, cols, winBegin, winEnd, -1, -1);
}

// fixRowA / fixRowB: window-local rows frozen as Dirichlet rows (-1 = none), see rtdd_frame_solve_band
static int strip_init_impl(rtdd_ctx *ctx, int level, const float *depth, size_t depthPitch, const uint8_t *scribble, size_t scribblePitch,
                           const uint8_t *gray, size_t grayPitch, int rows, int cols, int winBegin, int winEnd, int fixRowA, int fixRowB)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->lutLoaded) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_strip_init (rtdd_load_weights not called)");
    if (!depth || !scribble || !gray || level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_init");
    RtddLevel &L = ctx->lv[level];
    if (rows != L.rows || cols != L.cols || winBegin < 0 || winEnd > rows || winEnd <= winBegin || winEnd - winBegin > L.planeRows)
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_init");
    DeviceGuard guard(ctx->device);
    RtddLevel W = L;
    W.rows = winEnd - winBegin;
    const bool coarsest = (level == ctx->levels - 1);
    const int threshold = (level == 0) ? 0 : 4;
    const float *d = (const float *)((const char *)depth + (size_t)winBegin * depthPitch);
    // the window's last row needs the gray/depth row below it only if that row is inside the window; a window edge
    // inside the image simply loses that link, which only affects rows that go stale anyway
    RTDD_TRY(cudaMemsetAsync(L.dBad, 0, sizeof(unsigned int), ctx->stream), "rtdd_strip_init");
    RTDD_TRY(rtdd::launch_level_init(ctx->stream, W, d, depthPitch, scribble + (size_t)winBegin * scribblePitch, scribblePitch,
                                     gray + (size_t)winBegin * grayPitch, grayPitch, coarsest, threshold, L.x[0], nullptr, fixRowA, fixRowB), "rtdd_strip_init");
    ctx->launches++;
    L.stripBegin = winBegin; L.stripRows = W.rows; L.stripPair = 0;
    L.stripFused = false;
    // a proper strip: values also arrive from other ranks (a band between frozen rows is closed: nothing arrives)
    L.stripScan = (winBegin > 0 && fixRowA < 0) || (winEnd < rows && fixRowB < 0);
    L.dPeerBad = nullptr;
    L.stripFirstPassAbs = L.stripPassAbs;
    return 0;
}

int rtdd_ipc_export(rtdd_ctx *ctx, void *handle64)
{
    if (!ctx) return RTDD_E_ARG;
    if (!handle64) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_ipc_export");
    DeviceGuard guard(ctx->device);
    cudaIpcMemHandle_t h;
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    RTDD_TRY(cudaIpcGetMemHandle(&h, ctx->arena), "rtdd_ipc_export");
    memcpy(handle64, &h, sizeof(h));
    return 0;
}

int rtdd_ipc_import(rtdd_ctx *ctx, const void *handle64, void **peerArena)
{
    if (!ctx) return RTDD_E_ARG;
    if (!handle64 || !peerArena) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_ipc_import");
    DeviceGuard guard(ctx->device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    const int rc = rtdd_check(ctx, cudaIpcOpenMemHandle(peerArena, h, cudaIpcMemLazyEnablePeerAccess), "rtdd_ipc_import");
    if (rc) return rtdd_fail(ctx, RTDD_E_PEER, "rtdd_ipc_import (cudaIpcOpenMemHandle)");
    ctx->ipcImports.push_back(*peerArena);
    return 0;
}

int rtdd_arena(rtdd_ctx *ctx, void **base, size_t *bytes)
{
    if (!ctx) return RTDD_E_ARG;
    if (base) *base = ctx->arena;
    if (bytes) *bytes = ctx->arenaBytes;
    return 0;
}

int rtdd_strip_set_peers(rtdd_ctx *ctx, void *arenaAbove, void *arenaBelow)
{
    if (!ctx) return RTDD_E_ARG;
    ctx->peerUp = (char *)arenaAbove;
    ctx->peerDn = (char *)arenaBelow;
    return 0;
}

int rtdd_strip_neighbours(rtdd_ctx *ctx, int level, int ownBegin, int ownEnd, int halo, int aboveWinBegin, int belowWinBegin)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_neighbours");
    RtddLevel &L = ctx->lv[level];
    if (L.stripRows <= 0 || ownBegin < L.stripBegin || ownEnd > L.stripBegin + L.stripRows || ownEnd - ownBegin < halo || halo < 1)
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_neighbours");
    L.stripOwnBegin = ownBegin; L.stripOwnEnd = ownEnd; L.stripHalo = halo;
    L.stripUpWinBegin = aboveWinBegin; L.stripDnWinBegin = belowWinBegin;
    L.stripFused = !ctx->peerStaging;      // staged exchange: the passes stay the plain kernels
    L.stripPushOff = false;
    if (ctx->peerStaging) { L.stripScan = false; L.dPeerBad = ctx->dPeerBadWord; }      // the push kernels carry the neighbours' verdicts
    if (ctx->peerStaging && halo > RTDD_MAX_HALO) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_neighbours (halo beyond the staging area)");
    return 0;
}

// ---- staged peer exchange -------------------------------------------------------------------------
// staging rows of level L: [buffer][side: 0 = rows from the rank above, 1 = from the rank below][plane: x_k, x_{k-1}]
static float *stage_rows(const RtddLevel &L, char *arenaBase, const rtdd_ctx *ctx, int buffer, int side, int plane)
{
    const size_t off = (char *)L.stage - (char *)ctx->arena;
    return (float *)(arenaBase + off) + (size_t)((buffer * 2 + side) * 2 + plane) * RTDD_MAX_HALO * L.pitchF;
}

int rtdd_strip_push(rtdd_ctx *ctx, int level)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_push");
    RtddLevel &L = ctx->lv[level];
    if (!ctx->peerStaging || L.stripRows <= 0 || L.stripHalo < 1) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_strip_push (rtdd_strip_neighbours with staging not called)");
    DeviceGuard guard(ctx->device);
    const int H = L.stripHalo;
    const int gt = L.stripOwnBegin - L.stripBegin;
    const int own1 = gt + (L.stripOwnEnd - L.stripOwnBegin);
    const int buffer = (int)(L.peerSeq & 1u);
    const float *xk = L.x[L.stripPair], *xp = L.x[L.stripPair + 1];
    const size_t offW = (char *)L.dStripWords - (char *)ctx->arena;
    rtdd::HaloRows up = {}, dn = {};
    unsigned int *upFlag = nullptr, *dnFlag = nullptr;
    if (ctx->peerUp && L.stripUpWinBegin >= 0) {       // my first H own rows are the rank above's "rows from below"
        up.srcX = xk + (size_t)gt * L.pitchF; up.srcP = xp + (size_t)gt * L.pitchF;
        up.dstX = stage_rows(L, ctx->peerUp, ctx, buffer, 1, 0); up.dstP = stage_rows(L, ctx->peerUp, ctx, buffer, 1, 1);
        up.rows = H;
        upFlag = (unsigned int *)(ctx->peerUp + offW) + 6;
    }
    if (ctx->peerDn && L.stripDnWinBegin >= 0) {       // my last H own rows are the rank below's "rows from above"
        dn.srcX = xk + (size_t)(own1 - H) * L.pitchF; dn.srcP = xp + (size_t)(own1 - H) * L.pitchF;
        dn.dstX = stage_rows(L, ctx->peerDn, ctx, buffer, 0, 0); dn.dstP = stage_rows(L, ctx->peerDn, ctx, buffer, 0, 1);
        dn.rows = H;
        dnFlag = (unsigned int *)(ctx->peerDn + offW) + 5;
    }
    const size_t offBad = (char *)ctx->dPeerBadWord - (char *)ctx->arena;
    RTDD_TRY(rtdd::launch_halo_push(ctx->stream, up, dn, L.pitchF, L.dStripWords + 4, upFlag, dnFlag, L.peerSeq + 1u, L.dBad, ctx->dPeerBadWord,
                                    upFlag ? (unsigned int *)(ctx->peerUp + offBad) : nullptr, dnFlag ? (unsigned int *)(ctx->peerDn + offBad) : nullptr),
             "rtdd_strip_push");
    ctx->launches++;
    return 0;
}

int rtdd_strip_pull(rtdd_ctx *ctx, int level)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_pull");
    RtddLevel &L = ctx->lv[level];
    if (!ctx->peerStaging || L.stripRows <= 0 || L.stripHalo < 1) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_strip_pull (rtdd_strip_neighbours with staging not called)");
    DeviceGuard guard(ctx->device);
    const int H = L.stripHalo;
    const int gt = L.stripOwnBegin - L.stripBegin;
    const int own1 = gt + (L.stripOwnEnd - L.stripOwnBegin);
    const int buffer = (int)(L.peerSeq & 1u);
    float *xk = L.x[L.stripPair], *xp = L.x[L.stripPair + 1];
    rtdd::HaloRows up = {}, dn = {};
    const unsigned int *waitUp = nullptr, *waitDn = nullptr;
    if (ctx->peerUp && L.stripUpWinBegin >= 0) {       // rows from the rank above -> my upper ghost rows
        if (gt != H) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_strip_pull (upper ghost rows != halo)");
        up.srcX = stage_rows(L, (char *)ctx->arena, ctx, buffer, 0, 0); up.srcP = stage_rows(L, (char *)ctx->arena, ctx, buffer, 0, 1);
        up.dstX = xk; up.dstP = xp;
        up.rows = H;
        waitUp = L.dStripWords + 5;
    }
    if (ctx->peerDn && L.stripDnWinBegin >= 0) {       // rows from the rank below -> my lower ghost rows
        if (own1 + H != L.stripRows) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_strip_pull (lower ghost rows != halo)");
        dn.srcX = stage_rows(L, (char *)ctx->arena, ctx, buffer, 1, 0); dn.srcP = stage_rows(L, (char *)ctx->arena, ctx, buffer, 1, 1);
        dn.dstX = xk + (size_t)own1 * L.pitchF; dn.dstP = xp + (size_t)own1 * L.pitchF;
        dn.rows = H;
        waitDn = L.dStripWords + 6;
    }
    RTDD_TRY(rtdd::launch_halo_pull(ctx->stream, up, dn, L.pitchF, waitUp, waitDn, L.peerSeq + 1u, ctx->dErrWord, ctx->spinTimeoutMs), "rtdd_strip_pull");
    L.peerSeq++;
    ctx->launches++;
    return 0;
}

int rtdd_strip_push_enable(rtdd_ctx *ctx, int level, int on)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_push_enable");
    ctx->lv[level].stripPushOff = !on;
    return 0;
}

int rtdd_strip_wait(rtdd_ctx *ctx, int level)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_wait");
    RtddLevel &L = ctx->lv[level];
    if (!L.stripFused || L.stripPassAbs == L.stripFirstPassAbs) return 0;
    DeviceGuard guard(ctx->device);
    const unsigned int *wu = (ctx->peerUp && L.stripUpWinBegin >= 0) ? L.dStripWords + 1 : nullptr;
    const unsigned int *wd = (ctx->peerDn && L.stripDnWinBegin >= 0) ? L.dStripWords + 2 : nullptr;
    RTDD_TRY(rtdd::launch_halo_wait(ctx->stream, wu, wd, L.stripPassAbs, ctx->dErrWord, ctx->spinTimeoutMs), "rtdd_strip_wait");
    ctx->launches++;
    return 0;
}

static int strip_pass_impl(rtdd_ctx *ctx, int level, int firstSweep, int nsweeps, int haloT, float *depth, size_t depthPitch, uint8_t *u8, size_t u8Pitch);

int rtdd_strip_pass(rtdd_ctx *ctx, int level, int firstSweep, int nsweeps, int haloT)
{
    return strip_pass_impl(ctx, level, firstSweep, nsweeps, haloT, nullptr, 0, nullptr, 0);
}

// The level's LAST pass writing straight into the caller's pitched depth plane (and, optionally, the 8-bit map): replaces
// rtdd_strip_pass + rtdd_strip_finish where no halo exchange follows (the finest level).  depth / depthU8 are the FULL planes
// (row 0 of the level); every row of the window is written, the ghost rows with their stale values (they belong to other ranks).
int rtdd_strip_pass_to(rtdd_ctx *ctx, int level, int firstSweep, int nsweeps, int haloT, float *depth, size_t depthPitch, uint8_t *depthU8, size_t depthU8Pitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (!depth || !target_ok(depth, depthPitch)) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_pass_to (depth plane must be 16-byte aligned)");
    return strip_pass_impl(ctx, level, firstSweep, nsweeps, haloT, depth, depthPitch, depthU8, depthU8Pitch);
}

static int strip_pass_impl(rtdd_ctx *ctx, int level, int firstSweep, int nsweeps, int haloT, float *depth, size_t depthPitch, uint8_t *u8, size_t u8Pitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_pass");
    RtddLevel &L = ctx->lv[level];
    if (L.stripRows <= 0) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_strip_pass (rtdd_strip_init not called)");
    if (firstSweep < 0 || nsweeps < 1 || haloT < nsweeps || haloT > RTDD_MAX_T) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_pass");
    DeviceGuard guard(ctx->device);
    std::vector<float> om;
    omega_schedule(firstSweep + nsweeps, om);
    rtdd::OmegaPack pack;
    for (int i = 0; i < RTDD_MAX_T; i++) pack.w[i] = (i < nsweeps) ? om[firstSweep + i] : 0.0f;
    RtddLevel W = L;
    W.rows = L.stripRows;
    W.magnitudeCheck = L.stripScan;    // ghost rows from other GPUs without an exchange of verdicts: every pass scans its own tiles (sweep_cluster_kernel)
    const int src = L.stripPair, dst = src ^ 2;
    // on request, the residual of this pass's last sweep (over the whole window; stale ghost rows can only raise it).  Not by
    // default: measured on the 16K level-0 pass, accumulating it costs 4.14 vs 3.87 ms per pass (ncu launch lists,
    // profiles/r01_strip_path_vs_level_graph.txt)
    const bool wantResidual = ctx->stripResidual;
    rtdd::SweepTarget tgt = {nullptr, 0, nullptr, 0, wantResidual ? L.dResidual : nullptr};
    if (depth) {
        tgt.x = (float *)((char *)depth + (size_t)L.stripBegin * depthPitch);
        tgt.pitchX = (int)(depthPitch / sizeof(float));
        if (u8) { tgt.u8 = u8 + (size_t)L.stripBegin * u8Pitch; tgt.pitchU8 = (int)u8Pitch; }
    }
    if (wantResidual) RTDD_TRY(cudaMemsetAsync(L.dResidual, 0, sizeof(unsigned int), ctx->stream), "rtdd_strip_pass");
    rtdd::HaloPush hp = {};
    bool fused = L.stripFused && (ctx->peerUp || ctx->peerDn);
    // a pass that neither waits for nor feeds a neighbour (the finest level's only pass) runs the plain kernel
    const bool firstOfLevel = (L.stripPassAbs == L.stripFirstPassAbs);
    if (fused && L.stripPushOff && firstOfLevel) {
        fused = false;
        L.stripPassAbs++;               // keep the pass tickets of all ranks in step
    }
    if (fused) {
        // the same plane of the neighbour sits at the same offset of ITS arena
        const int H = L.stripHalo;
        const size_t offX = (char *)L.x[dst] - (char *)ctx->arena, offP = (char *)L.x[dst + 1] - (char *)ctx->arena;
        const size_t offW = (char *)L.dStripWords - (char *)ctx->arena;
        const int gt = L.stripOwnBegin - L.stripBegin;                       // ghost rows above my own rows
        const int own1 = gt + (L.stripOwnEnd - L.stripOwnBegin);
        hp.pitch = L.pitchF;
        hp.storeLo = 0;
        hp.storeHi = 0x7FFFFFFF;
        if (ctx->peerUp && L.stripUpWinBegin >= 0) hp.storeLo = gt;       // the rank above fills my upper ghost rows
        if (ctx->peerDn && L.stripDnWinBegin >= 0) hp.storeHi = own1;     // the rank below fills my lower ghost rows
        // The waits and the completion flags belong to the NEIGHBOUR RELATION, not to the push: a pass that keeps its
        // boundary rows to itself (stripPushOff, the finest level's last pass) still reads ghost rows its neighbours pushed
        // during the previous pass, so it must wait for them, and it still raises its flags (rtdd.h).
        if (ctx->peerUp && L.stripUpWinBegin >= 0) {
            if (!L.stripPushOff) {
                hp.upX = (float *)(ctx->peerUp + offX); hp.upP = (float *)(ctx->peerUp + offP);
                hp.upLo = gt; hp.upHi = gt + H;
                hp.upDelta = L.stripBegin - L.stripUpWinBegin;               // window-local row -> neighbour's window-local row
            }
            hp.upFlag = (unsigned int *)(ctx->peerUp + offW) + 2;            // "written by the rank below"
            hp.waitUp = L.dStripWords + 1;
        }
        if (ctx->peerDn && L.stripDnWinBegin >= 0) {
            if (!L.stripPushOff) {
                hp.dnX = (float *)(ctx->peerDn + offX); hp.dnP = (float *)(ctx->peerDn + offP);
                hp.dnLo = own1 - H; hp.dnHi = own1;
                hp.dnDelta = L.stripBegin - L.stripDnWinBegin;
            }
            hp.dnFlag = (unsigned int *)(ctx->peerDn + offW) + 1;            // "written by the rank above"
            hp.waitDn = L.dStripWords + 2;
        }
        hp.err = ctx->dErrWord;
        hp.timeoutMs = ctx->spinTimeoutMs;
        hp.counter = L.dStripWords;
        hp.doneTarget = L.stripCtaAbs;                                       // the launcher adds this pass's CTA count
        hp.flagValue = L.stripPassAbs + 1;
        hp.waitValue = (L.stripPassAbs > L.stripFirstPassAbs) ? L.stripPassAbs : 0;   // first pass of a level: nothing to wait for
    }
    RTDD_TRY(rtdd::launch_sweep_blocked(ctx->stream, W, ctx->dLut, L.x[src], L.x[src + 1], L.x[dst], L.x[dst + 1], pack, haloT, nsweeps, 0.99f,
                                        firstSweep == 0, ctx->smCount, (tgt.x || tgt.res) ? &tgt : nullptr, fused ? &hp : nullptr), "rtdd_strip_pass");
    if (fused) { L.stripCtaAbs = hp.doneTarget; L.stripPassAbs++; }
    ctx->launches++;
    L.stripPair = dst;
    return 0;
}

int rtdd_strip_planes(rtdd_ctx *ctx, int level, float **xk, float **xkm1, size_t *pitchBytes, int *winBegin, int *winRows)
{
    if (!ctx) return RTDD_E_ARG;
    if (level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_planes");
    RtddLevel &L = ctx->lv[level];
    if (L.stripRows <= 0) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_strip_planes");
    if (xk) *xk = L.x[L.stripPair];
    if (xkm1) *xkm1 = L.x[L.stripPair + 1];
    if (pitchBytes) *pitchBytes = (size_t)L.pitchF * sizeof(float);
    if (winBegin) *winBegin = L.stripBegin;
    if (winRows) *winRows = L.stripRows;
    return 0;
}

int rtdd_strip_finish(rtdd_ctx *ctx, int level, float *depth, size_t depthPitch, int rowBegin, int rowEnd)
{
    if (!ctx) return RTDD_E_ARG;
    if (!depth || level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_finish");
    RtddLevel &L = ctx->lv[level];
    if (L.stripRows <= 0 || rowBegin < L.stripBegin || rowEnd > L.stripBegin + L.stripRows || rowEnd <= rowBegin)
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_strip_finish");
    DeviceGuard guard(ctx->device);
    RtddLevel W = L;
    W.rows = rowEnd - rowBegin;
    const float *x = L.x[L.stripPair] + (size_t)(rowBegin - L.stripBegin) * L.pitchF;
    RTDD_TRY(rtdd::launch_copy_out(ctx->stream, W, x, (float *)((char *)depth + (size_t)rowBegin * depthPitch), depthPitch), "rtdd_strip_finish");
    ctx->launches++;
    return 0;
}

int rtdd_pyrup_depth_rows(rtdd_ctx *ctx, const float *src, size_t srcPitch, int srcRows, int srcCols,
                          float *dst, size_t dstPitch, int dstRows, int dstCols, int rowBegin, int rowEnd)
{
    if (!ctx) return RTDD_E_ARG;
    if (!src || !dst || srcRows < 1 || srcCols < 1 || dstRows < 2 * srcRows || dstRows > 2 * srcRows + 1 ||
        dstCols < 2 * srcCols || dstCols > 2 * srcCols + 1 || rowBegin < 0 || rowEnd > dstRows || rowEnd < rowBegin)
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_pyrup_depth_rows");
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_pyrup_depth_rows(ctx->stream, src, srcPitch, srcRows, srcCols, dst, dstPitch, dstRows, dstCols, rowBegin, rowEnd),
             "rtdd_pyrup_depth_rows");
    ctx->launches++;
    return 0;
}

// ---- GPUImageProcessing --------------------------------------------------------

int rtdd_convert_to_float(rtdd_ctx *ctx, const uint8_t *src, size_t srcPitch, float *dst, size_t dstPitch,
                          const uint8_t *mask, size_t maskPitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!src || !dst || !mask || rows < 0 || cols < 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_convert_to_float");
    if (rows == 0 || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_convert(ctx->stream, src, srcPitch, dst, dstPitch, mask, maskPitch, rows, cols), "rtdd_convert_to_float");
    ctx->launches++;
    return 0;
}

int rtdd_pyrdown_annotation(rtdd_ctx *ctx, const uint8_t *prevScribble, size_t prevScribblePitch,
                            const uint8_t *prevEdited, size_t prevEditedPitch, int previousRows, int previousCols,
                            uint8_t *currScribble, size_t currScribblePitch,
                            uint8_t *currEdited, size_t currEditedPitch, int currentRows, int currentCols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!prevScribble || !prevEdited || !currScribble || !currEdited || previousRows < 0 || previousCols < 0 || currentRows < 0 || currentCols < 0)
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_pyrdown_annotation");
    if (currentRows == 0 || currentCols == 0) return 0;
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_pyrdown_annotation(ctx->stream, prevScribble, prevScribblePitch, prevEdited, prevEditedPitch, previousRows, previousCols,
                                             currScribble, currScribblePitch, currEdited, currEditedPitch, currentRows, currentCols),
             "rtdd_pyrdown_annotation");
    ctx->launches++;
    return 0;
}

int rtdd_paint(rtdd_ctx *ctx, int x, int y, int scribbleColor, int scribbleRadius,
               uint8_t *edited, size_t editedPitch, uint8_t *scribble, size_t scribblePitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!edited || !scribble || rows < 0 || cols < 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_paint");
    DeviceGuard guard(ctx->device);
    int launched = 0;
    RTDD_TRY(rtdd::launch_paint(ctx->stream, x, y, scribbleColor, scribbleRadius, edited, editedPitch, scribble, scribblePitch, rows, cols, &launched),
             "rtdd_paint");
    ctx->launches += launched;
    return 0;
}

int rtdd_annotation_ingest(rtdd_ctx *ctx, const uint8_t *annotation, size_t annotationPitch, const uint8_t *bgr, size_t bgrPitch,
                           uint8_t *edited, size_t editedPitch, uint8_t *scribble, size_t scribblePitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!annotation || !bgr || !edited || !scribble || rows < 0 || cols < 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_annotation_ingest");
    if (rows == 0 || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_annotation_ingest(ctx->stream, annotation, annotationPitch, bgr, bgrPitch, edited, editedPitch, scribble, scribblePitch, rows, cols),
             "rtdd_annotation_ingest");
    ctx->launches++;
    return 0;
}

// ---- GPUDepthEffect ------------------------------------------------------------

int rtdd_desaturate(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                    const float *depth, size_t depthPitch, uint8_t *out, size_t outPitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!orig || !gray || !depth || !out || rows < 0 || cols < 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_desaturate");
    if (rows == 0 || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_desaturate(ctx->stream, orig, origPitch, gray, grayPitch, depth, depthPitch, out, outPitch, rows, cols), "rtdd_desaturate");
    ctx->launches++;
    return 0;
}

int rtdd_haze(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
              uint8_t *out, size_t outPitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!orig || !depth || !out || rows < 0 || cols < 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_haze");
    if (rows == 0 || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_haze(ctx->stream, orig, origPitch, depth, depthPitch, out, outPitch, rows, cols), "rtdd_haze");
    ctx->launches++;
    return 0;
}

static int ensure_sat(rtdd_ctx *ctx, int rows, int cols)
{
    const size_t need = rtdd::defocus_scratch_bytes(rows, cols);
    if (need <= ctx->satBytes) return 0;
    if (ctx->satScratch) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->satScratch); ctx->satScratch = nullptr; ctx->satBytes = 0; }
    RTDD_TRY(cudaMalloc(&ctx->satScratch, need), "defocus scratch");
    ctx->satBytes = need;
    return 0;
}

int rtdd_defocus(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                 uint8_t *out, size_t outPitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!orig || !depth || !out || rows < 0 || cols < 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_defocus");
    if (rows == 0 || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    int rc = ensure_sat(ctx, rows, cols);
    if (rc) return rc;
    ctx->frameSatValid = false;            // the scratch is about to hold the table of the caller's image
    int launched = 0;
    RTDD_TRY(rtdd::launch_defocus(ctx->stream, ctx->satScratch, orig, origPitch, nullptr, 0, depth, depthPitch, out, outPitch,
                                  nullptr, 0, nullptr, 0, rows, cols, &launched), "rtdd_defocus");
    ctx->launches += launched;
    return 0;
}

// Refocus parameters shared by rtdd_refocus and rtdd_frame_refocus: band half-width finite and >= 0; aperture <= 4096 after a
// negative one has been replaced by the reference's K for the image size.  (The focus depth is checked by the callers: the frame
// form may take it from the device instead.)
static bool refocus_params_ok(float depthOfField, int *aperture, int rows, int cols)
{
    if (*aperture < 0) *aperture = rtdd::defocus_kernel_size(rows, cols);
    return isfinite(depthOfField) && depthOfField >= 0.0f && *aperture <= RTDD_REFOCUS_MAX_APERTURE;
}

static bool focus_depth_ok(float f) { return f >= 0.0f && f <= 255.0f; }      // false for NaN

int rtdd_refocus(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                 uint8_t *out, size_t outPitch, int rows, int cols, float focusDepth, float depthOfField, int aperture)
{
    if (!ctx) return RTDD_E_ARG;
    if (!orig || !depth || !out || rows < 0 || cols < 0 || origPitch < (size_t)cols * 3 || outPitch < (size_t)cols * 3 ||
        depthPitch < (size_t)cols * sizeof(float) || !focus_depth_ok(focusDepth) || !refocus_params_ok(depthOfField, &aperture, rows, cols))
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_refocus");
    if (rows == 0 || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    int rc = ensure_sat(ctx, rows, cols);
    if (rc) return rc;
    ctx->frameSatValid = false;            // the scratch is about to hold the table of the caller's image
    int launched = 0;
    RTDD_TRY(rtdd::launch_sat_build(ctx->stream, ctx->satScratch, orig, origPitch, rows, cols, &launched), "rtdd_refocus (summed-area table)");
    ctx->launches += launched;
    RTDD_TRY(rtdd::launch_refocus(ctx->stream, ctx->satScratch, orig, origPitch, depth, depthPitch, out, outPitch, rows, cols,
                                  focusDepth, nullptr, depthOfField, aperture), "rtdd_refocus");
    ctx->launches++;
    return 0;
}

// Stereo outputs shared by rtdd_stereo and rtdd_frame_stereo: at least one plane, each with a full row of BGR bytes; the maximum
// disparity in [0, RTDD_STEREO_MAX_DISPARITY]; a row the kernel can hold.  (The convergence depth is checked by the callers.)
static bool stereo_params_ok(const uint8_t *left, size_t leftPitch, const uint8_t *right, size_t rightPitch,
                             const uint8_t *anaglyph, size_t anaglyphPitch, int cols, int maxDisparity)
{
    const size_t rowBytes = (size_t)cols * 3;
    return (left || right || anaglyph) && (!left || leftPitch >= rowBytes) && (!right || rightPitch >= rowBytes) &&
           (!anaglyph || anaglyphPitch >= rowBytes) && cols <= RTDD_STEREO_MAX_COLS &&
           maxDisparity >= 0 && maxDisparity <= RTDD_STEREO_MAX_DISPARITY;
}

int rtdd_stereo(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                uint8_t *left, size_t leftPitch, uint8_t *right, size_t rightPitch, uint8_t *anaglyph, size_t anaglyphPitch,
                int rows, int cols, float convergenceDepth, int maxDisparity)
{
    if (!ctx) return RTDD_E_ARG;
    if (!orig || !depth || rows < 0 || cols < 0 || origPitch < (size_t)cols * 3 || depthPitch < (size_t)cols * sizeof(float) ||
        (((uintptr_t)depth | depthPitch) & 3u) || !focus_depth_ok(convergenceDepth) ||
        !stereo_params_ok(left, leftPitch, right, rightPitch, anaglyph, anaglyphPitch, cols, maxDisparity))
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_stereo");
    if (rows == 0 || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_stereo(ctx->stream, orig, origPitch, depth, depthPitch, left, leftPitch, right, rightPitch, anaglyph, anaglyphPitch,
                                 rows, cols, convergenceDepth, nullptr, maxDisparity), "rtdd_stereo");
    ctx->launches++;
    return 0;
}

int rtdd_effects_fused(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                       const float *depth, size_t depthPitch, uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch,
                       uint8_t *defocus, size_t defocusPitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!orig || !gray || !depth || !desat || !haze || !defocus || rows < 0 || cols < 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_effects_fused");
    if (rows == 0 || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    int rc = ensure_sat(ctx, rows, cols);
    if (rc) return rc;
    ctx->frameSatValid = false;
    int launched = 0;
    RTDD_TRY(rtdd::launch_defocus(ctx->stream, ctx->satScratch, orig, origPitch, gray, grayPitch, depth, depthPitch, defocus, defocusPitch,
                                  desat, desatPitch, haze, hazePitch, rows, cols, &launched), "rtdd_effects_fused");
    ctx->launches += launched;
    return 0;
}

// DepthEffect on a row strip (SURVEY.md 8e row 3): rows [rowBegin, rowEnd) of the outputs, identical to what the whole-image calls
// put there.  Desaturation and haze are per pixel; defocus reads image rows up to half a box beyond the strip, so its summed-area
// table is built over the strip plus K/2 + 8 rows on each open side (K from the FULL image's diagonal, ref: src/GPUDepthEffect.cu:42;
// a depth beyond 255 can ask for more -- such a box takes the reference's raster path on the full image, still exact).
int rtdd_effects_rows(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                      const float *depth, size_t depthPitch, uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch,
                      uint8_t *defocus, size_t defocusPitch, int rows, int cols, int rowBegin, int rowEnd)
{
    if (!ctx) return RTDD_E_ARG;
    if (!orig || !depth || (desat && !gray) || rows < 0 || cols < 0 || rowBegin < 0 || rowEnd > rows || rowEnd < rowBegin)
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_effects_rows");
    if (rowEnd == rowBegin || cols == 0) return 0;
    DeviceGuard guard(ctx->device);
    cudaStream_t s = ctx->stream;
    const size_t o3 = (size_t)rowBegin, n = (size_t)(rowEnd - rowBegin);
    if (defocus) {
        const int K = rtdd::defocus_kernel_size(rows, cols);
        const int reach = K / 2 + 8;
        const int v0 = rowBegin - reach > 0 ? rowBegin - reach : 0;
        const int v1 = rowEnd + reach < rows ? rowEnd + reach : rows;
        int rc = ensure_sat(ctx, v1 - v0, cols);
        if (rc) return rc;
        ctx->frameSatValid = false;
        const bool all = desat && haze;
        int launched = 0;
        RTDD_TRY(rtdd::launch_defocus(s, ctx->satScratch, orig, origPitch, all ? gray : nullptr, grayPitch, depth, depthPitch, defocus, defocusPitch,
                                      all ? desat : nullptr, desatPitch, all ? haze : nullptr, hazePitch, rows, cols, &launched, true,
                                      rowBegin, rowEnd, v0, v1 - v0), "rtdd_effects_rows (defocus)");
        ctx->launches += launched;
        if (all) return 0;
    }
    if (desat) {
        RTDD_TRY(rtdd::launch_desaturate(s, orig + o3 * origPitch, origPitch, gray + o3 * grayPitch, grayPitch,
                                         (const float *)((const char *)depth + o3 * depthPitch), depthPitch, desat + o3 * desatPitch, desatPitch, (int)n, cols),
                 "rtdd_effects_rows (desaturation)");
        ctx->launches++;
    }
    if (haze) {
        RTDD_TRY(rtdd::launch_haze(s, orig + o3 * origPitch, origPitch, (const float *)((const char *)depth + o3 * depthPitch), depthPitch,
                                   haze + o3 * hazePitch, hazePitch, (int)n, cols), "rtdd_effects_rows (haze)");
        ctx->launches++;
    }
    return 0;
}

// ---- pyramid ops -----------------------------------------------------------------

int rtdd_bgr2gray(rtdd_ctx *ctx, const uint8_t *bgr, size_t bgrPitch, uint8_t *gray, size_t grayPitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!bgr || !gray || rows < 1 || cols < 1) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_bgr2gray");
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_bgr2gray(ctx->stream, bgr, bgrPitch, gray, grayPitch, rows, cols), "rtdd_bgr2gray");
    ctx->launches++;
    return 0;
}

int rtdd_pyrdown_gray(rtdd_ctx *ctx, const uint8_t *src, size_t srcPitch, int srcRows, int srcCols, uint8_t *dst, size_t dstPitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (!src || !dst || srcRows < 1 || srcCols < 1) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_pyrdown_gray");
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_pyrdown_gray(ctx->stream, src, srcPitch, srcRows, srcCols, dst, dstPitch), "rtdd_pyrdown_gray");
    ctx->launches++;
    return 0;
}

int rtdd_pyrup_depth(rtdd_ctx *ctx, const float *src, size_t srcPitch, int srcRows, int srcCols,
                     float *dst, size_t dstPitch, int dstRows, int dstCols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!src || !dst || srcRows < 1 || srcCols < 1 || dstRows < 2 * srcRows || dstRows > 2 * srcRows + 1 ||
        dstCols < 2 * srcCols || dstCols > 2 * srcCols + 1)
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_pyrup_depth");
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_pyrup_depth(ctx->stream, src, srcPitch, srcRows, srcCols, dst, dstPitch, dstRows, dstCols), "rtdd_pyrup_depth");
    ctx->launches++;
    return 0;
}

int rtdd_quantise_u8(rtdd_ctx *ctx, const float *src, size_t srcPitch, uint8_t *dst, size_t dstPitch, int rows, int cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!src || !dst || rows < 1 || cols < 1) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_quantise_u8");
    DeviceGuard guard(ctx->device);
    RTDD_TRY(rtdd::launch_quantise(ctx->stream, src, srcPitch, dst, dstPitch, rows, cols), "rtdd_quantise_u8");
    ctx->launches++;
    return 0;
}

// ---- frame driver (main.cpp:232-295 restated headless) -----------------------------

static int frame_alloc(rtdd_ctx *ctx)
{
    if (ctx->frameArena) return 0;
    ctx->fl.resize(ctx->levels);
    size_t total = 0;
    int gr = ctx->rows, gc = ctx->cols;   // gray sizes follow cv::pyrDown's ceil rule from the (ceil) level above
    for (int l = 0; l < ctx->levels; l++) {
        RtddFrameLevel &F = ctx->fl[l];
        F.rows = ctx->lv[l].rows; F.cols = ctx->lv[l].cols;
        if (l > 0) { gr = (gr + 1) / 2; gc = (gc + 1) / 2; }
        F.grayRows = gr; F.grayCols = gc;
        F.depthPitch = rtdd_round_up((size_t)F.cols * sizeof(float), 512);
        F.grayPitch = rtdd_round_up((size_t)F.grayCols, 512);
        F.scribblePitch = rtdd_round_up((size_t)F.cols, 512);
        F.editedPitch = rtdd_round_up((size_t)F.cols * 3, 512);
        total += F.depthPitch * F.rows + F.grayPitch * F.grayRows + F.scribblePitch * F.rows + F.editedPitch * F.rows;
    }
    ctx->bgrPitch = rtdd_round_up((size_t)ctx->cols * 3, 512);
    ctx->depthU8Pitch = rtdd_round_up((size_t)ctx->cols, 512);
    ctx->annotPitch = ctx->depthU8Pitch;
    total += ctx->bgrPitch * ctx->rows + ctx->depthU8Pitch * ctx->rows + ctx->annotPitch * ctx->rows;
    RTDD_TRY(cudaMalloc(&ctx->frameArena, total), "frame arena");
    char *p = (char *)ctx->frameArena;
    for (int l = 0; l < ctx->levels; l++) {
        RtddFrameLevel &F = ctx->fl[l];
        F.depth = (float *)p; p += F.depthPitch * F.rows;
        F.gray = (uint8_t *)p; p += F.grayPitch * F.grayRows;
        F.scribble = (uint8_t *)p; p += F.scribblePitch * F.rows;
        F.edited = (uint8_t *)p; p += F.editedPitch * F.rows;
    }
    ctx->bgr = (uint8_t *)p; p += ctx->bgrPitch * ctx->rows;
    ctx->depthU8 = (uint8_t *)p; p += ctx->depthU8Pitch * ctx->rows;
    ctx->annot = (uint8_t *)p;
    return 0;
}

int rtdd_frame_set_image(rtdd_ctx *ctx, const uint8_t *bgrHost, size_t bgrPitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (!bgrHost || bgrPitch < (size_t)ctx->cols * 3) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_set_image");
    DeviceGuard guard(ctx->device);
    int rc = frame_alloc(ctx);
    if (rc) return rc;
    cudaStream_t s = ctx->stream;
    RTDD_TRY(cudaMemcpy2DAsync(ctx->bgr, ctx->bgrPitch, bgrHost, bgrPitch, (size_t)ctx->cols * 3, ctx->rows, cudaMemcpyHostToDevice, s),
             "rtdd_frame_set_image (upload)");
    // annotation planes start at 0, depth planes at 255 (ref: src/main.cpp:130-136)
    for (int l = 0; l < ctx->levels; l++) {
        RtddFrameLevel &F = ctx->fl[l];
        RTDD_TRY(cudaMemsetAsync(F.scribble, 0, F.scribblePitch * F.rows, s), "rtdd_frame_set_image");
        RTDD_TRY(cudaMemsetAsync(F.edited, 0, F.editedPitch * F.rows, s), "rtdd_frame_set_image");
        RTDD_TRY(rtdd::launch_fill_f32(s, F.depth, F.depthPitch, F.rows, F.cols, 255.0f), "rtdd_frame_set_image");
        ctx->launches++;
    }
    // gray pyramid (ref: src/main.cpp:138-147); cached across frames because the image does not change
    RTDD_TRY(rtdd::launch_bgr2gray(s, ctx->bgr, ctx->bgrPitch, ctx->fl[0].gray, ctx->fl[0].grayPitch, ctx->rows, ctx->cols), "rtdd_frame_set_image");
    ctx->launches++;
    for (int l = 1; l < ctx->levels; l++) {
        RtddFrameLevel &P = ctx->fl[l - 1], &F = ctx->fl[l];
        RTDD_TRY(rtdd::launch_pyrdown_gray(s, P.gray, P.grayPitch, P.grayRows, P.grayCols, F.gray, F.grayPitch), "rtdd_frame_set_image");
        ctx->launches++;
    }
    ctx->imageSet = true;
    ctx->frameSatValid = false;
    return 0;
}

// rtdd_frame_set_image for an image that is already on the device (strip benches synthesise the 16K image there)
int rtdd_frame_set_image_device(rtdd_ctx *ctx, const uint8_t *bgrDevice, size_t bgrPitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (!bgrDevice || bgrPitch < (size_t)ctx->cols * 3) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_set_image_device");
    DeviceGuard guard(ctx->device);
    int rc = frame_alloc(ctx);
    if (rc) return rc;
    cudaStream_t s = ctx->stream;
    RTDD_TRY(cudaMemcpy2DAsync(ctx->bgr, ctx->bgrPitch, bgrDevice, bgrPitch, (size_t)ctx->cols * 3, ctx->rows, cudaMemcpyDeviceToDevice, s),
             "rtdd_frame_set_image_device (copy)");
    for (int l = 0; l < ctx->levels; l++) {
        RtddFrameLevel &F = ctx->fl[l];
        RTDD_TRY(cudaMemsetAsync(F.scribble, 0, F.scribblePitch * F.rows, s), "rtdd_frame_set_image_device");
        RTDD_TRY(cudaMemsetAsync(F.edited, 0, F.editedPitch * F.rows, s), "rtdd_frame_set_image_device");
        RTDD_TRY(rtdd::launch_fill_f32(s, F.depth, F.depthPitch, F.rows, F.cols, 255.0f), "rtdd_frame_set_image_device");
        ctx->launches++;
    }
    RTDD_TRY(rtdd::launch_bgr2gray(s, ctx->bgr, ctx->bgrPitch, ctx->fl[0].gray, ctx->fl[0].grayPitch, ctx->rows, ctx->cols), "rtdd_frame_set_image_device");
    ctx->launches++;
    for (int l = 1; l < ctx->levels; l++) {
        RtddFrameLevel &P = ctx->fl[l - 1], &F = ctx->fl[l];
        RTDD_TRY(rtdd::launch_pyrdown_gray(s, P.gray, P.grayPitch, P.grayRows, P.grayCols, F.gray, F.grayPitch), "rtdd_frame_set_image_device");
        ctx->launches++;
    }
    ctx->imageSet = true;
    ctx->frameSatValid = false;
    return 0;
}

// Zero-copy download (rtdd_set_tuning("zero_copy_out", 0/1), default on).  When the caller's 8-bit map lies in pinned (page-locked,
// device-visible) host memory, the last level-0 pass stores it there itself, next to the context's own copy: the 1 B/px cross PCIe
// WHILE the pass computes (tools/microbench/zero_copy_rate.cu: SM stores reach 50.5 GB/s against the copy engine's 55.9, and a
// store stream hidden under 0.08 ms of arithmetic still ends after 0.166 ms), instead of a copy that starts after the last kernel.
// Pageable host memory, or a plane that is not 4-byte aligned, takes the staged copy as before.

// device-visible alias of a caller's host plane, or null when the plane is pageable / misaligned / zero copy is switched off
static uint8_t *host_plane_alias(const rtdd_ctx *ctx, uint8_t *host, size_t pitch)
{
    if (!g_zeroCopyOut || !host || ((uintptr_t)host & 3u) || (pitch & 3u) || pitch > 0x7FFFFFFFu) return nullptr;
    cudaPointerAttributes at, last;
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    // the last byte of the plane must be page-locked too (a caller may have registered only part of a larger buffer)
    const uint8_t *end = host + (size_t)(ctx->rows - 1) * pitch + (size_t)ctx->cols - 1;
    if (cudaPointerGetAttributes(&last, end) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (last.type != cudaMemoryTypeHost || (const uint8_t *)last.devicePointer - (const uint8_t *)at.devicePointer != end - host) return nullptr;
    return (uint8_t *)at.devicePointer;
}

static int frame_solve_from(rtdd_ctx *ctx, int maxIterations, int startLevel, uint8_t *hostAlias = nullptr, size_t hostAliasPitch = 0,
                            bool *wroteHost = nullptr)
{
    if (wroteHost) *wroteHost = false;
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet || !ctx->lutLoaded) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_solve");
    if (maxIterations < 0 || startLevel < 0 || startLevel >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_solve");
    DeviceGuard guard(ctx->device);
    int rc = ensure_omega_table(ctx, maxIterations);
    if (rc) return rc;
    // the whole frame is ONE graph launch: every plane it touches is owned by the context, so the graph never goes stale
    RtddGraphKey key{};
    key.kind = 2; key.level = startLevel; key.iters = maxIterations; key.variant = ctx->variant; key.T = ctx->sweepsPerPass;
    // the pass that writes the host map exists only when level 0 sweeps at all and its depth plane takes float4 stores
    // ... and pays only under a pass of some length (stores into host memory hold the pass up while PCIe drains them)
    if (hostAlias && !(rtdd_level_iterations(maxIterations, ctx->levels, 0) >= 8 && target_ok(ctx->fl[0].depth, ctx->fl[0].depthPitch))) hostAlias = nullptr;
    if (hostAlias) { key.p[0] = hostAlias; key.pitch[0] = hostAliasPitch; }
    if (wroteHost) *wroteHost = hostAlias != nullptr;
    return run_cached_graph(ctx, key, [&](cudaStream_t cs, int *kernels) -> int {
        const int Lc = startLevel;          // coarsest level that is (re)solved; it starts from its current depth plane
        int n = 0;
        RTDD_TRY(cudaMemsetAsync(ctx->lv[0].dBad, 0, sizeof(unsigned int) * ctx->levels, cs), "frame: level flags");   // one node for all levels
        for (int l = 1; l <= Lc; l++) {                                       // main.cpp:249
            RtddFrameLevel &P = ctx->fl[l - 1], &F = ctx->fl[l];
            RTDD_TRY(rtdd::launch_pyrdown_annotation(cs, P.scribble, P.scribblePitch, P.edited, P.editedPitch, P.rows, P.cols,
                                                     F.scribble, F.scribblePitch, F.edited, F.editedPitch, F.rows, F.cols), "frame: annotation");
            n++;
        }
        {
            RtddFrameLevel &F = ctx->fl[Lc];                                      // main.cpp:257
            RTDD_TRY(rtdd::launch_convert(cs, F.edited, F.editedPitch, F.depth, F.depthPitch, F.scribble, F.scribblePitch, F.rows, F.cols), "frame: convert");
            n++;
        }
        bool fuseNext = false;
        for (int l = Lc; l >= 0; l--) {                                           // main.cpp:261-288
            RtddFrameLevel &F = ctx->fl[l];
            const int iters = rtdd_level_iterations(maxIterations, ctx->levels, l);
            // level 0 also emits the 8-bit map (main.cpp:290) from its last sweep pass
            LevelArgs args{l, iters, F.depth, F.depthPitch, F.scribble, F.scribblePitch, F.gray, F.grayPitch,
                           l == 0 ? ctx->depthU8 : nullptr, l == 0 ? ctx->depthU8Pitch : 0, nullptr, 0, 0, 0, nullptr, 0, false};
            if (l == 0 && hostAlias) { args.u8b = hostAlias; args.u8bPitch = hostAliasPitch; }
            if (fuseNext) {
                // this level's guess = prolongation of the level above + its own Dirichlet values, formed by its set-up kernel
                RtddFrameLevel &C = ctx->fl[l + 1];
                args.coarse = C.depth; args.coarsePitch = C.depthPitch; args.coarseRows = C.rows; args.coarseCols = C.cols;
                args.edited = F.edited; args.editedPitch = F.editedPitch;
            }
            int k = 0;
            const int r = enqueue_level(ctx, cs, args, true, &k);
            if (r) return r;
            n += k;
            fuseNext = false;
            if (l > 0) {
                RtddFrameLevel &N = ctx->fl[l - 1];
                // a level without sweeps must leave its guess in its depth plane: keep the separate kernels for it
                fuseNext = g_fusedProlong && rtdd_level_iterations(maxIterations, ctx->levels, l - 1) > 0 && target_ok(N.depth, N.depthPitch);
                if (!fuseNext) {
                    RTDD_TRY(rtdd::launch_pyrup_depth(cs, F.depth, F.depthPitch, F.rows, F.cols, N.depth, N.depthPitch, N.rows, N.cols), "frame: pyrUp");
                    RTDD_TRY(rtdd::launch_convert(cs, N.edited, N.editedPitch, N.depth, N.depthPitch, N.scribble, N.scribblePitch, N.rows, N.cols), "frame: convert");
                    n += 2;
                }
            }
        }
        *kernels = n;
        return 0;
    });
}

int rtdd_frame_solve(rtdd_ctx *ctx, int maxIterations)
{
    if (!ctx) return RTDD_E_ARG;
    return frame_solve_from(ctx, maxIterations, ctx->levels - 1);
}

int rtdd_frame_solve_incremental(rtdd_ctx *ctx, int maxIterations, int coarsestLevel)
{
    if (!ctx) return RTDD_E_ARG;
    return frame_solve_from(ctx, maxIterations, coarsestLevel);
}

int rtdd_frame_solve_host(rtdd_ctx *ctx, const uint8_t *scribbleHost, size_t scribblePitch,
                          const uint8_t *editedHost, size_t editedPitch, int maxIterations, uint8_t *depthU8Host, size_t depthU8Pitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_solve_host");
    if (!scribbleHost || !editedHost || scribblePitch < (size_t)ctx->cols || editedPitch < (size_t)ctx->cols * 3 ||
        (depthU8Host && depthU8Pitch < (size_t)ctx->cols))
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_solve_host");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = ctx->stream;
    RtddFrameLevel &F = ctx->fl[0];
    RTDD_TRY(cudaMemcpy2DAsync(F.scribble, F.scribblePitch, scribbleHost, scribblePitch, (size_t)ctx->cols, ctx->rows, cudaMemcpyHostToDevice, s),
             "rtdd_frame_solve_host (scribble upload)");                       // main.cpp:236
    RTDD_TRY(cudaMemcpy2DAsync(F.edited, F.editedPitch, editedHost, editedPitch, (size_t)ctx->cols * 3, ctx->rows, cudaMemcpyHostToDevice, s),
             "rtdd_frame_solve_host (edited upload)");                         // main.cpp:237
    bool wrote = false;
    int rc = frame_solve_from(ctx, maxIterations, ctx->levels - 1, host_plane_alias(ctx, depthU8Host, depthU8Pitch), depthU8Pitch, &wrote);
    if (rc) return rc;
    if (depthU8Host) {
        if (!wrote)
            RTDD_TRY(cudaMemcpy2DAsync(depthU8Host, depthU8Pitch, ctx->depthU8, ctx->depthU8Pitch, (size_t)ctx->cols, ctx->rows, cudaMemcpyDeviceToHost, s),
                     "rtdd_frame_solve_host (download)");                      // main.cpp:291
        RTDD_TRY(cudaStreamSynchronize(s), "rtdd_frame_solve_host");
    }
    return 0;
}

int rtdd_frame_solve_download(rtdd_ctx *ctx, int maxIterations, uint8_t *depthU8Host, size_t depthU8Pitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_solve_download");
    if (!depthU8Host || depthU8Pitch < (size_t)ctx->cols) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_solve_download");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = ctx->stream;
    bool wrote = false;
    int rc = frame_solve_from(ctx, maxIterations, ctx->levels - 1, host_plane_alias(ctx, depthU8Host, depthU8Pitch), depthU8Pitch, &wrote);
    if (rc) return rc;
    if (!wrote)
        RTDD_TRY(cudaMemcpy2DAsync(depthU8Host, depthU8Pitch, ctx->depthU8, ctx->depthU8Pitch, (size_t)ctx->cols, ctx->rows, cudaMemcpyDeviceToHost, s),
                 "rtdd_frame_solve_download");                                 // main.cpp:291
    RTDD_TRY(cudaStreamSynchronize(s), "rtdd_frame_solve_download");
    return 0;
}

// The same frame fed with the reference's persistent annotation format (ref: src/main.cpp:160-170): ONE gray plane, 32 = not
// annotated.  1 B/px crosses PCIe instead of the 4 B/px of scribble + 3-channel edited; the expansion main.cpp does on
// the host runs on the device (annotation_ingest_kernel).  Results are identical to rtdd_frame_solve_host on the planes
// main.cpp would have derived from the same annotation.
int rtdd_frame_solve_host_annotation(rtdd_ctx *ctx, const uint8_t *annotationHost, size_t annotationPitch, int maxIterations,
                                     uint8_t *depthU8Host, size_t depthU8Pitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_solve_host_annotation");
    if (!annotationHost || annotationPitch < (size_t)ctx->cols || (depthU8Host && depthU8Pitch < (size_t)ctx->cols))
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_solve_host_annotation");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = ctx->stream;
    RtddFrameLevel &F = ctx->fl[0];
    RTDD_TRY(cudaMemcpy2DAsync(ctx->annot, ctx->annotPitch, annotationHost, annotationPitch, (size_t)ctx->cols, ctx->rows, cudaMemcpyHostToDevice, s),
             "rtdd_frame_solve_host_annotation (upload)");
    RTDD_TRY(rtdd::launch_annotation_ingest(s, ctx->annot, ctx->annotPitch, ctx->bgr, ctx->bgrPitch, F.edited, F.editedPitch, F.scribble, F.scribblePitch,
                                            ctx->rows, ctx->cols), "rtdd_frame_solve_host_annotation (ingest)");
    ctx->launches++;
    bool wrote = false;
    int rc = frame_solve_from(ctx, maxIterations, ctx->levels - 1, host_plane_alias(ctx, depthU8Host, depthU8Pitch), depthU8Pitch, &wrote);
    if (rc) return rc;
    if (depthU8Host) {
        if (!wrote)
            RTDD_TRY(cudaMemcpy2DAsync(depthU8Host, depthU8Pitch, ctx->depthU8, ctx->depthU8Pitch, (size_t)ctx->cols, ctx->rows, cudaMemcpyDeviceToHost, s),
                     "rtdd_frame_solve_host_annotation (download)");
        RTDD_TRY(cudaStreamSynchronize(s), "rtdd_frame_solve_host_annotation");
    }
    return 0;
}

// ---- extension, NOT parity: re-solve a band of rows around an edit (live strokes) -------------------------------------------
// ref for what a frame is: src/main.cpp:232-295; the reference itself always re-solves everything.
// Level-0 rows [rowBegin, rowEnd) changed (a brush stroke).  Per level, coarse to fine: the band = those rows scaled to the level,
// widened by `dilation` rows on each side.  Levels the band covers by >= 60 %, and every level small enough for the
// cluster-resident kernel, are solved whole from the parity guess (prolongation of the new coarser solution + Dirichlet values):
// up to there the result EQUALS the parity frame.  On the finer levels only the band is re-solved -- same sweeps, same schedule,
// between two frozen rows of the previous solution -- and the rows outside receive the prolongated change of the coarser level
// (band_prolong_kernel).  tools/live_strokes.py and tests report how far this is from the parity frame.
int rtdd_frame_solve_band(rtdd_ctx *ctx, int maxIterations, int rowBegin, int rowEnd, int dilation)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet || !ctx->lutLoaded) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_solve_band");
    if (maxIterations < 0 || rowBegin < 0 || rowEnd > ctx->rows || rowEnd <= rowBegin || dilation < 1) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_solve_band");
    DeviceGuard guard(ctx->device);
    int rc = ensure_omega_table(ctx, maxIterations);
    if (rc) return rc;
    const int L = ctx->levels;
    cudaStream_t s = ctx->stream;
    if (!ctx->bandArena && L > 1) {
        size_t total = 0;
        for (int l = 1; l < L; l++) total += rtdd_round_up(ctx->fl[l].depthPitch * ctx->fl[l].rows, 256);
        RTDD_TRY(cudaMalloc(&ctx->bandArena, total), "rtdd_frame_solve_band (scratch)");
        ctx->bandOld.assign(L, nullptr);
        char *p = (char *)ctx->bandArena;
        for (int l = 1; l < L; l++) { ctx->bandOld[l] = (float *)p; p += rtdd_round_up(ctx->fl[l].depthPitch * ctx->fl[l].rows, 256); }
    }
    for (int l = 1; l < L; l++) {                                                            // main.cpp:249
        RtddFrameLevel &P = ctx->fl[l - 1], &F = ctx->fl[l];
        RTDD_TRY(rtdd::launch_pyrdown_annotation(s, P.scribble, P.scribblePitch, P.edited, P.editedPitch, P.rows, P.cols,
                                                 F.scribble, F.scribblePitch, F.edited, F.editedPitch, F.rows, F.cols), "band: annotation");
        ctx->launches++;
    }
    for (int l = L - 1; l >= 0; l--) {
        RtddFrameLevel &F = ctx->fl[l];
        RtddLevel &Lv = ctx->lv[l];
        const int iters = rtdd_level_iterations(maxIterations, L, l);
        int b0 = (rowBegin >> l) - dilation, b1 = ((rowEnd + (1 << l) - 1) >> l) + dilation;
        if (b0 < 0) b0 = 0;
        if (b1 > F.rows) b1 = F.rows;
        // below ~1 M pixels a pass costs its latency, not its area (measured: a 54-row band of a 480x270 level took longer than the
        // whole level inside its graph), so only the large levels are banded
        const bool whole = (l == L - 1) || (long)Lv.rows * Lv.cols < (1L << 20) || (long)(b1 - b0) * 10 >= (long)F.rows * 6;
        if (whole) { b0 = 0; b1 = F.rows; }
        if (l >= 1)         // the finer level needs this level's previous solution for the change it prolongates
            RTDD_TRY(cudaMemcpy2DAsync(ctx->bandOld[l], F.depthPitch, F.depth, F.depthPitch, (size_t)F.cols * sizeof(float), F.rows, cudaMemcpyDeviceToDevice, s),
                     "band: keep previous solution");
        if (l < L - 1) {
            RtddFrameLevel &C = ctx->fl[l + 1];
            RTDD_TRY(rtdd::launch_band_prolong(s, C.depth, ctx->bandOld[l + 1], C.depthPitch, C.rows, C.cols, F.depth, F.depthPitch, F.rows, F.cols, b0, b1),
                     "band: prolongation");
            ctx->launches++;
        }
        RTDD_TRY(rtdd::launch_convert(s, F.edited, F.editedPitch, F.depth, F.depthPitch, F.scribble, F.scribblePitch, F.rows, F.cols), "band: convert");
        ctx->launches++;
        if (whole) {
            rc = rtdd_solve_level(ctx, F.depth, F.depthPitch, F.scribble, F.scribblePitch, F.gray, F.grayPitch, F.rows, F.cols, iters, l);
            if (rc) return rc;
            continue;
        }
        // the band between two frozen rows (or an image edge)
        const int w0 = b0 > 0 ? b0 - 1 : 0, w1 = b1 < F.rows ? b1 + 1 : F.rows;
        rc = strip_init_impl(ctx, l, F.depth, F.depthPitch, F.scribble, F.scribblePitch, F.gray, F.grayPitch, F.rows, F.cols, w0, w1,
                             b0 > 0 ? 0 : -1, b1 < F.rows ? (w1 - w0 - 1) : -1);
        if (rc) return rc;
        const int T = 8;
        for (int k = 0; k < iters; k += T) {
            const int n = iters - k < T ? iters - k : T;
            rc = rtdd_strip_pass(ctx, l, k, n, T);
            if (rc) return rc;
        }
        rc = rtdd_strip_finish(ctx, l, F.depth, F.depthPitch, b0, b1);
        if (rc) return rc;
    }
    RTDD_TRY(rtdd::launch_quantise(s, ctx->fl[0].depth, ctx->fl[0].depthPitch, ctx->depthU8, ctx->depthU8Pitch, ctx->rows, ctx->cols), "band: quantise");
    ctx->launches++;
    return 0;
}

// The 8-bit depth map of the last solved frame -> HOST (ref: src/main.cpp:291 download).  sync = 0 leaves the copy in flight on the
// context stream (the caller synchronises later: several contexts' frames then overlap from one host thread).
int rtdd_frame_read_depth_u8(rtdd_ctx *ctx, uint8_t *depthU8Host, size_t depthU8Pitch, int sync)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_read_depth_u8");
    if (!depthU8Host || depthU8Pitch < (size_t)ctx->cols) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_read_depth_u8");
    DeviceGuard guard(ctx->device);
    RTDD_TRY(cudaMemcpy2DAsync(depthU8Host, depthU8Pitch, ctx->depthU8, ctx->depthU8Pitch, (size_t)ctx->cols, ctx->rows, cudaMemcpyDeviceToHost, ctx->stream),
             "rtdd_frame_read_depth_u8");
    if (sync) RTDD_TRY(cudaStreamSynchronize(ctx->stream), "rtdd_frame_read_depth_u8");
    return 0;
}

// The three depth effects on the frame's own planes (level-0 image, gray, solved depth).  The image of a frame context
// only changes in rtdd_frame_set_image, so the defocus summed-area table is built once per image and reused by every later
// call -- main.cpp re-applies the effects to the same image after every solve (ref: src/main.cpp:190-230).
int rtdd_frame_effects(rtdd_ctx *ctx, uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch, uint8_t *defocus, size_t defocusPitch)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_effects");
    const size_t rowBytes = (size_t)ctx->cols * 3;
    if ((desat && desatPitch < rowBytes) || (haze && hazePitch < rowBytes) || (defocus && defocusPitch < rowBytes))
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_effects");
    DeviceGuard guard(ctx->device);
    cudaStream_t s = ctx->stream;
    RtddFrameLevel &F = ctx->fl[0];
    const int rows = ctx->rows, cols = ctx->cols;
    if (defocus) {
        int rc = ensure_sat(ctx, rows, cols);
        if (rc) return rc;
        const bool build = !ctx->frameSatValid;
        const bool all = desat && haze;
        int launched = 0;
        RTDD_TRY(rtdd::launch_defocus(s, ctx->satScratch, ctx->bgr, ctx->bgrPitch, all ? F.gray : nullptr, all ? F.grayPitch : 0, F.depth, F.depthPitch,
                                      defocus, defocusPitch, all ? desat : nullptr, desatPitch, all ? haze : nullptr, hazePitch, rows, cols, &launched, build),
                 "rtdd_frame_effects (defocus)");
        ctx->frameSatValid = true;
        ctx->launches += launched;
        if (all) return 0;
    }
    if (desat) {
        RTDD_TRY(rtdd::launch_desaturate(s, ctx->bgr, ctx->bgrPitch, F.gray, F.grayPitch, F.depth, F.depthPitch, desat, desatPitch, rows, cols), "rtdd_frame_effects (desaturation)");
        ctx->launches++;
    }
    if (haze) {
        RTDD_TRY(rtdd::launch_haze(s, ctx->bgr, ctx->bgrPitch, F.depth, F.depthPitch, haze, hazePitch, rows, cols), "rtdd_frame_effects (haze)");
        ctx->launches++;
    }
    return 0;
}

// Refocus of the frame's own image by its solved level-0 depth, over the summed-area table rtdd_frame_effects caches too.  A focus
// point makes the kernel read the depth under it, so a captured graph of this call follows every later solve.
int rtdd_frame_refocus(rtdd_ctx *ctx, uint8_t *out, size_t outPitch, int focusX, int focusY, float focusDepth,
                       float depthOfField, int aperture)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_refocus");
    const int rows = ctx->rows, cols = ctx->cols;
    const bool byDepth = focusX == -1 && focusY == -1;
    const bool pointOk = focusX >= 0 && focusX < cols && focusY >= 0 && focusY < rows;
    if (!out || outPitch < (size_t)cols * 3 || !(byDepth ? focus_depth_ok(focusDepth) : pointOk) ||
        !refocus_params_ok(depthOfField, &aperture, rows, cols))
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_refocus");
    DeviceGuard guard(ctx->device);
    RtddFrameLevel &F = ctx->fl[0];
    const float *focusAt = byDepth ? nullptr : (const float *)((const char *)F.depth + (size_t)focusY * F.depthPitch) + focusX;
    int rc = ensure_sat(ctx, rows, cols);
    if (rc) return rc;
    if (!ctx->frameSatValid) {
        int launched = 0;
        RTDD_TRY(rtdd::launch_sat_build(ctx->stream, ctx->satScratch, ctx->bgr, ctx->bgrPitch, rows, cols, &launched), "rtdd_frame_refocus (summed-area table)");
        ctx->frameSatValid = true;
        ctx->launches += launched;
    }
    RTDD_TRY(rtdd::launch_refocus(ctx->stream, ctx->satScratch, ctx->bgr, ctx->bgrPitch, F.depth, F.depthPitch, out, outPitch, rows, cols,
                                  byDepth ? focusDepth : 0.0f, focusAt, depthOfField, aperture), "rtdd_frame_refocus");
    ctx->launches++;
    return 0;
}

// Stereo views of the frame's own image by its solved level-0 depth.  Needs no scratch, so the summed-area table that
// rtdd_frame_effects and rtdd_frame_refocus cache stays valid.  A convergence point makes the kernel read the depth under it, so a
// captured graph of this call follows every later solve.
int rtdd_frame_stereo(rtdd_ctx *ctx, uint8_t *left, size_t leftPitch, uint8_t *right, size_t rightPitch,
                      uint8_t *anaglyph, size_t anaglyphPitch, int convergenceX, int convergenceY,
                      float convergenceDepth, int maxDisparity)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_stereo");
    const int rows = ctx->rows, cols = ctx->cols;
    const bool byDepth = convergenceX == -1 && convergenceY == -1;
    const bool pointOk = convergenceX >= 0 && convergenceX < cols && convergenceY >= 0 && convergenceY < rows;
    if (!(byDepth ? focus_depth_ok(convergenceDepth) : pointOk) ||
        !stereo_params_ok(left, leftPitch, right, rightPitch, anaglyph, anaglyphPitch, cols, maxDisparity))
        return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_stereo");
    DeviceGuard guard(ctx->device);
    RtddFrameLevel &F = ctx->fl[0];
    const float *convAt = byDepth ? nullptr : (const float *)((const char *)F.depth + (size_t)convergenceY * F.depthPitch) + convergenceX;
    RTDD_TRY(rtdd::launch_stereo(ctx->stream, ctx->bgr, ctx->bgrPitch, F.depth, F.depthPitch, left, leftPitch, right, rightPitch,
                                 anaglyph, anaglyphPitch, rows, cols, byDepth ? convergenceDepth : 0.0f, convAt, maxDisparity),
             "rtdd_frame_stereo");
    ctx->launches++;
    return 0;
}

int rtdd_frame_paint(rtdd_ctx *ctx, int x, int y, int scribbleColor, int scribbleRadius)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->imageSet) return rtdd_fail(ctx, RTDD_E_STATE, "rtdd_frame_paint");
    RtddFrameLevel &F = ctx->fl[0];
    return rtdd_paint(ctx, x, y, scribbleColor, scribbleRadius, F.edited, F.editedPitch, F.scribble, F.scribblePitch, F.rows, F.cols);
}

int rtdd_frame_plane(rtdd_ctx *ctx, int which, int level, void **ptr, size_t *pitch, int *rows, int *cols)
{
    if (!ctx) return RTDD_E_ARG;
    if (!ctx->frameArena) { DeviceGuard guard(ctx->device); int rc = frame_alloc(ctx); if (rc) return rc; }
    if (level < 0 || level >= ctx->levels) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_plane");
    RtddFrameLevel &F = ctx->fl[level];
    void *p = nullptr; size_t pi = 0; int r = F.rows, c = F.cols;
    switch (which) {
    case RTDD_PLANE_DEPTH: p = F.depth; pi = F.depthPitch; break;
    case RTDD_PLANE_GRAY: p = F.gray; pi = F.grayPitch; r = F.grayRows; c = F.grayCols; break;
    case RTDD_PLANE_SCRIBBLE: p = F.scribble; pi = F.scribblePitch; break;
    case RTDD_PLANE_EDITED: p = F.edited; pi = F.editedPitch; break;
    case RTDD_PLANE_BGR: if (level != 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_plane"); p = ctx->bgr; pi = ctx->bgrPitch; break;
    case RTDD_PLANE_DEPTH_U8: if (level != 0) return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_plane"); p = ctx->depthU8; pi = ctx->depthU8Pitch; break;
    default: return rtdd_fail(ctx, RTDD_E_ARG, "rtdd_frame_plane");
    }
    if (ptr) *ptr = p;
    if (pitch) *pitch = pi;
    if (rows) *rows = r;
    if (cols) *cols = c;
    return 0;
}

}  // extern "C"
